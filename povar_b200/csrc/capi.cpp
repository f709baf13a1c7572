// extern "C" surface of libpovar_b200.so (include/povar_b200.h): thin forwarding to Engine.
#include <cstring>
#include <string>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace povar {
int nccl_unique_id(uint8_t id[128], std::string* err);
int nccl_finalize();
int host_unique_id(uint8_t id[128]);
int debug_cholesky(int n, const double* A, const double* b, double* x, int* info_out);
int debug_sparse_cholesky(int n, int block, const double* A, const double* b, double* x, int* info_out,
                          long long* stored_tiles);
}

struct povar_handle {
  povar::Engine* engine = nullptr;
  std::string create_error;
};

static thread_local std::string g_last_global_error;

template <typename F>
static int make_handle(povar_handle** out, F&& create) {
  if (!out) return POVAR_ERR_INVALID;
  *out = nullptr;
  povar_handle* h = new povar_handle();
  const int rc = create(&h->engine, &h->create_error);
  if (rc != POVAR_OK) {
    g_last_global_error = h->create_error;
    delete h;
    return rc;
  }
  *out = h;
  return POVAR_OK;
}

extern "C" {

int povar_abi_version(void) { return POVAR_ABI_VERSION; }

int64_t povar_abi_sizeof(int32_t which) {
  switch (which) {
    case 0: return sizeof(povar_options);
    case 1: return sizeof(povar_problem_desc);
    case 2: return sizeof(povar_comm_desc);
    case 3: return sizeof(povar_residual_info);
    case 4: return sizeof(povar_iteration);
    case 5: return sizeof(povar_solve_summary);
    case 6: return sizeof(povar_bal_data);
    case 7: return sizeof(povar_ba_log_info);
    case 8: return sizeof(povar_phase_times);
    case 9: return sizeof(povar_device_problem_desc);
    default: return -1;
  }
}

void povar_options_default(povar_options* o) {
  if (!o) return;
  // code defaults of bal/solver_options.hpp:88-307 and bal_residual_options.hpp:52-60
  o->solver_type_step_1 = POVAR_POWER_VARPROJ;
  o->solver_type_step_2 = POVAR_RIPOBA;
  o->robust_norm = POVAR_NORM_NONE;
  o->optimized_cost = POVAR_COST_ERROR;
  o->huber_parameter = 1.0;
  o->alpha = 0.01;
  o->max_num_iterations_step_1 = 50;
  o->max_num_iterations_step_2 = 50;
  o->min_relative_decrease = 0.0;
  o->initial_trust_region_radius = 1e4;
  o->min_trust_region_radius = 1e-32;
  o->max_trust_region_radius = 1e16;
  o->min_linear_solver_iterations = 0;
  o->max_linear_solver_iterations = 500;
  o->eta = 1e-2;
  o->r_tolerance = -1.0;
  o->jacobi_scaling_epsilon = 0.0;
  o->function_tolerance = 1e-6;
  o->power_sc_iterations = 10;
  o->verbosity_level = 2;
  o->initial_vee = 2.0;
  o->vee_factor = 2.0;
}

int povar_comm_unique_id(uint8_t id[128]) {
  std::string err;
  const int rc = povar::nccl_unique_id(id, &err);
  if (rc != POVAR_OK) g_last_global_error = err;
  return rc;
}

int povar_comm_host_id(uint8_t id[128]) {
  if (!id) return POVAR_ERR_INVALID;
  return povar::host_unique_id(id);
}

int povar_comm_finalize(void) { return povar::nccl_finalize(); }

int povar_create(const povar_problem_desc* desc, const povar_options* opt, const povar_comm_desc* comm,
                 povar_handle** out) {
  return make_handle(out, [&](povar::Engine** e, std::string* err) { return povar::Engine::create(desc, opt, comm, e, err); });
}

int povar_create_device(const povar_device_problem_desc* desc, const povar_options* opt, const povar_comm_desc* comm,
                        povar_handle** out) {
  return make_handle(out, [&](povar::Engine** e, std::string* err) {
    return povar::Engine::create_device(desc, opt, comm, e, err);
  });
}

void povar_destroy(povar_handle* h) {
  if (!h) return;
  delete h->engine;
  delete h;
}

const char* povar_last_error(const povar_handle* h) {
  if (!h || !h->engine) return g_last_global_error.c_str();
  return h->engine->last_error();
}

#define PV_ENGINE(h)                              \
  if (!(h) || !(h)->engine) return POVAR_ERR_INVALID; \
  povar::Engine& e = *(h)->engine

int povar_init_varproj(povar_handle* h, double alpha) {
  PV_ENGINE(h);
  return e.init_varproj(alpha);
}

int povar_cost_pose(povar_handle* h, double alpha, povar_residual_info* out) {
  PV_ENGINE(h);
  if (!out) return POVAR_ERR_INVALID;
  return e.cost(false, alpha, out);
}

int povar_cost_homogeneous(povar_handle* h, povar_residual_info* out) {
  PV_ENGINE(h);
  if (!out) return POVAR_ERR_INVALID;
  return e.cost(true, 0.0, out);
}

int povar_linearize_pose(povar_handle* h, double alpha) {
  PV_ENGINE(h);
  return e.linearize(false, alpha);
}

int povar_linearize_homogeneous(povar_handle* h) {
  PV_ENGINE(h);
  return e.linearize(true, 0.0);
}

int povar_solve_pose(povar_handle* h, double lambda, double* inc, int32_t* its) {
  PV_ENGINE(h);
  return e.solve(false, lambda, inc, its);
}

int povar_solve_joint(povar_handle* h, double lambda, double* inc, int32_t* its) {
  PV_ENGINE(h);
  return e.solve(true, lambda, inc, its);
}

int povar_apply_pose(povar_handle* h, double alpha, double* l_diff) {
  PV_ENGINE(h);
  return e.apply(false, alpha, l_diff);
}

int povar_apply_joint(povar_handle* h, double* l_diff) {
  PV_ENGINE(h);
  return e.apply(true, 0.0, l_diff);
}

int povar_backup(povar_handle* h, int32_t which) {
  PV_ENGINE(h);
  return e.backup(which);
}

int povar_restore(povar_handle* h, int32_t which) {
  PV_ENGINE(h);
  return e.restore(which);
}

int povar_to_homogeneous(povar_handle* h) {
  PV_ENGINE(h);
  return e.to_homogeneous();
}

int povar_normalize_joint(povar_handle* h) {
  PV_ENGINE(h);
  return e.normalize_joint();
}

int povar_get_state(povar_handle* h, int32_t which, double* cam_P, double* lms) {
  PV_ENGINE(h);
  return e.get_state(which, cam_P, lms);
}

int povar_set_state(povar_handle* h, int32_t which, const double* cam_P, const double* lms) {
  PV_ENGINE(h);
  return e.set_state(which, cam_P, lms);
}

int povar_get_state_device(povar_handle* h, int32_t which, double* cam_P, double* lms, void* stream) {
  PV_ENGINE(h);
  return e.get_state_device(which, cam_P, lms, static_cast<cudaStream_t>(stream));
}

int povar_set_state_device(povar_handle* h, int32_t which, const double* cam_P, const double* lms, void* stream) {
  PV_ENGINE(h);
  return e.set_state_device(which, cam_P, lms, static_cast<cudaStream_t>(stream));
}

int povar_bundle_adjust_async(povar_handle* h, const povar_options* opt, povar_iteration* iterations,
                              int32_t max_iterations, povar_solve_summary* summary, int32_t* status, void* stream) {
  PV_ENGINE(h);
  // the checks of povar_bundle_adjust (check_options, bal_bundle_adjustment.cpp:228-250)
  if (!opt || max_iterations < 0 || !(opt->min_trust_region_radius <= opt->initial_trust_region_radius) ||
      !(opt->initial_trust_region_radius <= opt->max_trust_region_radius) || opt->jacobi_scaling_epsilon < 0) {
    return POVAR_ERR_INVALID;
  }
  return e.bundle_adjust_async(*opt, iterations, max_iterations, summary, status, static_cast<cudaStream_t>(stream));
}

int64_t povar_debug_read(povar_handle* h, const char* name, double* out, int64_t capacity) {
  if (!h || !h->engine) return POVAR_ERR_INVALID;
  return h->engine->debug_read(name, out, capacity);
}

int povar_right_mul_e0(povar_handle* h, int32_t which, const double* x, double* out) {
  PV_ENGINE(h);
  if (!x || !out) return POVAR_ERR_INVALID;
  return e.right_mul_e0(which == POVAR_STATE_JOINT, x, out);
}

int povar_bench_power_terms(povar_handle* h, int32_t which, int32_t terms, double* seconds_per_term) {
  PV_ENGINE(h);
  return e.bench_power_terms(which == POVAR_STATE_JOINT, terms, seconds_per_term);
}

int povar_bench_power_kernels(povar_handle* h, int32_t which, int32_t reps, double seconds[4]) {
  PV_ENGINE(h);
  return e.bench_power_kernels(which == POVAR_STATE_JOINT, reps, seconds);
}

int povar_get_timings(const povar_handle* h, povar_phase_times* out) {
  if (!h || !h->engine || !out) return POVAR_ERR_INVALID;
  const povar::PhaseTimes& t = h->engine->last_times();
  out->residual_evaluation_time = t.residual;
  out->jacobian_evaluation_time = t.linearize;
  out->prepare_time = t.prepare;
  out->solve_reduced_system_time = t.reduced_solve;
  out->back_substitution_time = t.back_substitution;
  return POVAR_OK;
}

int povar_reset_timings(povar_handle* h) {
  PV_ENGINE(h);
  e.reset_times();
  return POVAR_OK;
}

int64_t povar_launch_count(const povar_handle* h) {
  if (!h || !h->engine) return 0;
  return h->engine->launches();
}

int povar_debug_sell_max_degree(int64_t num_obs, int32_t sms) {
  return povar::sell_max_degree(num_obs, sms > 0 ? sms : 148);
}

int povar_debug_sell_layout(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                            int32_t threads, int32_t max_deg, int32_t* slice_ptr, int32_t* sell_lm,
                            int32_t* long_lms, int64_t sizes[3]) {
  if (num_cams <= 0 || num_lms < 0 || !lm_ptr || !sizes) return POVAR_ERR_INVALID;
  std::vector<int> lp(static_cast<size_t>(num_lms) + 1);
  for (int32_t l = 0; l <= num_lms; ++l) lp[l] = static_cast<int>(lm_ptr[l]);
  povar::SellLayout sell;
  povar::set_host_threads_override(threads);
  povar::build_sell(lp, obs_cam, num_cams, povar::kSellWindow, &sell, max_deg > 0 ? max_deg : 32);
  povar::set_host_threads_override(0);
  sizes[0] = static_cast<int64_t>(sell.slice_ptr.size());
  sizes[1] = static_cast<int64_t>(sell.sell_lm.size());
  sizes[2] = static_cast<int64_t>(sell.long_lms.size());
  if (slice_ptr) std::copy(sell.slice_ptr.begin(), sell.slice_ptr.end(), slice_ptr);
  if (sell_lm) std::copy(sell.sell_lm.begin(), sell.sell_lm.end(), sell_lm);
  if (long_lms) std::copy(sell.long_lms.begin(), sell.long_lms.end(), long_lms);
  return POVAR_OK;
}

int povar_debug_landmark_plan(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                              int32_t model, int32_t sms, int32_t max_deg, int64_t info[8], int32_t* range_slice,
                              int32_t* blk_lo) {
  if (num_cams <= 0 || num_lms < 0 || !lm_ptr || !info || model < 0 || model > 2 || sms <= 0) return POVAR_ERR_INVALID;
  std::vector<int> lp(static_cast<size_t>(num_lms) + 1);
  for (int32_t l = 0; l <= num_lms; ++l) lp[l] = static_cast<int>(lm_ptr[l]);
  povar::SellLayout sell;
  povar::build_sell(lp, obs_cam, num_cams, povar::kSellWindow, &sell, max_deg > 0 ? max_deg : 32);
  const int rec_bytes = 8 * (model == 1 ? povar::kCamRecJoint : povar::kCamRecPose);
  const int stage_bytes = model == 0 ? povar::kStagePose : povar::kStageWide;
  const povar::LmPlanHost h = povar::plan_landmark_half(sell, num_cams, static_cast<int>(sell.long_lms.size()),
                                                        rec_bytes, stage_bytes, sms);
  info[0] = h.p.warps;
  info[1] = h.p.stages;
  info[2] = h.p.blocks_per_sm;
  info[3] = h.p.blocks;
  info[4] = h.p.ranges;
  info[5] = h.p.win_cams;
  info[6] = h.p.covered;
  info[7] = static_cast<int64_t>(h.smem_bytes);
  if (range_slice) std::copy(h.range_slice.begin(), h.range_slice.end(), range_slice);
  if (blk_lo) std::copy(h.blk_lo.begin(), h.blk_lo.begin() + h.p.blocks, blk_lo);
  return POVAR_OK;
}

int povar_debug_walk_trace(uint64_t* out, int32_t n) {
  if (!out || n <= 0 || n > 4096) return POVAR_ERR_INVALID;
  return povar::debug_walk_trace(reinterpret_cast<unsigned long long*>(out), n);
}

int povar_debug_cholesky(int32_t n, const double* A, const double* b, double* x, int32_t* info) {
  return povar::debug_cholesky(n, A, b, x, info);
}

int povar_debug_sparse_cholesky(int32_t n, int32_t block, const double* A, const double* b, double* x, int32_t* info,
                                int64_t* stored_tiles) {
  long long tiles = 0;
  const int rc = povar::debug_sparse_cholesky(n, block, A, b, x, info, &tiles);
  if (stored_tiles) *stored_tiles = tiles;
  return rc;
}

int povar_debug_cholesky_symbolic(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                                  int32_t threads, int32_t* perm, int64_t* stored_tiles) {
  if (num_cams <= 0 || num_lms < 0 || !lm_ptr || lm_ptr[0] != 0 || (lm_ptr[num_lms] > 0 && !obs_cam)) {
    return POVAR_ERR_INVALID;
  }
  for (int32_t l = 0; l < num_lms; ++l) {
    if (lm_ptr[l + 1] < lm_ptr[l]) return POVAR_ERR_INVALID;
  }
  for (int64_t i = 0; i < lm_ptr[num_lms]; ++i) {
    if (obs_cam[i] < 0 || obs_cam[i] >= num_cams) return POVAR_ERR_INVALID;
  }
  std::vector<unsigned int> bits;
  povar::covisibility_host(num_cams, num_lms, lm_ptr, obs_cam, &bits);
  povar::CholPattern p;
  povar::chol_symbolic(num_cams, 12, bits, threads, &p);
  if (perm) std::copy(p.perm.begin(), p.perm.end(), perm);
  if (stored_tiles) *stored_tiles = p.tiles();
  return POVAR_OK;
}

int povar_debug_set_cholesky_storage(povar_handle* h, int32_t mode) {
  PV_ENGINE(h);
  if (mode != 0 && mode != 1) return POVAR_ERR_INVALID;
  e.debug_set_cholesky_storage(mode);
  return POVAR_OK;
}

int povar_debug_set_window(povar_handle* h, int32_t cams) {
  PV_ENGINE(h);
  e.debug_set_window(cams);
  return POVAR_OK;
}

int povar_peer_exchange_active(const povar_handle* h) {
  if (!h || !h->engine) return 0;
  return h->engine->peer_exchange_active() ? 1 : 0;
}

void* povar_cuda_stream(const povar_handle* h) {
  if (!h || !h->engine) return nullptr;
  return reinterpret_cast<void*>(h->engine->stream());
}

}  // extern "C"

// used by the driver (host/lm_driver.cpp) to pull phase times without widening the ABI
namespace povar {
const PhaseTimes& handle_times(povar_handle* h) { return h->engine->last_times(); }
void handle_reset_times(povar_handle* h) { h->engine->reset_times(); }
int handle_rank(povar_handle* h) { return h->engine->rank(); }
int handle_linearize_deferred(povar_handle* h, bool joint, double alpha) { return h->engine->linearize(joint, alpha, true); }
int handle_trial(povar_handle* h, bool joint, double alpha, double lambda, int32_t* iterations, double* l_diff,
                 povar_residual_info* ri) {
  return h->engine->trial(joint, alpha, lambda, iterations, l_diff, ri);
}
}  // namespace povar
