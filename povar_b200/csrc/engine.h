// Engine: owns the device state of one shard and sequences the kernels of the hot path.
#pragma once

#include <functional>
#include <string>
#include <vector>

#include "povar_internal.h"

namespace povar {

struct NcclApi;  // dlopen'ed entry points (engine.cu)
struct PeerShared;
struct HostRendezvous;

struct PhaseTimes {
  double residual = 0, linearize = 0, prepare = 0, reduced_solve = 0, back_substitution = 0;
};

class Engine {
 public:
  static int create(const povar_problem_desc* desc, const povar_options* opt,
                    const povar_comm_desc* comm, Engine** out, std::string* err);
  static int create_device(const povar_device_problem_desc* desc, const povar_options* opt,
                           const povar_comm_desc* comm, Engine** out, std::string* err);
  ~Engine();

  int init_varproj(double alpha);
  int cost(bool joint, double alpha, povar_residual_info* out);
  int linearize(bool joint, double alpha, bool defer_check = false);
  int solve(bool joint, double lambda, double* inc, int32_t* iterations);
  int apply(bool joint, double alpha, double* l_diff);
  // One LM trial with ONE host synchronisation: solve, backup, apply, (step 2: normalise,) cost -- what the
  // caller of the Linearizor does between two accept/reject decisions (solver/bal_bundle_adjustment.cpp:346-420,
  // 655-720).  Returns the solve's status; after POVAR_NUM_NONFINITE_INC the state is garbage until restore().
  // A linearize(.., defer_check = true) before it has its failure flag checked here.
  int trial(bool joint, double alpha, double lambda, int32_t* iterations, double* l_diff, povar_residual_info* ri);
  int backup(int which);
  int restore(int which);
  int to_homogeneous();
  int normalize_joint();
  int get_state(int which, double* cam_P, double* lms);
  int set_state(int which, const double* cam_P, const double* lms);
  int get_state_device(int which, double* cam_P, double* lms, cudaStream_t caller);
  int set_state_device(int which, const double* cam_P, const double* lms, cudaStream_t caller);
  // povar_bundle_adjust_async: the solve as one CUDA graph (built on the first call with these options), enqueued
  // behind the work on `caller`; the results land in device memory
  int bundle_adjust_async(const povar_options& opt, povar_iteration* iterations, int max_iterations,
                          povar_solve_summary* summary, int* status, cudaStream_t caller);
  int64_t debug_read(const char* name, double* out, int64_t capacity);
  int right_mul_e0(bool joint, const double* x, double* out);
  int bench_power_terms(bool joint, int terms, double* seconds_per_term);
  int bench_power_kernels(bool joint, int reps, double* seconds);

  const char* last_error() const { return err_.c_str(); }
  long long launches() const { return launches_; }
  cudaStream_t stream() const { return stream_; }
  const povar_options& options() const { return opt_; }
  const PhaseTimes& last_times() const { return times_; }
  void reset_times() { times_ = PhaseTimes(); }
  int world_size() const { return world_; }
  bool peer_exchange_active() const { return peer_ok_; }
  void debug_set_window(int cams) { d_.debug_window_cams = cams; }
  void debug_set_cholesky_storage(int mode) { chol_storage_ = mode; }
  int rank() const { return rank_; }

 private:
  Engine() = default;
  int fail(int code, const std::string& what);
  int check(cudaError_t e, const char* what);
  // device, stream, communicator; then `upload` fills the index and the state
  static int create_with(const povar_options* opt, const povar_comm_desc* comm, Engine** out, std::string* err,
                         const std::function<int(Engine*)>& upload);
  // the two front halves of the index build (host list in canonical order / device list in any order) and the
  // shared back half (build_index)
  int upload(const povar_problem_desc* desc);
  int upload_device(const povar_device_problem_desc* desc);
  int build_index(int sell_n, const int* long_lms, const double* host_uv, const double* cam_P);
  int check_device_ptr(const void* p, const char* what);
  int wait_for(cudaStream_t waiter, cudaStream_t producer);   // waiter waits for the work enqueued on producer
  int allreduce(double* buf, size_t n, bool skip_when_done = false);
  int setup_peer_exchange();
  TermMode term_mode() const { return peer_ok_ ? kTermPeer : (world_ == 1 ? kTermFused : kTermRaw); }
  const PeerExchange* exchange() const;
  int sum_setup_words(unsigned int* host, int words, int phase, int round);
  void set_model(double alpha);
  // work buffers allocated on first use (linearize, solve_cholesky) and before a capture (build_solve_graph)
  int alloc_lin_buffers(bool joint);
  int alloc_cholesky(bool* tiled);
  int solve_power(bool joint, double lambda);
  int solve_pcg(bool joint, double lambda);
  int solve_cholesky(double lambda);
  int setup_cholesky_tiles();
  int prepare_reduced_system(bool joint, double lambda, double lambda_lm);
  int schur_product(bool joint, const double* p, double* out, bool skip_when_done);
  int e0_product(bool joint, bool skip_when_done, bool fused_reduce);
  int finish_solve(bool joint, double* inc, int32_t* iterations);
  int enqueue_solve(bool joint, double lambda);
  int enqueue_cost(bool joint, double alpha, bool reduce = true);
  int enqueue_apply(bool joint, double alpha, bool reduce = true);
  int enqueue_series(bool joint);
  // solve, backup, apply, (step 2: normalise,) cost, one exchange of trial_out[0..9): one LM trial, no read-back
  int enqueue_trial(bool joint, double alpha, double lambda);
  static void decode_cost(const double* v, povar_residual_info* out);
  // the series graph and the device-side solve (bundle_adjust_async): stream capture into nested conditional nodes
  cudaError_t mark(int k);   // ev_[k], or a %globaltimer stamp into lm_->stamp[k] while capturing
  int capture_graph(void** exec, const std::function<int()>& body);
  int new_cond(unsigned long long* h);
  int capture_cond(int type, unsigned long long h, const std::function<int()>& body);
  int capture_series(bool joint);
  int capture_lm_step(const povar_options& opt, bool joint, unsigned long long ok);
  int build_solve_graph(const povar_options& opt);
  LaunchCfg lc() { return LaunchCfg{stream_, &launches_}; }
  double elapsed(cudaEvent_t a, cudaEvent_t b);

  povar_options opt_{};
  DeviceState d_{};
  ModelParams mp_{};
  std::vector<void*> allocs_;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [6], [7]: linearize
  cudaEvent_t join_ev_ = nullptr;   // wait_for: ordering against a caller's stream
  long long launches_ = 0;
  std::string err_;
  PhaseTimes times_;
  // solver state
  int joint_lin_ = -1;            // model of the current linearisation: -1 none, 0 pOSE, 1 joint
  bool have_solve_ = false;       // a solve ran on the current linearisation (apply needs its increment)
  int dim_ = 12;
  double* P_prev_ = nullptr;      // cameras of the linearisation point during a VarPro apply
  bool lin_check_pending_ = false;  // linearize(defer_check): the flag is read with the next trial
  double* host_out_ = nullptr;    // pinned: [SeriesCtl (64 B) | trial_out (16 doubles)]
  // a power series as one CUDA graph per model (pOSE / joint): prefix + WHILE node around one term
  void* series_graph_[2] = {nullptr, nullptr};   // cudaGraphExec_t
  int series_calls_[2] = {0, 0};
  ModelParams series_mp_[2] = {};                // the model parameters each series graph was captured with
  bool series_terms_counted_ = true;             // the term launches of the last series are in launches_
  void count_series_terms(int terms);
  bool capturing_ = false;          // the enqueue functions are being captured into the solve graph
  void* cap_graph_ = nullptr;       // cudaGraph_t the capture writes to
  const double* lambda_dev_ = nullptr;   // while capturing: the damping in device memory (lm_->loop.lambda)
  LmCtl* lm_ = nullptr;
  povar_iteration* lm_log_ = nullptr;   // [lm_cap_] log of the device-side solve
  int lm_cap_ = 0;
  povar_solve_summary* lm_sum_ = nullptr;
  int* lm_status_ = nullptr;
  void* solve_graph_ = nullptr;     // cudaGraphExec_t of the solve, for solve_opt_ and the debug settings below
  povar_options solve_opt_{};
  int solve_window_ = 0, solve_storage_ = 0;
  double* chol_linv_ = nullptr;   // CHOLESKY: inverses of the factor's diagonal tiles [n_pad / 64][64][64]
  double* chol_rhs_ = nullptr;    // CHOLESKY: padded right-hand side / solution [n_pad]
  // CHOLESKY on tile-sparse storage (when the dense matrix would exceed kCholDenseCap, or forced)
  int chol_storage_ = 0;          // povar_debug_set_cholesky_storage: 0 automatic, 1 tile-sparse
  bool chol_tiled_ready_ = false; // the pattern below is built (at the first tile-sparse solve)
  bool chol_tiled_active_ = false;  // the last CHOLESKY solve used the tiles
  CholPattern chol_pat_;
  CholTilesDev chol_dev_;
  // distributed
  int rank_ = 0, world_ = 1, device_ = 0;
  void* nccl_comm_ = nullptr;
  NcclApi* nccl_ = nullptr;
  HostRendezvous* rdv_ = nullptr;   // povar_comm_host_id: shared-memory rendezvous instead of a communicator
  // peer-memory exchange of the per-term camera sums (world_ > 1; falls back to ncclAllReduce when
  // CUDA IPC / peer access is not available or the term grid would not be resident)
  // The mapping belongs to a process-wide cache next to the communicator (one per communicator and
  // camera count; povar_comm_finalize releases it): one solve in flight per communicator.
  PeerShared* peer_ = nullptr;
  std::string comm_key_;
  bool peer_ok_ = false;
  bool peer_small_ = true;        // cost scalars, b, Kronecker sums ... also go over the peer buffers (always)
  bool peer_owned_ = false;       // POVAR_PEER_EXCHANGE=self: a private buffer, not the communicator's
  // host mirrors
  int C_ = 0, L_ = 0;
  long long nnz_ = 0;
};

struct SellLayout {
  std::vector<int> slice_ptr;   // [num_slices+1] rows
  std::vector<int> sell_lm;     // [8*num_slices]
  std::vector<int> slice_lo;    // [num_slices] smallest camera the slice's landmarks observe
  std::vector<int> slice_hi;    // [num_slices] largest
  std::vector<int> long_lms;    // landmarks with more than 32 observations
  int rows = 0;
};
void set_host_threads_override(int n);   // 0 = automatic
void build_sell(const std::vector<int>& lm_ptr, const int* obs_cam, int num_cams, int max_window,
                SellLayout* out, int max_deg = 32);
int sell_window(int landmarks, int max_window);
int sell_key(const int* cams, int deg, int span);

// plan of the landmark half for records of rec_bytes per camera and ring stages of stage_bytes per row
// (LmPlan without the device arrays; range_slice / blk_lo come back as host vectors)
struct LmPlanHost {
  LmPlan p;
  std::vector<int> range_slice, blk_lo;
  size_t smem_bytes = 0;
};
LmPlanHost plan_landmark_half(const SellLayout& sell, int num_cams, int num_long, int rec_bytes, int stage_bytes,
                              int sms, int max_warps_per_sm = 32, int reserve_bytes = 0);
size_t landmark_half_smem(int warps, int stages, int stage_bytes, int win_cams, int rec_bytes);

// host-side index construction (engine.cu), exposed for the CPU tests through the C ABI
void build_items(const std::vector<int>& cam_ptr, int item_len, std::vector<int>* item_ptr,
                 std::vector<int>* item_cam, std::vector<int>* cam_item_ptr);
int choose_item_len(long long nnz);

}  // namespace povar
