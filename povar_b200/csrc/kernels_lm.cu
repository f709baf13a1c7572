// The LM loops of povar_bundle_adjust as one-thread kernels of the solve's CUDA graph (Engine::bundle_adjust_async):
// the decision of a trial is lm_step.h's, the same code the host driver runs, on a control block in device memory
// (LmCtl).  The kernels set the conditions of the graph's WHILE / IF nodes (cudaGraphSetConditional).  Times come from
// %globaltimer stamps placed where the host route records its CUDA events.
//
// This translation unit is compiled with -fmad=false: no multiply-add is contracted that the host does not contract.
#include <cuda_runtime.h>

#include "povar_internal.h"

namespace povar {

namespace {

inline void count(const LaunchCfg& lc, int n = 1) {
  if (lc.launch_counter) *lc.launch_counter += n;
}

__device__ __forceinline__ unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ double seconds(unsigned long long a, unsigned long long b) {
  return b > a ? static_cast<double>(b - a) * 1e-9 : 0.0;
}

__device__ __forceinline__ void set_cond(unsigned long long h, bool v) {
  if (h != kNoCond) cudaGraphSetConditional(static_cast<cudaGraphConditionalHandle>(h), v ? 1u : 0u);
}

// Engine::decode_cost
__device__ __forceinline__ void decode_cost(const double* v, povar_residual_info* out) {
  out->error_all = v[0];
  out->residual_sum_all = v[1];
  out->error_valid = v[2];
  out->residual_sum_valid = v[3];
  out->num_obs_all = static_cast<long long>(v[4] + 0.5);
  out->num_obs_valid = static_cast<long long>(v[5] + 0.5);
  out->is_numerically_valid = v[6] > 0 ? 0 : 1;
}

// the time columns of entry e: iteration / cumulative time and the phase times since the last entry
__device__ void stamp_entry(LmCtl* c, povar_iteration* e) {
  const unsigned long long t = now_ns();
  if (e) {
    e->iteration_time = seconds(c->t_it, t);
    e->cumulative_time = seconds(c->t_start, t);
    e->residual_evaluation_time = c->times[0];
    e->jacobian_evaluation_time = c->times[1];
    e->prepare_time = c->times[2];
    e->solve_reduced_system_time = c->times[3];
    e->back_substitution_time = c->times[4];
  }
  for (int k = 0; k < 5; ++k) c->times[k] = 0.0;
}

__device__ __forceinline__ povar_iteration* entry(LmCtl* c, povar_iteration* log, int capacity) {
  return c->log.count < capacity ? log + c->log.count : nullptr;
}

__device__ void fail(LmCtl* c, int status, int message, const LmConds& h) {
  c->status = status;
  c->message = message;
  set_cond(h.run, false);
  set_cond(h.lin, false);
  set_cond(h.restore, false);
}

__global__ void k_lm_stamp(unsigned long long* at) { *at = now_ns(); }

__global__ void k_lm_top(LmCtl* c, LmConds h) {
  c->t_it = now_ns();
  set_cond(h.lin, c->lin_next != 0);
}

__global__ void k_lm_begin(LmCtl* c, const double* __restrict__ trial_out, povar_options opt, int step,
                           povar_iteration* log, int capacity, LmConds h) {
  if (step == 1) {   // a new solve: everything but the stamps of its start and of its first cost evaluation
    const LmCtl keep = *c;
    *c = LmCtl{};
    c->t_start = keep.t_start;
    c->t_it = keep.t_it;
    c->stamp[0] = keep.stamp[0];
    c->stamp[1] = keep.stamp[1];
    c->status = POVAR_OK;
    c->termination[0] = c->termination[1] = 1;   // NO_CONVERGENCE
  }
  c->times[0] += seconds(c->stamp[0], c->stamp[1]);
  decode_cost(trial_out, &c->ri);
  c->lin_next = 0;
  if (!c->ri.is_numerically_valid) {   // CHECK(ri.is_numerically_valid), :312
    fail(c, POVAR_NUM_LINEARIZATION, LM_MSG_LINEARIZATION, h);
    return;
  }
  povar_iteration* e = entry(c, log, capacity);
  lm_begin(opt, step == 2, c->loop, c->log, e, c->ri);
  stamp_entry(c, e);
  const int max_iter = step == 2 ? opt.max_num_iterations_step_2 : opt.max_num_iterations_step_1;
  c->lin_next = 1;
  set_cond(h.run, c->loop.it <= max_iter);
}

__global__ void k_lm_decide(LmCtl* c, const double* __restrict__ trial_out, const SeriesCtl* __restrict__ sctl,
                            povar_options opt, int step, int power, povar_iteration* log, int capacity, LmConds h) {
  const unsigned long long* s = c->stamp;
  c->times[2] += seconds(s[0], s[1]);
  c->times[3] += seconds(s[1], s[2]);
  c->times[4] += seconds(s[2], s[3]);
  c->times[0] += seconds(s[3], s[4]);
  if (c->lin_next) {   // this trial linearised first (Engine::trial with a deferred linearisation check)
    c->lin_next = 0;
    c->times[1] += seconds(s[6], s[7]);
    if (trial_out[9] > 0) {
      fail(c, POVAR_NUM_LINEARIZATION, LM_MSG_LINEARIZATION, h);
      return;
    }
  }
  const int lin_it = sctl->iterations;
  if (sctl->peer_timeout) {
    fail(c, POVAR_ERR_NCCL, LM_MSG_PEER_TIMEOUT, h);
    return;
  }
  if (power) {
    c->power_terms += lin_it;
    c->power_time += c->times[3];
  }
  povar_residual_info ri2;
  decode_cost(trial_out, &ri2);
  povar_iteration* e = entry(c, log, capacity);
  const bool accepted = lm_trial_step(opt, step == 2, c->loop, c->log, e, c->ri, ri2, sctl->nonfinite != 0,
                                      trial_out[8], lin_it, nullptr);
  stamp_entry(c, e);
  if (accepted) c->ri = ri2;   // the state is the one this trial evaluated
  const int max_iter = step == 2 ? opt.max_num_iterations_step_2 : opt.max_num_iterations_step_1;
  const bool run = c->loop.stop == LM_RUNNING && c->loop.it <= max_iter;
  c->lin_next = accepted && run;
  set_cond(h.run, run);
  set_cond(h.restore, !accepted);
}

__global__ void k_lm_end_step(LmCtl* c, int step, int max_iter, unsigned long long ok) {
  if (c->status == POVAR_OK) {
    c->termination[step - 1] = c->loop.stop == LM_STOP_FUNCTION_TOLERANCE ? 0 : 1;
    c->message = c->loop.stop == LM_STOP_FUNCTION_TOLERANCE ? LM_MSG_FUNCTION_TOLERANCE
                 : c->loop.stop == LM_STOP_MAX_DAMPING      ? LM_MSG_MAX_DAMPING
                                                             : LM_MSG_MAX_ITERATIONS;
    c->message_iterations = max_iter;
  }
  if (step == 1) {
    c->t_step1 = now_ns();
    set_cond(ok, c->status == POVAR_OK);
  }
}

__device__ int put(char* out, int at, const char* s) {
  while (*s && at < 255) out[at++] = *s++;
  return at;
}

__global__ void k_lm_finish(LmCtl* c, int capacity, povar_solve_summary* sum, int* status) {
  const unsigned long long t = now_ns();
  char* raw = reinterpret_cast<char*>(sum);
  for (size_t i = 0; i < sizeof(povar_solve_summary); ++i) raw[i] = 0;
  sum->num_iterations = c->log.count < capacity ? c->log.count : capacity;
  sum->termination_type_step_1 = c->termination[0];
  sum->termination_type_step_2 = c->termination[1];
  sum->total_time = seconds(c->t_start, t);
  sum->step1_time = seconds(c->t_start, c->t_step1);
  sum->step2_time = sum->total_time - sum->step1_time;
  sum->power_terms = c->power_terms;
  sum->power_series_time = c->power_time;
  sum->num_successful_steps = c->log.num_successful - 1;
  sum->num_unsuccessful_steps = c->log.num_unsuccessful;
  sum->initial_cost = c->log.initial_cost;
  sum->final_cost = c->log.final_cost;
  char* m = sum->message;
  switch (c->message) {   // the host driver's wording; the function-tolerance message without its %g figures
    case LM_MSG_LINEARIZATION:
      put(m, 0, "did not expect numerical failure during linearization");
      break;
    case LM_MSG_PEER_TIMEOUT:
      put(m, 0, "peer exchange of the camera sums timed out (a rank is gone?)");
      break;
    case LM_MSG_FUNCTION_TOLERANCE:
      put(m, 0, "Function tolerance reached.");
      break;
    case LM_MSG_MAX_DAMPING:
      put(m, 0, "Solver did not converge and reached maximum damping lambda");
      break;
    case LM_MSG_MAX_ITERATIONS: {
      int at = put(m, 0, "Solver did not converge after maximum number of ");
      char digits[12];
      int n = 0;
      long long v = c->message_iterations;
      if (v < 0) {
        at = put(m, at, "-");
        v = -v;
      }
      do {
        digits[n++] = static_cast<char>('0' + v % 10);
        v /= 10;
      } while (v > 0 && n < 11);
      while (n > 0 && at < 255) m[at++] = digits[--n];
      put(m, at, " iterations");
      break;
    }
    default:
      break;
  }
  *status = c->status;
}

__global__ void k_lm_clip(povar_solve_summary* sum, int max_iterations) {
  const int cap = max_iterations > 0 ? max_iterations : 0;
  if (sum->num_iterations > cap) sum->num_iterations = cap;
}

__global__ void k_chol_status(const int* __restrict__ info, SeriesCtl* ctl) {
  ctl->done = 1;
  ctl->iterations = 0;   // the reference reports 0 linear solver iterations for the direct solve
  ctl->nonfinite = *info != 0 ? 1 : 0;   // not positive definite: an invalid step
  ctl->peer_timeout = 0;
  ctl->term = 0;
}

__global__ void k_cg_loop(SeriesCtl* ctl, int* base, int max_it, int advance, unsigned long long handle) {
  if (advance) *base += 10;
  else *base = 0;
  set_cond(handle, !ctl->done && *base < max_it);
}

}  // namespace

void launch_lm_stamp(unsigned long long* at, const LaunchCfg& lc) {
  k_lm_stamp<<<1, 1, 0, lc.stream>>>(at);
  count(lc);
}

void launch_lm_top(LmCtl* ctl, const LmConds& h, const LaunchCfg& lc) {
  k_lm_top<<<1, 1, 0, lc.stream>>>(ctl, h);
  count(lc);
}

void launch_lm_begin(LmCtl* ctl, const double* trial_out, const povar_options& opt, int step, povar_iteration* log,
                     int capacity, const LmConds& h, const LaunchCfg& lc) {
  k_lm_begin<<<1, 1, 0, lc.stream>>>(ctl, trial_out, opt, step, log, capacity, h);
  count(lc);
}

void launch_lm_decide(LmCtl* ctl, const double* trial_out, const SeriesCtl* sctl, const povar_options& opt, int step,
                      bool power, povar_iteration* log, int capacity, const LmConds& h, const LaunchCfg& lc) {
  k_lm_decide<<<1, 1, 0, lc.stream>>>(ctl, trial_out, sctl, opt, step, power ? 1 : 0, log, capacity, h);
  count(lc);
}

void launch_lm_end_step(LmCtl* ctl, int step, int max_iter, unsigned long long ok, const LaunchCfg& lc) {
  k_lm_end_step<<<1, 1, 0, lc.stream>>>(ctl, step, max_iter, ok);
  count(lc);
}

void launch_lm_finish(LmCtl* ctl, int capacity, povar_solve_summary* summary, int* status, const LaunchCfg& lc) {
  k_lm_finish<<<1, 1, 0, lc.stream>>>(ctl, capacity, summary, status);
  count(lc);
}

void launch_lm_clip(povar_solve_summary* summary, int max_iterations, const LaunchCfg& lc) {
  k_lm_clip<<<1, 1, 0, lc.stream>>>(summary, max_iterations);
  count(lc);
}

void launch_chol_status(const int* info, SeriesCtl* ctl, const LaunchCfg& lc) {
  k_chol_status<<<1, 1, 0, lc.stream>>>(info, ctl);
  count(lc);
}

void launch_cg_loop(SeriesCtl* ctl, int* base, int max_it, bool advance, unsigned long long handle, const LaunchCfg& lc) {
  k_cg_loop<<<1, 1, 0, lc.stream>>>(ctl, base, max_it, advance ? 1 : 0, handle);
  count(lc);
}

}  // namespace povar
