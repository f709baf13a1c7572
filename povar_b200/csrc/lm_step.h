// The scalar decision of one LM trial and the log entry it makes: ONE copy, used by the host driver
// (host/lm_driver.cpp) and by the decision kernels of the device-side solve (kernels_lm.cu).
//
// The arithmetic is written so that the host and the device compute the same bits: plain IEEE operations in the
// order the reference's loops use (kernels_lm.cu is compiled with -fmad=false, the host compiler contracts nothing
// without FMA hardware flags).  The one exception is the cube of the lambda update, std::pow(2 rho - 1, 3) in the
// reference: on the host a libm call, on the device the correctly rounded cube (lm_cube).  The two can differ in
// the last bit of a trust-region radius.
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>

#include "../../include/povar_b200.h"

#if defined(__CUDACC__)
#define POVAR_HD __host__ __device__
#else
#define POVAR_HD
#endif

namespace povar {

// what summary.iterations of the reference holds as far as the LM loops read it
// (bal_bundle_adjustment.cpp:75-78, ba_log_utils.cpp:128-147, finish_solve :97-159)
struct LmLog {
  int32_t count = 0;
  // cost (all / valid) of summary.iterations.back(): cost_change of a trial is measured against the previous LIST entry
  double back_cost = 0.0, back_cost_valid = 0.0;
  // last logged values (for failed trials the log repeats them)
  double logged_cost = 0.0, logged_cost_valid = 0.0;
  double logged_res_mean = 0.0, logged_res_valid_mean = 0.0;
  int64_t logged_valid = 0;
  int32_t num_successful = 0, num_unsuccessful = 0;
  double initial_cost = 0.0, final_cost = 0.0;
};

// state of one LM loop between two trials
enum LmStop { LM_RUNNING = 0, LM_STOP_FUNCTION_TOLERANCE = 1, LM_STOP_MAX_DAMPING = 2 };
struct LmLoop {
  double lambda = 0.0, vee = 0.0;
  int32_t it = 0;        // number of the next log entry of this step (iteration counters count trials)
  int32_t stop = LM_RUNNING;
  double ftol_ratio = 0.0;   // |cost_change| / cost when stop == LM_STOP_FUNCTION_TOLERANCE
};

// what the host prints about a trial
struct LmEval {
  double f_diff = 0.0, l_diff = 0.0, rho = 0.0;
  bool valid = false;
};

POVAR_HD inline double lm_max(double a, double b) { return (a < b) ? b : a; }   // std::max, NaN behaviour included

POVAR_HD inline double lm_nan() {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(0x7ff8000000000000LL);
#else
  return std::nan("");
#endif
}

// (2 rho - 1)^3 of the lambda update (bal_bundle_adjustment.cpp:461-463)
POVAR_HD inline double lm_cube(double t) {
#ifdef __CUDA_ARCH__
  // double-double product rounded once: t^2 = p + pe and p t = h + he exactly, (p + pe) t = h + (he + pe t)
  const double p = __dmul_rn(t, t);
  const double pe = fma(t, t, -p);
  const double h = __dmul_rn(p, t);
  const double he = fma(p, t, -h);
  return __dadd_rn(h, fma(pe, t, he));
#else
  return std::pow(t, 3);
#endif
}

// whether the solver of a step is a power series (its iterations count as power_terms)
inline bool lm_power_step(const povar_options& opt, bool joint) {
  return joint ? opt.solver_type_step_2 == POVAR_RIPOBA
               : (opt.solver_type_step_1 == POVAR_POWER_VARPROJ ||
                  opt.solver_type_step_1 == POVAR_POWER_SCHUR_COMPLEMENT);
}

// one log entry without the times: entry `e` (nullptr: no room) gets the non-timing columns
POVAR_HD inline void lm_log_push(LmLog& L, povar_iteration* e, int step, int it, bool valid, bool successful,
                                 double trial_cost, const povar_residual_info* ri, double rel, double radius,
                                 int lin_it) {
  if (successful || L.count == 0 || (it == 0)) {
    if (ri) {
      L.logged_cost = ri->error_all;
      L.logged_cost_valid = ri->error_valid;
      L.logged_valid = ri->num_obs_valid;
      L.logged_res_mean = ri->num_obs_all > 0 ? ri->residual_sum_all / static_cast<double>(ri->num_obs_all) : 0.0;
      L.logged_res_valid_mean =
          ri->num_obs_valid > 0 ? ri->residual_sum_valid / static_cast<double>(ri->num_obs_valid) : 0.0;
    }
  }
  L.back_cost = ri ? ri->error_all : 0.0;   // an "Invalid" trial leaves a default-constructed cost
  L.back_cost_valid = ri ? ri->error_valid : 0.0;
  if (L.count == 0) L.initial_cost = L.logged_cost;
  if (successful) {
    ++L.num_successful;
    L.final_cost = L.logged_cost;
  } else {
    ++L.num_unsuccessful;
  }
  if (e) {
    e->step = step;
    e->iteration = it;
    e->step_is_valid = valid ? 1 : 0;
    e->step_is_successful = successful ? 1 : 0;
    e->cost = L.logged_cost;
    e->cost_valid = L.logged_cost_valid;
    e->trial_cost = trial_cost;
    e->num_obs_valid = L.logged_valid;
    e->relative_decrease = successful ? rel : 0.0;
    e->trust_region_radius = radius;
    e->linear_solver_iterations = lin_it;
    e->residual_mean = L.logged_res_mean;
    e->residual_valid_mean = L.logged_res_valid_mean;
  }
  ++L.count;
}

// iteration 0 of a step: error evaluation and logging only (:316-328)
POVAR_HD inline void lm_begin(const povar_options& opt, bool joint, LmLoop& s, LmLog& L, povar_iteration* e,
                              const povar_residual_info& ri) {
  s.lambda = 1.0 / opt.initial_trust_region_radius;
  s.vee = opt.initial_vee;
  s.stop = LM_RUNNING;
  s.ftol_ratio = 0.0;
  lm_log_push(L, e, joint ? 2 : 1, 0, true, true, ri.error_all, &ri, 0.0, 1.0 / s.lambda, 0);
  s.it = 1;
}

// What the loop does with the results of one trial (:346-542 / :655-843): `ri` is the cost of the state the trial
// started from, `ri2` the trial's; `nonfinite` the solve's increment had NaN / Inf (:362-401).  Updates lambda / vee,
// logs entry `e`, advances the iteration and sets s.stop.  Returns true when the step is accepted (the caller keeps
// the state and linearises again); otherwise the caller restores the backup.
POVAR_HD inline bool lm_trial_step(const povar_options& opt, bool joint, LmLoop& s, LmLog& L, povar_iteration* e,
                                   const povar_residual_info& ri, const povar_residual_info& ri2, bool nonfinite,
                                   double l_diff, int lin_it, LmEval* ev) {
  const int step = joint ? 2 : 1;
  const double min_lambda = 1.0 / opt.max_trust_region_radius;
  const double max_lambda = 1.0 / opt.min_trust_region_radius;
  if (nonfinite) {   // the reference does not apply such an increment: "Invalid"
    s.lambda = s.vee * s.lambda;
    s.vee *= opt.vee_factor;
    lm_log_push(L, e, step, s.it, false, false, lm_nan(), nullptr, 0.0, 1.0 / s.lambda, lin_it);
    ++s.it;
    if (s.lambda > max_lambda) s.stop = LM_STOP_MAX_DAMPING;
    return false;
  }
  bool valid = false, successful = false;
  double rho = 0.0, f_diff = 0.0;
  if (ri2.is_numerically_valid) {
    switch (opt.optimized_cost) {   // compute_cost_decrease, :163-176
      case POVAR_COST_ERROR_VALID:
        f_diff = ri.error_valid - ri2.error_valid;
        break;
      case POVAR_COST_ERROR_VALID_AVG:
        f_diff = (ri.num_obs_valid > 0 ? ri.error_valid / ri.num_obs_valid : 0.0) -
                 (ri2.num_obs_valid > 0 ? ri2.error_valid / ri2.num_obs_valid : 0.0);
        l_diff /= static_cast<double>(ri.num_obs_valid);
        break;
      default:
        f_diff = ri.error_all - ri2.error_all;
    }
    rho = f_diff / l_diff;
    if (joint) {   // :742-745
      valid = l_diff > 0;
      successful = valid && rho > opt.min_relative_decrease;
    } else {       // :442-445
      valid = true;
      successful = f_diff > 0;
    }
  }
  if (ev) {
    ev->f_diff = f_diff;
    ev->l_diff = l_diff;
    ev->rho = rho;
    ev->valid = valid;
  }
  if (successful) {
    s.lambda *= lm_max(1.0 / 3, 1 - lm_cube(2 * rho - 1));   // :461-463
    s.lambda = lm_max(min_lambda, s.lambda);
    s.vee = opt.initial_vee;
    const double prev_cost = L.back_cost, prev_cost_valid = L.back_cost_valid;
    lm_log_push(L, e, step, s.it, true, true, ri2.error_all, &ri2, rho, 1.0 / s.lambda, lin_it);
    ++s.it;
    // function_tolerance_reached (:179-205): cost_change against the previous list entry
    double cost_now, change;
    if (opt.optimized_cost == POVAR_COST_ERROR) {
      cost_now = ri2.error_all;
      change = fabs(prev_cost - ri2.error_all);
    } else {
      cost_now = ri2.error_valid;
      change = fabs(prev_cost_valid - ri2.error_valid);   // |cost_change.valid.error|, :190-194
    }
    if (change <= opt.function_tolerance * cost_now) {
      s.stop = LM_STOP_FUNCTION_TOLERANCE;
      s.ftol_ratio = change / cost_now;
    }
    return true;
  }
  s.lambda = s.vee * s.lambda;   // :498-499
  s.vee *= opt.vee_factor;
  lm_log_push(L, e, step, s.it, valid, false, ri2.error_all, &ri2, 0.0, 1.0 / s.lambda, lin_it);
  ++s.it;
  if (s.lambda > max_lambda) s.stop = LM_STOP_MAX_DAMPING;
  return false;
}

}  // namespace povar
