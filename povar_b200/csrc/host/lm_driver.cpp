// Host C++ driver: the Levenberg-Marquardt / VarPro outer loops of both steps, on top of the
// C ABI only (it is a client of include/povar_b200.h like any other caller).
//
// Control flow follows /root/reference/src/rootba_povar/solver/bal_bundle_adjustment.cpp:
//   step 1  optimize_lm_ours_pOSE       :252-542   (accept iff f_diff > 0, :443-445)
//   bridge  create_homogeneous_landmark :544-553
//   step 2  optimize_homogeneous_joint  :557-843   (accept iff l_diff > 0 and rho > min_relative_decrease)
// including its quirks (SURVEY F6/H1): lambda update uses rho = f_diff / l_diff in both steps,
// iteration counters count trials, the function-tolerance test compares with the previous LIST
// entry (which may be a rejected trial), step 2 restarts lambda from the initial radius.
//
// What is NOT repeated: the reference evaluates the cost again at the top of the iteration that follows an
// accepted step (:306-312, :608-612) -- on the state it has just evaluated.  The cost kernels have fixed
// reduction trees, so that second evaluation returns the same bits; the accepted trial's ResidualInfo is
// reused instead.  Every trial costs one host synchronisation (Engine::trial).
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../engine.h"
#include "../lm_step.h"

namespace povar {
const PhaseTimes& handle_times(povar_handle* h);
void handle_reset_times(povar_handle* h);
int handle_rank(povar_handle* h);
// the library's own driver takes two shortcuts behind the per-method ABI (engine.h): a linearisation whose
// failure flag is read with the next trial, and a whole trial (solve, backup, apply, normalise, cost) with one
// host synchronisation
int handle_linearize_deferred(povar_handle* h, bool joint, double alpha);
int handle_trial(povar_handle* h, bool joint, double alpha, double lambda, int32_t* iterations, double* l_diff,
                 povar_residual_info* ri);
}  // namespace povar

namespace {

using Clock = std::chrono::steady_clock;

double seconds_since(Clock::time_point t0) {
  return std::chrono::duration<double>(Clock::now() - t0).count();
}

// the log of a solve: the non-timing columns are lm_log_push's (lm_step.h), the times are the host clock's and the
// events'
struct Log {
  povar_iteration* out;
  int32_t capacity;
  povar::LmLog st;

  void stamp(povar_handle* h, povar_iteration* e, double it_time, double cum_time) {
    const povar::PhaseTimes& t = povar::handle_times(h);
    if (e) {
      e->iteration_time = it_time;
      e->cumulative_time = cum_time;
      e->residual_evaluation_time = t.residual;
      e->jacobian_evaluation_time = t.linearize;
      e->prepare_time = t.prepare;
      e->solve_reduced_system_time = t.reduced_solve;
      e->back_substitution_time = t.back_substitution;
    }
    povar::handle_reset_times(h);
  }
  // the entry the next push writes (nullptr: no room)
  povar_iteration* next() { return (st.count < capacity && out) ? out + st.count : nullptr; }
};

struct StepResult {
  int termination = 1;   // NO_CONVERGENCE
  std::string message;
  int rc = POVAR_OK;
};

// one LM loop; `joint` selects step 2.  The decisions are lm_step.h's (shared with the device-side solve).
StepResult run_step(povar_handle* h, const povar_options& opt, bool joint, Log& log,
                    Clock::time_point t_total, bool verbose, long long* power_terms,
                    double* power_time) {
  StepResult res;
  const int max_iter = joint ? opt.max_num_iterations_step_2 : opt.max_num_iterations_step_1;
  const bool power = povar::lm_power_step(opt, joint);
  povar::LmLoop s;
  s.lambda = 1.0 / opt.initial_trust_region_radius;
  bool first = true;

  auto cost = [&](povar_residual_info* ri) {
    return joint ? povar_cost_homogeneous(h, ri) : povar_cost_pose(h, opt.alpha, ri);
  };

  povar_residual_info ri_accepted;   // cost of the state an accepted trial left behind
  bool have_accepted = false;
  for (int it = 0; it <= max_iter && s.stop == povar::LM_RUNNING;) {
    Clock::time_point t_it = Clock::now();
    povar_residual_info ri;
    if (!joint && first) {
      res.rc = povar_init_varproj(h, opt.alpha);   // :302-304
      if (res.rc != POVAR_OK) return res;
    }
    first = false;
    if (have_accepted) {
      ri = ri_accepted;   // the state is the one that trial evaluated
    } else {
      res.rc = cost(&ri);
      if (res.rc != POVAR_OK) return res;
    }
    if (verbose) {
      std::printf("Iteration %d, error: %.4e (mean res: %.2f, num: %lld), error valid: %.4e (num: %lld)\n",
                  it, ri.error_all, ri.num_obs_all > 0 ? ri.residual_sum_all / ri.num_obs_all : 0.0,
                  static_cast<long long>(ri.num_obs_all), ri.error_valid,
                  static_cast<long long>(ri.num_obs_valid));
    }
    if (!ri.is_numerically_valid) {   // CHECK(ri.is_numerically_valid), :312
      res.rc = POVAR_NUM_LINEARIZATION;
      res.message = "did not expect numerical failure during linearization";
      return res;
    }
    if (it == 0) {   // iteration 0 is just error evaluation and logging, :316-328
      povar_iteration* e = log.next();
      povar::lm_begin(opt, joint, s, log.st, e, ri);
      log.stamp(h, e, seconds_since(t_it), seconds_since(t_total));
      it = s.it;
      continue;
    }
    res.rc = povar::handle_linearize_deferred(h, joint, opt.alpha);
    if (res.rc != POVAR_OK) {
      res.message = povar_last_error(h);
      return res;
    }

    for (int j = 0; it <= max_iter && s.stop == povar::LM_RUNNING; ++j) {
      if (j > 0) {
        if (verbose) std::printf("Iteration %d, backtracking\n", it);
        t_it = Clock::now();
      }
      int32_t lin_it = 0;
      double l_diff = 0.0;
      povar_residual_info ri2;
      // solve, backup, apply, (step 2) normalise, cost: :346-420 / :655-720, one synchronisation
      const int src = povar::handle_trial(h, joint, opt.alpha, s.lambda, &lin_it, &l_diff, &ri2);
      if (src < 0 || src == POVAR_NUM_LINEARIZATION) {
        res.rc = src;
        res.message = povar_last_error(h);
        return res;
      }
      if (power) {
        *power_terms += lin_it;
        *power_time += povar::handle_times(h).reduced_solve;
      }
      const double lambda = s.lambda;   // of this trial (printed)
      const bool nonfinite = src == POVAR_NUM_NONFINITE_INC;
      povar::LmEval ev;
      povar_iteration* e = log.next();
      const bool accepted = povar::lm_trial_step(opt, joint, s, log.st, e, ri, ri2, nonfinite, l_diff, lin_it, &ev);
      log.stamp(h, e, seconds_since(t_it), seconds_since(t_total));
      it = s.it;
      if (verbose) {
        if (nonfinite) {
          std::printf("\t[Invalid] Numeric issues when computing increment (contains NaNs), lambda: %.1e, cg_iter: %d\n",
                      lambda, lin_it);
        } else {
          if (ri2.is_numerically_valid) {
            std::printf("\t[EVAL] f_diff %.4e l_diff %.4e ri1 %.4e ri2 %.4e\n", ev.f_diff, ev.l_diff,
                        ri.error_valid, ri2.error_valid);
          }
          std::printf("\t[%s] error: %.4e (num valid: %lld), lambda: %.1e, cg_iter: %d, it_time: %.3fs, total_time: %.3fs\n",
                      accepted ? "Success" : (ev.valid ? "Reject" : "Invalid"), ri2.error_all,
                      static_cast<long long>(ri2.num_obs_valid), lambda, lin_it, seconds_since(t_it),
                      seconds_since(t_total));
        }
      }
      if (accepted) {
        ri_accepted = ri2;
        have_accepted = true;
        break;   // stop inner lm loop
      }
      // the reference does not apply a non-finite increment; here it was applied to the copy the backup protects
      res.rc = povar_restore(h, joint ? POVAR_STATE_JOINT : POVAR_STATE_POSE);
      if (res.rc != POVAR_OK) return res;
    }
  }
  if (s.stop == povar::LM_STOP_FUNCTION_TOLERANCE) {
    res.termination = 0;
    char buf[160];
    std::snprintf(buf, sizeof(buf), "Function tolerance reached. |cost_change|/cost: %g <= %g", s.ftol_ratio,
                  opt.function_tolerance);
    res.message = buf;
  } else if (s.stop == povar::LM_STOP_MAX_DAMPING) {
    res.termination = 1;
    res.message = "Solver did not converge and reached maximum damping lambda";
  } else {
    res.termination = 1;
    char buf[128];
    std::snprintf(buf, sizeof(buf), "Solver did not converge after maximum number of %d iterations", max_iter);
    res.message = buf;
  }
  return res;
}

}  // namespace

extern "C" int povar_bundle_adjust(povar_handle* h, const povar_options* opt_in, povar_iteration* iterations,
                                   int32_t max_iterations, povar_solve_summary* summary) {
  if (!h || !opt_in) return POVAR_ERR_INVALID;
  const povar_options opt = *opt_in;
  // check_options, bal_bundle_adjustment.cpp:228-250
  if (!(opt.min_trust_region_radius <= opt.initial_trust_region_radius) ||
      !(opt.initial_trust_region_radius <= opt.max_trust_region_radius) || opt.jacobi_scaling_epsilon < 0) {
    return POVAR_ERR_INVALID;
  }
  const bool verbose = opt.verbosity_level >= 2 && povar::handle_rank(h) == 0;
  Log log{iterations, iterations ? max_iterations : 0};
  long long power_terms = 0;
  double power_time = 0.0;
  povar::handle_reset_times(h);
  const Clock::time_point t_total = Clock::now();

  StepResult s1 = run_step(h, opt, false, log, t_total, verbose, &power_terms, &power_time);
  const double t_step1 = seconds_since(t_total);
  StepResult s2;
  if (s1.rc == POVAR_OK) {
    if (verbose) std::printf("Step 1: %s\n", s1.message.c_str());
    s1.rc = povar_to_homogeneous(h);
  }
  if (s1.rc == POVAR_OK) {
    s2 = run_step(h, opt, true, log, t_total, verbose, &power_terms, &power_time);
    if (verbose && s2.rc == POVAR_OK) std::printf("Step 2: %s\n", s2.message.c_str());
  }
  const double t_all = seconds_since(t_total);

  if (summary) {
    std::memset(summary, 0, sizeof(*summary));
    summary->num_iterations = std::min(log.st.count, log.capacity);
    summary->termination_type_step_1 = s1.termination;
    summary->termination_type_step_2 = s2.termination;
    summary->total_time = t_all;
    summary->step1_time = t_step1;
    summary->step2_time = t_all - t_step1;
    summary->power_terms = power_terms;
    summary->power_series_time = power_time;
    // finish_solve (:97-159): iteration 0 entries count as successful; the reference subtracts one
    summary->num_successful_steps = log.st.num_successful - 1;
    summary->num_unsuccessful_steps = log.st.num_unsuccessful;
    summary->initial_cost = log.st.initial_cost;
    summary->final_cost = log.st.final_cost;
    const std::string& msg = (s1.rc != POVAR_OK) ? s1.message : s2.message;
    std::snprintf(summary->message, sizeof(summary->message), "%s", msg.c_str());
  }
  if (s1.rc != POVAR_OK) return s1.rc;
  return s2.rc;
}
