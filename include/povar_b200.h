/*
 * povar_b200.h -- C ABI of the B200-native PoVar hot path (libpovar_b200.so).
 *
 * This is the drop-in boundary for the reference's `Linearizor<Scalar>` plugin
 * interface (/root/reference/src/rootba_povar/solver/linearizor.hpp:47-82) and for
 * the two-step driver built on it (solver/bal_bundle_adjustment.cpp:848-876).
 * The reference keeps cameras/landmarks in host structs and mutates them through
 * the Linearizor; here the state lives in HBM behind an opaque handle, so the
 * caller-side backup/restore/normalise steps of the reference move behind the
 * ABI as well.  Every entry point cites the reference interface it replaces.
 *
 * Conventions
 *   - plain C types, host pointers owned by the caller, sizes in elements;
 *   - return 0 = OK; < 0 = CUDA / NCCL / usage error (text via povar_last_error);
 *     > 0 = numerical condition (POVAR_NUM_*), which the reference surfaces as a
 *     non-finite increment or a failed CHECK;
 *   - one driving host thread per handle; one handle per GPU (one process per GPU
 *     when sharded, landmarks partitioned across ranks, cameras replicated);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     returns POVAR_ERR_NO_DEVICE.
 */
#ifndef POVAR_B200_H_
#define POVAR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POVAR_ABI_VERSION 3

/* status codes */
enum {
  POVAR_OK = 0,
  POVAR_NUM_NONFINITE_INC = 1,     /* increment has NaN/Inf: "Invalid" step, bal_bundle_adjustment.cpp:362-401 */
  POVAR_NUM_LINEARIZATION = 2,     /* non-finite residual/Jacobian: the reference CHECK-aborts, linearizor_power_varproj.cpp:59 */
  POVAR_ERR_INVALID = -1,
  POVAR_ERR_CUDA = -2,
  POVAR_ERR_NCCL = -3,
  POVAR_ERR_NO_DEVICE = -4,
  POVAR_ERR_IO = -5,
  POVAR_ERR_UNSUPPORTED = -6
};

/* SolverOptions::SolverType / SolverTypeRiemannian, bal/solver_options.hpp:60-69 (same order) */
enum { POVAR_PCG = 0, POVAR_POWER_SCHUR_COMPLEMENT = 1, POVAR_POWER_VARPROJ = 2, POVAR_CHOLESKY = 3 };
enum { POVAR_RIPOBA = 0, POVAR_RIPCG = 1 };
/* BalResidualOptions::RobustNorm, bal/bal_residual_options.hpp:44-48 */
enum { POVAR_NORM_NONE = 0, POVAR_NORM_HUBER = 1, POVAR_NORM_CAUCHY = 2 };
/* SolverOptions::OptimizedCost, bal/solver_options.hpp:48-53 */
enum { POVAR_COST_ERROR = 0, POVAR_COST_ERROR_VALID = 1, POVAR_COST_ERROR_VALID_AVG = 2 };
enum { POVAR_STATE_POSE = 0, POVAR_STATE_JOINT = 1 };

/* The fields of SolverOptions (bal/solver_options.hpp:88-307) that the path reads;
 * povar_options_default() fills the reference's CODE defaults (alpha 0.01,
 * power_sc_iterations 10, eta 0.01 ... -- not the README's). */
typedef struct povar_options {
  int32_t solver_type_step_1;          /* POVAR_POWER_VARPROJ */
  int32_t solver_type_step_2;          /* POVAR_RIPOBA */
  int32_t robust_norm;                 /* POVAR_NORM_NONE */
  int32_t optimized_cost;              /* POVAR_COST_ERROR */
  double huber_parameter;              /* 1.0 */
  double alpha;                        /* 0.01 */
  int32_t max_num_iterations_step_1;   /* 50 */
  int32_t max_num_iterations_step_2;   /* 50 */
  double min_relative_decrease;        /* 0 */
  double initial_trust_region_radius;  /* 1e4 */
  double min_trust_region_radius;      /* 1e-32 */
  double max_trust_region_radius;      /* 1e16 */
  int32_t min_linear_solver_iterations; /* 0 */
  int32_t max_linear_solver_iterations; /* 500 */
  double eta;                          /* 1e-2 */
  double r_tolerance;                  /* -1 */
  double jacobi_scaling_epsilon;       /* 0 => sqrt(1e-10) */
  double function_tolerance;           /* 1e-6 */
  int32_t power_sc_iterations;         /* 10 */
  int32_t verbosity_level;             /* 2 */
  double initial_vee;                  /* 2 */
  double vee_factor;                   /* 2 */
} povar_options;

void povar_options_default(povar_options* opt);

/* One shard of a BAL problem in the reference's canonical order: landmark index,
 * then camera index ascending (std::map<cam,obs> per landmark, bal_problem.hpp:226;
 * pose_idx_ of landmark_block.hpp:104-108).  Image coordinates are the values AFTER
 * the loader's y flip (bal_problem.cpp:240). */
typedef struct povar_problem_desc {
  int32_t num_cams;        /* C, all cameras (replicated on every rank) */
  int32_t num_lms;         /* landmarks in this shard */
  int64_t num_obs;         /* observations in this shard */
  const int64_t* lm_ptr;   /* [num_lms+1] CSR offsets into obs_* */
  const int32_t* obs_cam;  /* [num_obs] camera index, ascending inside a landmark */
  const double* obs_uv;    /* [num_obs*2] */
  const double* cam_P;     /* [C*12] 3x4 camera matrices, row-major */
} povar_problem_desc;

/* An observation list that already lives in device memory, in any order (povar_create_device puts it into the
 * canonical order above on the GPU).  The handle takes the landmarks [lm_begin, lm_end) of it: landmark l becomes
 * local landmark l - lm_begin, exactly as in a shard handed to povar_create; the entries of other landmarks are
 * checked (index ranges, duplicate pairs) but otherwise ignored, so every rank may pass the whole list. */
typedef struct povar_device_problem_desc {
  int32_t num_cams;          /* C */
  int32_t num_lms;           /* landmarks of the whole problem: every obs_lm is < num_lms */
  int64_t num_obs;           /* entries of the three lists, in any order */
  int32_t lm_begin, lm_end;  /* landmarks of this handle: 0, num_lms on one GPU; povar_partition_landmarks bounds when sharded */
  const int32_t* obs_cam;    /* device [num_obs] */
  const int32_t* obs_lm;     /* device [num_obs] */
  const double* obs_uv;      /* device [num_obs*2], the convention of povar_problem_desc.obs_uv (after the y flip) */
  const double* cam_P;       /* device [C*12], row-major 3x4 */
  void* stream;              /* cudaStream_t on which the caller produced the arrays; NULL = legacy default stream */
} povar_device_problem_desc;

/* bal/residual_info.hpp:59-102 */
typedef struct povar_residual_info {
  int64_t num_obs_all;
  double error_all;
  double residual_sum_all;
  int64_t num_obs_valid;
  double error_valid;
  double residual_sum_valid;
  int32_t is_numerically_valid;
} povar_residual_info;

/* how ranks find each other when landmarks are sharded over several GPUs */
typedef struct povar_comm_desc {
  int32_t rank;
  int32_t world_size;
  int32_t device;            /* CUDA device ordinal for this rank */
  uint8_t nccl_id[128];      /* from povar_comm_unique_id() on rank 0, broadcast by the launcher */
} povar_comm_desc;

typedef struct povar_handle povar_handle;

/* ---------- host-side, no GPU needed ------------------------------------------------ */

int povar_abi_version(void);
/* sizeof of the public structs as this library was compiled, for bindings that mirror them (ctypes, cgo ...):
 * 0 povar_options, 1 povar_problem_desc, 2 povar_comm_desc, 3 povar_residual_info, 4 povar_iteration,
 * 5 povar_solve_summary, 6 povar_bal_data, 7 povar_ba_log_info, 8 povar_phase_times, 9 povar_device_problem_desc;
 * -1 for anything else */
int64_t povar_abi_sizeof(int32_t which);

/* BAL text reader for the 15-parameter format written by --create-dataset:
 * replaces BalProblem::load_bal_eccv (bal/bal_problem.cpp:182-303) up to and including
 * the y flip and the canonical re-ordering; duplicate (cam,lm) pairs are an error
 * (bal_problem.cpp:227).  Output arrays are malloc'ed; release with povar_bal_free. */
typedef struct povar_bal_data {
  int32_t num_cams;
  int32_t num_lms;
  int64_t num_obs;
  int64_t* lm_ptr;      /* [num_lms+1] */
  int32_t* obs_cam;     /* [num_obs] */
  double* obs_uv;       /* [num_obs*2] */
  double* cam_params;   /* [num_cams*15]: 12 matrix entries + f,k1,k2 (intrinsics unused by the path) */
} povar_bal_data;

int povar_bal_read(const char* path, povar_bal_data* out, char* err, size_t err_len);
void povar_bal_free(povar_bal_data* data);

/* --create-dataset (BalProblem::load_bal_varproj_space_matrix_write, bal/bal_problem.cpp:306-471): turns an
 * original BAL file (9 parameters per camera) into the 15-parameter file povar_bal_read loads -- same
 * observations, the first two rows of every camera matrix drawn from N(0,1), third row 0 0 0 1, f k1 k2
 * and the landmark block copied through, in the reference's text layout.  seed < 0 seeds from
 * std::random_device like the reference; seed >= 0 makes the output reproducible. */
int povar_bal_create_dataset(const char* input, const char* output, int64_t seed, char* err, size_t err_len);

/* canonical order of an unordered observation list: fills perm[num_obs] (indices into the
 * input, landmark-major, camera ascending) and lm_ptr[num_lms+1]; returns POVAR_ERR_INVALID on
 * a duplicate pair or an index out of range. */
int povar_canonical_order(int32_t num_cams, int32_t num_lms, int64_t num_obs, const int32_t* cam,
                          const int32_t* lm, int64_t* perm, int64_t* lm_ptr);

/* contiguous landmark ranges balanced by observation count: bounds[world_size+1]. */
int povar_partition_landmarks(int32_t num_lms, const int64_t* lm_ptr, int32_t world_size,
                              int32_t* bounds);

/* ---------- life cycle ---------------------------------------------------------------- */

int povar_comm_unique_id(uint8_t id[128]);
/* An id for ranks on ONE host that need no NCCL communicator: the handles swap their CUDA IPC handles through a
 * POSIX shared-memory rendezvous named by the id, and every reduction of the path (camera sums per power-series
 * term, cost scalars, Kronecker sums ...) goes over the peer-mapped buffers.  Unlike NCCL this allows several
 * ranks on the same device (povar_comm_desc.device may repeat), so the sharded arithmetic can be exercised on a
 * one-GPU box; povar_create fails if CUDA IPC / peer access is unavailable (there is nothing to fall back to).
 * Broadcast the id to the other ranks like an NCCL id.  The reference has no counterpart (single process). */
int povar_comm_host_id(uint8_t id[128]);
/* The NCCL communicator of a (nccl_id, rank) pair is made by the first povar_create that names it and
 * shared by every later handle of this process with the same descriptor (the reference makes a step-1
 * and a step-2 linearizor per solve, solver/linearizor.cpp:47-79; both ride on one communicator).
 * povar_comm_finalize destroys the cached communicators; call it after the last povar_destroy. */
int povar_comm_finalize(void);

/* replaces Linearizor<Scalar>::create / create_homogeneous (solver/linearizor.cpp:47-79):
 * uploads the shard, builds the camera-major index, allocates all device state.
 * comm == NULL means a single GPU (device 0). */
int povar_create(const povar_problem_desc* desc, const povar_options* opt,
                 const povar_comm_desc* comm, povar_handle** out);
/* povar_create from device-resident observations (povar_device_problem_desc), in any order.
 *   - The arrays are read after the work already enqueued on desc->stream: the handle's stream waits on an event
 *     recorded there; the caller's stream is not synchronised with the host.
 *   - The arrays are never written, and are no longer needed when the call returns.
 *   - The canonical order and the index are made on the device; the same observations give the same index arrays,
 *     and so the same results, as povar_canonical_order + povar_create of the same landmark range.
 *   - POVAR_ERR_INVALID (text via povar_last_error(NULL)): an index out of range, a duplicate (cam, lm) pair anywhere
 *     in the list, lm_begin > lm_end or a bound outside [0, num_lms], a pointer that is not device memory of the
 *     handle's device (comm->device, or 0).  POVAR_ERR_UNSUPPORTED: 2^31 or more entries.  POVAR_ERR_NO_DEVICE
 *     without a GPU. */
int povar_create_device(const povar_device_problem_desc* desc, const povar_options* opt,
                        const povar_comm_desc* comm, povar_handle** out);
/* povar_destroy frees the device state (back to the device's memory pool, which keeps it for the next handle) and
 * hands the handle's stream, events and 256 bytes of page-locked scratch to the next povar_create on the same device
 * instead of destroying them: a process keeps one such set per handle it ever had alive at the same time. */
void povar_destroy(povar_handle* h);
const char* povar_last_error(const povar_handle* h);

/* ---------- the Linearizor interface, in call order ------------------------------------ */

/* initialize_varproj_lm_pOSE (solver/linearizor_base.cpp:60-67; helper.cpp:75-114) */
int povar_init_varproj(povar_handle* h, double alpha);
/* compute_error_pOSE / compute_error_homogeneous (solver/linearizor_base.cpp:69-87) */
int povar_cost_pose(povar_handle* h, double alpha, povar_residual_info* out);
int povar_cost_homogeneous(povar_handle* h, povar_residual_info* out);
/* linearize_pOSE / linearize_projective_space_homogeneous
 * (solver/linearizor_power_varproj.cpp:44-110, solver/linearizor_sc.cpp:174-239) */
int povar_linearize_pose(povar_handle* h, double alpha);
int povar_linearize_homogeneous(povar_handle* h);
/* solve / solve_joint (solver/linearizor_power_varproj.cpp:113-243, linearizor_sc.cpp:91-325).
 * The increment stays on the device for the following apply; `inc` (C*12 resp. C*11 doubles)
 * may be NULL.  Returns POVAR_NUM_NONFINITE_INC if the increment is not finite. */
int povar_solve_pose(povar_handle* h, double lambda, double* inc, int32_t* linear_solver_iterations);
int povar_solve_joint(povar_handle* h, double lambda, double* inc, int32_t* linear_solver_iterations);
/* apply / apply_joint (solver/linearizor_power_varproj.cpp:245-308): back-substitution,
 * camera update, model cost change l_diff. */
int povar_apply_pose(povar_handle* h, double alpha, double* l_diff);
int povar_apply_joint(povar_handle* h, double* l_diff);

/* ---------- what the reference's caller does on host structs --------------------------- */

/* BalProblem::backup_pOSE/restore_pOSE/backup_joint/restore_joint (bal/bal_problem.cpp:647-708) */
int povar_backup(povar_handle* h, int32_t which);
int povar_restore(povar_handle* h, int32_t which);
/* create_homogeneous_landmark (solver/bal_bundle_adjustment.cpp:544-553) */
int povar_to_homogeneous(povar_handle* h);
/* per-trial normalisation P/|P|_F, X/X[3] (solver/bal_bundle_adjustment.cpp:700-705) */
int povar_normalize_joint(povar_handle* h);

/* cameras [C*12]; landmarks of this shard [num_lms*3] (POVAR_STATE_POSE) or [num_lms*4] (JOINT) */
int povar_get_state(povar_handle* h, int32_t which, double* cam_P, double* lms);
int povar_set_state(povar_handle* h, int32_t which, const double* cam_P, const double* lms);
/* The same in device memory of the handle's device, with the same layouts (set: POVAR_STATE_POSE writes w = 1).
 * Stream-ordered, no host synchronisation: the copies run after the work enqueued on `stream` (cudaStream_t, NULL =
 * legacy default stream) so far, and `stream` waits for them.  Either pointer may be NULL. */
int povar_get_state_device(povar_handle* h, int32_t which, double* cam_P, double* lms, void* stream);
int povar_set_state_device(povar_handle* h, int32_t which, const double* cam_P, const double* lms, void* stream);

/* ---------- the two-step driver -------------------------------------------------------- */

/* one entry per LM trial, the columns of ba_log.json the parity harness reads
 * (bal/ba_log.hpp:147-245, bal/ba_log_utils.cpp:99-160) */
typedef struct povar_iteration {
  int32_t step;                       /* 1 or 2 */
  int32_t iteration;                  /* restarts at 0 with step 2 */
  int32_t step_is_valid;
  int32_t step_is_successful;
  double cost;                        /* as logged: previous cost for failed trials */
  double cost_valid;
  double trial_cost;                  /* cost evaluated in this trial (NaN if none) */
  int64_t num_obs_valid;
  double relative_decrease;
  double trust_region_radius;
  int32_t linear_solver_iterations;
  double iteration_time;              /* seconds, host clock around the trial */
  double cumulative_time;
  /* phase times from CUDA events, seconds (solver/solver_summary.hpp:172-212) */
  double residual_evaluation_time;
  double jacobian_evaluation_time;    /* linearize_* */
  double prepare_time;                /* solve: everything before the reduced solve */
  double solve_reduced_system_time;   /* power series / PCG / Cholesky */
  double back_substitution_time;      /* apply_* */
  /* mean |r| per observation, all / valid, as logged (repeated for failed trials): residual_block_mean and
   * residual_block_valid_mean of the reference's log (bal/ba_log_utils.cpp:116-117) */
  double residual_mean;
  double residual_valid_mean;
} povar_iteration;

typedef struct povar_solve_summary {
  int32_t num_iterations;             /* entries written to `iterations` */
  int32_t termination_type_step_1;    /* 0 CONVERGENCE, 1 NO_CONVERGENCE (solver_summary.hpp) */
  int32_t termination_type_step_2;
  int32_t num_successful_steps;
  int32_t num_unsuccessful_steps;
  double initial_cost;
  double final_cost;
  double total_time;                  /* seconds, both steps (the reference's timing.optimize) */
  double step1_time;
  double step2_time;
  int64_t power_terms;                /* sum of linear_solver_iterations over power-series solves */
  double power_series_time;           /* device seconds spent in them */
  char message[256];
} povar_solve_summary;

/* bundle_adjust_manual (solver/bal_bundle_adjustment.cpp:848-876): step 1 (pOSE LM/VarPro loop,
 * :252-542), conversion to homogeneous (:544-553), step 2 (Riemannian LM loop, :557-843) on the
 * state held by the handle.  `iterations` has room for `max_iterations` entries. */
int povar_bundle_adjust(povar_handle* h, const povar_options* opt, povar_iteration* iterations,
                        int32_t max_iterations, povar_solve_summary* summary);

/* povar_bundle_adjust, enqueued: the same two-step solve on the state held by the handle, ordered after the work
 * enqueued on `stream` (cudaStream_t, NULL = legacy default stream) so far; `stream` waits for it.  No host
 * synchronisation, nothing printed.  `iterations` (room for max_iterations entries; may be NULL when max_iterations
 * is 0), `summary` and `status` are device memory of the handle's device, written when the solve ends: *status =
 * what povar_bundle_adjust returns for the same handle, state and options.
 * Both LM loops run on the device, with the host driver's decisions (the same code) and log columns; the times
 * come from the GPU's global timer, and the function-tolerance message ends after "Function tolerance reached.".
 * The radius update's cube is correctly rounded on the device, so a trust-region radius may differ from the host
 * driver's in the last bit.  The first call with given options (and debug settings) builds and instantiates one
 * CUDA graph for the solve; later calls with byte-identical options only launch it.  Not advanced by it:
 * povar_get_timings, povar_launch_count.
 * POVAR_ERR_INVALID: the checks of povar_bundle_adjust, max_iterations < 0, an output pointer that is not device
 * memory of the handle's device.  POVAR_ERR_UNSUPPORTED: a sharded handle whose reductions go through ncclAllReduce
 * (povar_peer_exchange_active(h) == 0 with more than one rank). */
int povar_bundle_adjust_async(povar_handle* h, const povar_options* opt, povar_iteration* iterations,
                              int32_t max_iterations, povar_solve_summary* summary, int32_t* status, void* stream);

/* ba_log.json with the reference's complete key set (bal/ba_log.hpp:85-245, bal/ba_log_utils.cpp:100-175), so that
 * the reference's python/rootba tooling loads it unchanged; what `bal --log-log-path` writes.  lm_ptr may be NULL
 * (then per_lm_obs is zero).  Host only. */
typedef struct povar_ba_log_info {
  const char* input_path;
  int32_t num_cams;
  int32_t num_lms;
  int64_t num_obs;
  const int64_t* lm_ptr;     /* [num_lms+1] of the whole problem, or NULL */
  double load_time;          /* seconds, timing.load */
  int32_t num_gpus;
} povar_ba_log_info;
int povar_write_ba_log(const char* path, const povar_ba_log_info* info, const povar_options* opt,
                       const povar_iteration* iterations, int32_t num_iterations, const povar_solve_summary* summary);

/* ---------- instrumentation ------------------------------------------------------------ */

/* Phase times of the Linearizor methods, seconds, from CUDA events on the handle's stream, accumulated since the
 * last povar_reset_timings: what the reference's linearizors write into IterationSummary through IF_SET(it_summary_)
 * (solver/linearizor_power_varproj.cpp:16-17; fields of solver/solver_summary.hpp:172-212). */
typedef struct povar_phase_times {
  double residual_evaluation_time;     /* compute_error_* */
  double jacobian_evaluation_time;     /* linearize_*: Jacobians, Jp^T Jp, Jacobi scalings */
  double prepare_time;                 /* solve: Hll^-1, B^-1, b (the reference's stage2 / prepare columns) */
  double solve_reduced_system_time;    /* power series / PCG / Cholesky */
  double back_substitution_time;       /* apply_* */
} povar_phase_times;
int povar_get_timings(const povar_handle* h, povar_phase_times* out);
int povar_reset_timings(povar_handle* h);

/* copy an internal device array to the host for parity tests.  Names: "pose_scale" [C*12],
 * "lm_scale" [L*4], "hll_inv" [L*6], "b_inv" [C*D*D], "b" [C*D], "inc" [C*D], "lm_ptr", ...
 * returns the element count, or < 0. */
int64_t povar_debug_read(povar_handle* h, const char* name, double* out, int64_t capacity);

/* E0 * x for a caller-supplied camera-space vector (C*12 for POSE, C*11 for JOINT) with the
 * current linearisation: right_mul_e0_pOSE / right_mul_e0_joint
 * (sc/linearization_power_varproj.hpp:364-453).  Used by tests and by the SpMV benchmark. */
int povar_right_mul_e0(povar_handle* h, int32_t which, const double* x, double* out);

/* run `terms` power-series terms back to back on the current linearisation (no early exit) and
 * return the device time per term in seconds: the SpMV roofline measurement of bench.py. */
int povar_bench_power_terms(povar_handle* h, int32_t which, int32_t terms, double* seconds_per_term);

/* average device time (seconds) of each kernel of one power-series term, each launched `reps`
 * times back to back between two CUDA events on the handle's stream:
 * seconds[0] landmark half of E0, [1] camera half of E0, [2] per-camera item reduction,
 * [3] B^-1 apply + accumulate + norms + convergence test. */
int povar_bench_power_kernels(povar_handle* h, int32_t which, int32_t reps, double seconds[4]);

/* kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t povar_launch_count(const povar_handle* h);

/* host-side sliced-ELL order of the landmark half of the E0 product (DESIGN.md 2), exposed for the CPU tests:
 * call with NULL outputs to get sizes = {len(slice_ptr), len(sell_lm), len(long_lms)}, then again with buffers.
 * `threads` > 0 fixes the number of host threads (the result must not depend on it), 0 = automatic. */
int povar_debug_sell_layout(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                            int32_t threads, int32_t max_deg, int32_t* slice_ptr, int32_t* sell_lm,
                            int32_t* long_lms, int64_t sizes[3]);
/* largest number of observations of a landmark of that order (`max_deg` above; 0 = 32) that povar_create uses for a
 * shard of num_obs observations on a device with `sms` multiprocessors: 32, less on small shards */
int povar_debug_sell_max_degree(int64_t num_obs, int32_t sms);

/* host-side plan of the landmark half for that order (DESIGN.md 4): which slices every warp walks and which
 * cameras every block stages in shared memory.  model: 0 step 1, 1 step 2, 2 step 1 with HUBER weights;
 * sms: streaming multiprocessors to plan for.  info = {warps per block, ring stages, blocks per SM, blocks,
 * ranges, cameras per window, 1 if every block's window holds every camera its slices meet, bytes of shared
 * memory per block}.  range_slice [ranges + 1] and blk_lo [blocks] may be NULL (sizes come back in info). */
int povar_debug_landmark_plan(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                              int32_t model, int32_t sms, int32_t max_deg, int64_t info[8], int32_t* range_slice,
                              int32_t* blk_lo);

/* Tuning builds only (-DPOVAR_WALK_TRACE; POVAR_ERR_UNSUPPORTED otherwise): per block of the last landmark-half
 * launches, four globaltimer stamps (entry, window staged, slices walked, done); reset on read. */
int povar_debug_walk_trace(uint64_t* out, int32_t n);

/* The direct solver of CHOLESKY (blocked LL^T on FP64 tensor-core tiles + substitution, kernels_chol.cu) on a
 * caller-supplied symmetric matrix: x = A^-1 b for a row-major n x n matrix of which the lower triangle is read.
 * *info = 0, or 1 + the index of the first 64-row tile with a non-positive pivot (x is then undefined).  What the
 * reference does with Eigen::SimplicialLLT (sc/linearization_sc.hpp:236-245); exposed for the tests. */
int povar_debug_cholesky(int32_t n, const double* A, const double* b, double* x, int32_t* info);

/* CHOLESKY keeps the reduced camera system dense while that takes at most 96 GB and switches to tile-sparse storage
 * beyond: only the 64x64 tiles of the factor that can be non-zero, cameras in reverse Cuthill-McKee order of their
 * co-visibility graph (DESIGN.md 4).  If the tile-sparse factor does not fit the device's free memory either, the
 * solve fails with POVAR_ERR_UNSUPPORTED.  mode 0: that automatic choice, 1: tile-sparse always (tests).
 * povar_debug_read names "chol_perm" [C] (position of every camera in the factor order) and "chol_tiles" [1]
 * (stored tiles) have 0 elements unless the handle's last CHOLESKY solve ran on tile-sparse storage. */
int povar_debug_set_cholesky_storage(povar_handle* h, int32_t mode);

/* povar_debug_cholesky on tile-sparse storage: the pattern is that of the non-zero block x block blocks of A's lower
 * triangle, ordered and factorised symbolically as a handle's S is (one block per camera), and the same kernels run.
 * *stored_tiles: 64x64 tiles of the factor kept. */
int povar_debug_sparse_cholesky(int32_t n, int32_t block, const double* A, const double* b, double* x,
                                int32_t* info, int64_t* stored_tiles);

/* the host ordering and symbolic factorisation of the tile-sparse CHOLESKY for a landmark-major index (the
 * co-visibility bitmap built on the host): perm [num_cams] = position of every camera, *stored_tiles.  `threads` > 0
 * fixes the number of host threads (the result does not depend on it), 0 = automatic. */
int povar_debug_cholesky_symbolic(int32_t num_cams, int32_t num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                                  int32_t threads, int32_t* perm, int64_t* stored_tiles);

/* Caps the number of camera records the landmark half of a power-series term stages in shared memory (0 = as many
 * as fit).  The result must not depend on it: cameras outside the staged window are read from global memory.  Tests
 * use it to exercise that path on problems whose whole camera table would fit. */
int povar_debug_set_window(povar_handle* h, int32_t cams);

/* 1 if this handle exchanges the per-term camera sums over peer memory (CUDA IPC + NVLink stores fused
 * into the term kernel), 0 if it uses ncclAllReduce per term (single GPU: 0).  POVAR_PEER_EXCHANGE=0 in
 * the environment forces NCCL, =1 makes povar_create fail instead of falling back. */
int povar_peer_exchange_active(const povar_handle* h);

/* the cudaStream_t every kernel of this handle is launched on, so that a caller can bracket calls
 * with its own CUDA events (the reference's counterpart is the wall-clock Timer around
 * optimize_lm_ours_pOSE, solver/bal_bundle_adjustment.cpp:256, 868-871) */
void* povar_cuda_stream(const povar_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* POVAR_B200_H_ */
