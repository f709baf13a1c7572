// Internal declarations shared by the CUDA translation units and the host driver.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/povar_b200.h"
#include "lm_step.h"

namespace povar {

// per-observation arrays, landmark-major (canonical order) and camera-major (CSC)
struct DeviceIndex {
  int C = 0;          // cameras (global)
  int L = 0;          // landmarks in this shard
  int nnz = 0;        // observations in this shard
  // landmark-major
  int* lm_ptr = nullptr;      // [L+1]
  int* obs_cam = nullptr;     // [nnz]
  int* obs_lm = nullptr;      // [nnz]
  double2* obs_uv = nullptr;  // [nnz]
  // landmark-major, sliced ELL for the landmark half of E0 (kernels_series.cu): landmarks with 1..32
  // observations, ordered by the centre of their cameras, sorted by degree inside windows of kSellWindow
  // landmarks of that order, kSellWidth (32) per slice; slot
  // 32 * row + g holds the row-th observation of the g-th landmark of the slice (camera -1 = padding)
  int num_slices = 0;
  int sell_max_deg = 32;      // landmarks with more observations than this are `long` (sell_max_degree, engine.cu)
  int* slice_ptr = nullptr;   // [num_slices+1] first row of the slice
  int* sell_lm = nullptr;     // [32*num_slices] landmark of lane g, -1 = none
  int* sell_cam = nullptr;    // [32*rows] k-th observation of a landmark in row k of its slice
  double2* sell_uv = nullptr; // [32*rows]
  // the copy the power-series term kernel streams: inside a landmark the observations sit in the rows
  // k_sell_rows chose (fewer shared-memory bank conflicts between the lanes of a quarter warp)
  int* sell_cam_e0 = nullptr;           // [32*rows]
  double2* sell_uv_e0 = nullptr;        // [32*rows]
  unsigned char* sell_row_e0 = nullptr; // [32*rows] by slot of the first copy: row inside the slice in the second
  int* obs_slot = nullptr;    // [nnz] slot of the observation, -1 for landmarks outside the SELL set
  long long sell_slots = 0;   // 32 * rows
  int num_long = 0;           // landmarks with more than 32 observations: one warp each, CSR arrays
  int* long_lm = nullptr;     // [num_long]
  // camera-major
  int* cam_ptr = nullptr;     // [C+1]
  int* csc_lm = nullptr;      // [nnz] landmark of the entry (ascending inside a camera)
  double2* csc_uv = nullptr;  // [nnz]
  int* item_cam = nullptr;    // [num_items] camera of the work item
  int* item_ptr = nullptr;    // [num_items+1] entry ranges, never crossing a camera boundary
  int* cam_item_ptr = nullptr;  // [C+1] items of a camera
  int num_items = 0;
};

constexpr double kEpsSqrtHost = 1e-5;  // Sophus::Constants<double>::epsilonSqrt()
constexpr int kKron = 60;     // unique entries of sum_i E_i (x) (X X^T): 6 x 10
constexpr int kSellWidth = 32;      // landmarks per slice of the sliced-ELL order: one per lane of a warp
constexpr int kSellWindow = 4096;   // sorting window of the sliced-ELL landmark order
constexpr int kSliceCost = 2;        // rows a slice costs on top of its own when the walks are balanced
constexpr int kSellKeySpan = 896;   // cameras the key of a landmark (build_sell) tries to centre
constexpr int kCamRecStride = 26;   // doubles per camera record, the larger of the two models (CamRec::stride)
constexpr int kCamRecPose = 22, kCamRecJoint = 26;   // CamRec::stride(false / true)
// per-camera tables of the once-per-trial landmark walks (kernels_landmark.cu): [P | pad], [A | B | pad]
constexpr int kCamTab1 = 14, kCamTab2 = 26;
// bytes of one row of the observation stream of the landmark half: 32 camera indices + 32 x (u, v) in step 1
// (+ 32 robust weights with HUBER), 32 camera indices + 3 x 32 coefficients in step 2
constexpr int kStagePose = 128 + 512, kStageWide = 128 + 768;
// the linearisation walk also streams the 32 row numbers of sell_row_e0
constexpr int kStageLin = kStagePose + 32;
// shared memory of a block of the landmark half ahead of the rings: one mbarrier for the window and one per
// ring stage, rounded up to 128 bytes
__host__ __device__ constexpr int lm_bar_bytes(int warps, int stages) { return ((1 + warps * stages) * 8 + 127) / 128 * 128; }
// per-landmark record read by the camera-major passes: [X0 X1 H0 H1 | X2 X3 H2 H3].  The two 32-byte halves are what
// the two lanes of an entry of the camera half need, so each takes its half with ONE 256-bit load (lm_rec_half,
// device_math.cuh): the gather costs one L1 wavefront per entry instead of two
constexpr int kLmRec = 8;
constexpr int kLmRecX0 = 0, kLmRecH0 = 2, kLmRecX2 = 4, kLmRecH2 = 6;

// series control block, lives in device memory
struct SeriesCtl {
  int done;            // early exit taken: later kernels of the series return at once
  int iterations;      // summary.num_iterations
  int nonfinite;       // increment has NaN/Inf
  int peer_timeout;    // a peer's camera sums never arrived (PeerExchange): the solve fails loudly
  double norm0;        // |accum_0| when r_tolerance > 0
  double last_tmp_norm;
  double last_acc_norm;
  unsigned int ticket; // last-block election
  unsigned int next_block;  // peer mode: logical block numbers in dispatch order
  int term;            // terms of the running series that are complete (the loop of the series graph counts here)
  // landmark half: the landmarks with many observations are handed out to the warps as they finish their slices
  unsigned int long_next;   // next one to take
  unsigned int long_left;   // blocks of the launch that have left the queue (the last one resets both)
};

// The series as a loop of a CUDA graph (Engine::capture_series: the series graph of enqueue_series, or a node of the
// solve graph): `handle` is the conditional handle of the WHILE node whose body is one term; k_series_start and the
// last block of k_term16 set it (cudaGraphSetConditional), so a series runs exactly the terms the reference's stopping
// rule asks for and nothing is enqueued to be skipped.
struct SeriesLoop {
  unsigned long long handle = 0;   // cudaGraphConditionalHandle
  int active = 0;                  // 0: terms are enqueued one by one with their number (eager launches, benchmarks)
  int max_terms = 0;
};

// scalars of the preconditioned conjugate gradients (PCG / RIPCG), kept on the device: the iteration decides there
struct CgState {
  double rho, last_rho, alpha, beta, q0, norm_b;
};

// Peer-memory exchange of the per-term camera sums when landmarks are sharded over several GPUs
// (engine.cu Engine::setup_peer_exchange, kernels_camera.cu k_term16<.., kTermPeer>).  Every rank owns
// a receive buffer [2 parities][world][stride] of 16-byte slots {lo, epoch, hi, epoch}; recv[r] is rank r's
// buffer as mapped into this process (CUDA IPC over NVLink; recv[rank] is the local one).  stride = 60*C
// slots: the largest camera-sized vector that is reduced (the Kronecker sums); the per-term exchange uses the
// first 12*C of them, scalar reductions the first few.
constexpr int kMaxPeers = 8;
struct PeerExchange {
  double* recv[kMaxPeers];
  int rank, world;
  // count[0]: exchanges performed so far on this buffer (device memory, local); the next exchange has number
  // count[0] + 1 (its tag; parity = number & 1) and the kernel that performs it stores the new count.
  // count[1]: block ticket of k_peer_allreduce.
  unsigned int* count;
  unsigned long long stride;
};
// where k_term16 takes the reduced camera sums from
enum TermMode { kTermRaw = 0, kTermFused = 1, kTermPeer = 2 };

struct CostAccum {
  double err_all, rsum_all, err_valid, rsum_valid;
  long long n_all, n_valid;
  int nonfinite;
  int pad;
};

// How the landmark half of a power-series term (kernels_series.cu) walks the sliced-ELL order: `ranges`
// contiguous slice ranges with (nearly) equal numbers of rows, one per warp; a block of `warps` warps takes
// consecutive ranges and stages the camera records [blk_lo[b], blk_lo[b] + win_cams) in shared memory.  Made
// once per handle and model by plan_landmark_half (engine.cu) from what fits in shared memory.
struct LmPlan {
  int warps = 0;          // warps per block: 8, 16, 24 or 32
  int stages = 0;         // depth of every warp's stream ring: 2 or 3 rows
  int blocks_per_sm = 1;
  int blocks = 0;
  int ranges = 0;
  int win_cams = 0;       // cameras staged per block (C if the whole table fits)
  int covered = 0;        // 1: every block's window holds every camera its slices meet
  int* range_slice = nullptr;   // [ranges + 1] first slice of every range
  int* blk_lo = nullptr;        // [blocks] first camera of the block's window
};

// everything a kernel launcher needs
struct DeviceState {
  DeviceIndex ix;
  // state (current and backup)
  double* P = nullptr;        // [C*12]
  double* P_bak = nullptr;
  double* X = nullptr;        // [L*4]  step 1: [x y z 1]; step 2: homogeneous
  double* X_bak = nullptr;
  // linearisation
  double* pose_scale = nullptr;  // [C*12]
  double* lm_scale = nullptr;    // [L*4]
  double* lm_hraw = nullptr;     // [L*10] sum_i w Jl_raw^T Jl_raw (packed symmetric; 6 used in step 1)
  double* lm_graw = nullptr;     // [L*4]  sum_i w Jl_raw^T r
  double* hll_inv = nullptr;     // [L*6]
  double* lm_rec = nullptr;      // [L*8]  X and H for the camera-major passes (kLmRec)
  double* lm_fold = nullptr;     // [L*10] S (Pi) Hll^-1 (Pi^T) S, packed symmetric: H_l = fold_l G_l
  double* cam_rec = nullptr;     // [C*32] per-camera record of the landmark-major E0 pass (CamRec<>)
  double* obs_d = nullptr;       // [nnz*3] step 2: sqrt(w) (1/z, -x/z^2, -y/z^2) at the linearisation point
  double* csc_d = nullptr;       // [nnz*3] the same, camera-major
  double* obs_w = nullptr;       // [nnz]   step 1, HUBER only: robust weight at the linearisation point
  double* sell_d = nullptr;      // [rows][3][32] obs_d in SELL order, one plane per coefficient and row
  // per-landmark data of the sliced-ELL set as lane-major planes [slice][component][32]: what the walks read
  // and write with one coalesced line per component (the landmarks with more than 32 observations use the
  // by-landmark arrays above)
  double* sell_x = nullptr;      // [slices][4][32]  X at the linearisation point
  double* sell_hraw = nullptr;   // [slices][10][32]
  double* sell_graw = nullptr;   // [slices][4][32]
  double* sell_scale = nullptr;  // [slices][4][32]
  double* sell_hinv = nullptr;   // [slices][6][32]  Hll^-1 of the last solve
  double* sell_fold = nullptr;   // [slices][10][32]
  double* sell_step = nullptr;   // [slices][4][32]  VarPro back-substitution: the landmark step between its walks
  double* sell_w = nullptr;      // [slots]   obs_w in SELL order
  double* csc_w = nullptr;       // [nnz]   the same, camera-major
  double* kron = nullptr;        // [C*60]
  double* kron2 = nullptr;       // [C*60] diagonal blocks of sum_l Hpl Hll^-1 Hlp (PCG preconditioner)
  double* item_kron = nullptr;   // [num_items*60]
  double* item_part = nullptr;   // [num_items*12]
  double* cam_raw = nullptr;     // [C*12] per-camera sums of the camera-major pass (allreduced)
  double* Bmat = nullptr;        // [C*144]
  double* Binv = nullptr;        // [C*144]
  double* b = nullptr;           // [C*12]
  double* vec_tmp = nullptr;     // [C*12]
  double* vec_acc = nullptr;     // [C*12]  the increment
  double* vec_y = nullptr;       // [C*12]  s o x (step 1) / s o (Pi x) (step 2): what the passes gather
  double* vec_x = nullptr;       // [C*12]  scratch (right_mul_e0 input, PCG vectors)
  double* cg_r = nullptr;        // PCG work vectors [C*12] each
  double* cg_p = nullptr;
  double* cg_z = nullptr;
  double* cg_q = nullptr;
  double* cg_x = nullptr;
  double* Mprec = nullptr;       // [C*144] block-Jacobi preconditioner (inverse blocks)
  double* norm_part = nullptr;   // [C*4]   per-camera partial norms / dots
  double* cost_part = nullptr;   // [blocks * 8]
  CostAccum* cost_out = nullptr;
  double* scalar_part = nullptr; // [blocks] l_diff partials
  // what one LM trial reports, as doubles so that shards can be summed in place (Engine::allreduce):
  // [0..7] cost {err_all, rsum_all, err_valid, rsum_valid, n_all, n_valid, nonfinite, -}, [8] l_diff,
  // [9] numerical-failure flag of the linearisation
  double* trial_out = nullptr;   // [16]
  int* flags = nullptr;          // [4] numerical-failure flags
  SeriesCtl* ctl = nullptr;
  CgState* cg = nullptr;
  // plans of the sliced-ELL walks: [0] landmark half of a term, step 1; [1] step 2; [2] step 1 with HUBER
  // weights; [3] once-per-trial walks over [P]; [4] over [A | B]
  LmPlan plan[5];
  double* cam_tab = nullptr;     // [C*26] the table of the walks of plan 3 / 4, packed right before each
  int debug_window_cams = 0;     // > 0: cap on the cameras the landmark half stages (povar_debug_set_window)
  double* dense_S = nullptr;     // CHOLESKY: [n_pad x n_pad], n_pad = 12 C rounded up to 64
};

// streaming multiprocessors of the current device (grids are sized in multiples of it)
inline int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
      cached = n;
    } else {
      cached = 148;   // B200
    }
  }
  return cached;
}

struct LaunchCfg {
  cudaStream_t stream = nullptr;
  long long* launch_counter = nullptr;
};

// Largest degree of a landmark of the sliced-ELL set.  A slice is walked row by row by ONE warp, so a slice of 32
// rows is a chain of 32 dependent steps (0.76 us each when the SM is not full); on a large shard every warp has
// dozens of rows anyway, on a small one (a venice-1778 shard on 8 GPUs: one slice of ~5 rows per warp) the few
// slices of 30 rows set the time of the whole launch (27 us where the median block needs 19).  There the
// landmarks with more than about twice the rows a warp has anyway go to the warp-per-landmark kernels instead
// (32 observations per step): 31 -> 22 us per launch with 12, measured on that shard.  (Host and device: the
// device canonical order makes the landmark table with it, kernels_index.cu.)
__host__ __device__ inline int sell_max_degree(long long nnz, int sms) {
  const long long rows_per_warp = nnz / (32LL * 32 * sms);   // rows of one resident wave of warps
  if (rows_per_warp >= 16) return 32;
  long long t = (2 * rows_per_warp + 3) / 4 * 4;
  if (t < 8) t = 8;
  if (t > 32) t = 32;
  return static_cast<int>(t);
}

struct ModelParams {
  double c1, c2;        // sqrt(1-alpha), sqrt(alpha)
  int robust_norm;
  double huber;
  double jacobi_eps;
};

// ---- device-side index construction (kernels_index.cu) ----
size_t sell_sort_temp_bytes(int L, int num_cams, int n, int window);
cudaError_t build_device_sell(int L, int num_cams, int n, int window, int max_deg, const int* lm_ptr, const int* obs_cam,
                              int* keys_a, int* keys_b, int* ids_a, int* ids_b, void* sort_temp,
                              size_t sort_temp_bytes, int* sell_lm, int* slice_len, int* slice_lo, int* slice_hi,
                              const LaunchCfg& lc);
// range / order check of the camera indices and the per-camera counts on the device: out[0..C) counts, out[C] flags
cudaError_t validate_obs(int L, int C, int sms, const int* lm_ptr, const int* obs_cam, int* out, const LaunchCfg& lc);
size_t index_sort_temp_bytes(int nnz, int num_cams);
cudaError_t build_device_index(const DeviceIndex& ix, int* iota, int* keys_out, int* perm, int* lm_slot,
                               void* sort_temp, size_t sort_temp_bytes, const LaunchCfg& lc);
// canonical order of an unordered device list (povar_create_device): keys + counts, radix sort, then the shard's
// entries gathered into ix.lm_ptr / obs_cam / obs_lm / obs_uv and the landmark table.  info: kOrderInfo zeroed ints.
enum { kOrderBefore = 0, kOrderCount = 1, kOrderFlags = 2, kOrderSell = 3, kOrderLong = 4, kOrderInfo = 5 };
int order_cam_bits(int num_cams);
int order_end_bit(int num_cams, int num_lms);
size_t device_order_temp_bytes(int n, int L, int end_bit);
cudaError_t device_order_keys(int n, int C, int num_lms, int lm_begin, int lm_end, const int* obs_cam, const int* obs_lm,
                              unsigned long long* keys, int* pos, int* info, const LaunchCfg& lc);
cudaError_t device_order_sort(int n, int end_bit, const unsigned long long* keys_in, unsigned long long* keys_out,
                              const int* pos_in, int* pos_out, void* temp, size_t temp_bytes, const LaunchCfg& lc);
// is_long [ix.L], long_lms [ix.L] scratch: the first info[kOrderLong] of long_lms are the long landmarks, ascending
cudaError_t device_order_place(int n, int C, int lm_begin, int sms, const unsigned long long* keys, const int* pos,
                               const double* obs_uv_in, int* info, const DeviceIndex& ix, unsigned char* is_long,
                               int* long_lms, void* temp, size_t temp_bytes, const LaunchCfg& lc);

// ---- landmark-major kernels (kernels_landmark.cu) ----
void launch_init_varproj(const DeviceState& d, const ModelParams& mp, const LaunchCfg& lc);
void launch_cost(const DeviceState& d, const ModelParams& mp, bool joint, const LaunchCfg& lc);
// trial_out[9] = flags[0] as a double
void launch_flag_to_double(const DeviceState& d, const LaunchCfg& lc);
void launch_lin_landmark(const DeviceState& d, const ModelParams& mp, bool joint, bool scale_jl,
                         const LaunchCfg& lc);
// hinv_by_landmark: also store Hll^-1 of the sliced-ELL landmarks by landmark (PCG / CHOLESKY read it camera-major)
// lambda_dev (not null): the damping is read from device memory instead (the device-side solve)
void launch_prep_landmark(const DeviceState& d, bool joint, double lambda_lm, bool hinv_by_landmark,
                          const LaunchCfg& lc, const double* lambda_dev = nullptr);
void launch_backsub_varpro(const DeviceState& d, const ModelParams& mp, const double* inc,
                           const LaunchCfg& lc);
void launch_backsub_poba(const DeviceState& d, const ModelParams& mp, const double* y,
                         const LaunchCfg& lc);
void launch_backsub_joint(const DeviceState& d, const ModelParams& mp, const double* y,
                          const LaunchCfg& lc);
void launch_to_homogeneous(const DeviceState& d, const LaunchCfg& lc);
void launch_normalize_joint(const DeviceState& d, const LaunchCfg& lc);
int cost_blocks(const DeviceState& d);
int scalar_blocks(const DeviceState& d);

// ---- camera-major kernels (kernels_camera.cu) ----
enum KronKind { KRON_HPP = 0, KRON_SDIAG = 1 };
void launch_kron(const DeviceState& d, const ModelParams& mp, bool joint, KronKind kind,
                 const LaunchCfg& lc);
void launch_reduce_items(const DeviceState& d, const double* item_vals, int width, double* out,
                         bool in_series, const LaunchCfg& lc);
void launch_cam_scale(const DeviceState& d, const ModelParams& mp, const LaunchCfg& lc);
void launch_cam_binv(const DeviceState& d, bool joint, double lambda, const LaunchCfg& lc,
                     const double* lambda_dev = nullptr);
void launch_cam_precond(const DeviceState& d, bool joint, const double* kron_sdiag, const LaunchCfg& lc);
void launch_passB(const DeviceState& d, const ModelParams& mp, bool joint, const LaunchCfg& lc);
// series bookkeeping
void launch_series_start(const DeviceState& d, double r_tolerance, int max_terms, const LaunchCfg& lc,
                         const SeriesLoop& loop = SeriesLoop());
// mode kTermFused: the term kernel adds the item partials of the camera half itself (single GPU);
// kTermPeer: it also pushes them to every rank's receive buffer and adds the ranks' sums in rank order
// (px, with px->epoch set for this exchange); kTermRaw: it reads cam_raw (after launch_reduce_items and
// the NCCL all-reduce)
// term > 0: the number of the term; 0 (inside the loop of the series graph): one more than ctl->term
void launch_series_term(const DeviceState& d, bool joint, int term, double eta, double r_tolerance,
                        TermMode mode, const PeerExchange* px, const LaunchCfg& lc,
                        const SeriesLoop& loop = SeriesLoop());

// buf[0..n) += the other ranks' buf, over the peer buffers (n <= px.stride): what ncclAllReduce(sum) would do,
// every rank adding in rank order
void launch_peer_allreduce(const DeviceState& d, double* buf, size_t n, const PeerExchange& px, const LaunchCfg& lc,
                           bool skip_when_done = false);
void launch_finish_b(const DeviceState& d, bool joint, const LaunchCfg& lc);
void launch_e0_finish(const DeviceState& d, bool joint, double* out, const LaunchCfg& lc);
void launch_make_y(const DeviceState& d, bool joint, const double* x, double* y, const LaunchCfg& lc);
// cam_rec: matrix part (after a linearisation) -- the y part is written by whoever makes y
void launch_cam_rec_static(const DeviceState& d, bool joint, const LaunchCfg& lc);
int debug_walk_trace(unsigned long long* out, int n);   // tuning builds only, POVAR_ERR_UNSUPPORTED otherwise
// ---- power-series term kernels, lane-group layout (kernels_series.cu) ----
void launch_e0_landmark_v2(const DeviceState& d, const ModelParams& mp, bool joint, bool in_series,
                           const LaunchCfg& lc);
void launch_passB_e0_v2(const DeviceState& d, const ModelParams& mp, bool joint, bool in_series,
                        const LaunchCfg& lc);
void launch_cam_update_pose(const DeviceState& d, const double* inc, const LaunchCfg& lc);
void launch_cam_update_joint(const DeviceState& d, const double* y, const LaunchCfg& lc);
void launch_normalize_cams(const DeviceState& d, const LaunchCfg& lc);
// PCG / Cholesky helpers (kernels_schur.cu)
void launch_block_matvec(const DeviceState& d, int dim, const double* blocks, const double* x,
                         double* out, const LaunchCfg& lc);
// out = a * x + b * y (y may be nullptr)
void launch_axpby(const DeviceState& d, int n, double a, const double* x, double b, const double* y,
                  double* out, const LaunchCfg& lc);
// CHOLESKY (kernels_chol.cu): dense reduced camera system of step 1, S = blockdiag(Bmat) - sum_l Hpl Hll^-1 Hlp,
// lower block triangle, fixed summation order; blocked LL^T on 64x64 tiles; substitution
int chol_padded(int n);
void launch_schur_lower(const DeviceState& d, const ModelParams& mp, double* S, int n_pad, const LaunchCfg& lc);
void launch_cholesky_factor(double* S, int n_pad, double* linv, int* info, const LaunchCfg& lc);
void launch_cholesky_solve(const double* S, int n_pad, const double* linv, double* r, const int* info,
                           const LaunchCfg& lc);
void launch_finite_check(const DeviceState& d, int n, const double* x, const LaunchCfg& lc);

// CHOLESKY on tile-sparse storage: only the 64x64 tiles of the factor that can be non-zero, in a fill-reducing block
// order.  Made once per handle on the host (host/chol_symbolic.cpp).
struct CholPattern {
  int nb = 0, block = 0, n_pad = 0, T = 0;   // nb blocks (cameras) of `block` rows; T = n_pad / 64 tile rows
  std::vector<int> perm;               // [nb] position of block c in the factor order (reverse Cuthill-McKee)
  std::vector<int> col_ptr, col_row;   // [T + 1], [tiles]: tile rows of column J, ascending, the diagonal first;
                                       // the index into col_row is the tile's slot in storage
  std::vector<int> row_ptr, row_col;   // [T + 1], [tiles]: tile columns of row I, ascending, the diagonal last
  std::vector<int> slot;               // [T * T] slot of tile (I, J), I >= J, or -1
  long long tiles() const { return static_cast<long long>(col_row.size()); }
};
// bits: nb rows of (nb + 31) / 32 words, bit (a, b) set when blocks a and b are coupled (symmetric); threads = 0:
// automatic.  The result does not depend on `threads`.
void chol_symbolic(int nb, int block, const std::vector<unsigned int>& bits, int threads, CholPattern* out);
// the camera co-visibility bitmap of a landmark-major index, [C][(C + 31) / 32] words: on the host (tests) and in
// HBM (kernels_index.cu, one pass over lm_ptr / obs_cam)
void covisibility_host(int num_cams, int num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                       std::vector<unsigned int>* bits);
cudaError_t build_covisibility(int L, int C, const int* lm_ptr, const int* obs_cam, unsigned int* bits,
                               const LaunchCfg& lc);
// the pattern in device memory
struct CholTilesDev {
  int T = 0;
  double* tiles = nullptr;   // [tiles][64][64], row-major tiles in slot order
  const int* slot = nullptr;      // [T * T]
  const int* col_ptr = nullptr;   // [T + 1]
  const int* col_row = nullptr;
  const int* row_ptr = nullptr;   // [T + 1]
  const int* row_col = nullptr;
  const int* perm = nullptr;      // [C] (assembly of a handle's S)
};
// S in the tiled, permuted layout (lower tile triangle of the factor order; tiles must be zero on entry)
void launch_schur_tiles(const DeviceState& d, const ModelParams& mp, const CholTilesDev& s, int n_pad, const LaunchCfg& lc);
void launch_cholesky_factor_tiles(const CholPattern& p, const CholTilesDev& s, double* linv, int* info, const LaunchCfg& lc);
void launch_cholesky_solve_tiles(const CholPattern& p, const CholTilesDev& s, const double* linv, double* r,
                                 const int* info, const LaunchCfg& lc);
// r[12 perm[c] + k] = -b[12 c + k] (r zero elsewhere beforehand) / x[12 c + k] = r[12 perm[c] + k]
void launch_perm_gather_neg(int C, const int* perm, const double* b, double* r, const LaunchCfg& lc);
void launch_perm_scatter(int C, const int* perm, const double* r, double* x, const LaunchCfg& lc);
// PCG / RIPCG with the scalars and the termination tests on the device (kernels_schur.cu); every kernel returns
// at once when ctl->done is set
enum CgStage { CG_BEGIN = 0, CG_RHO = 1, CG_PQ = 2, CG_ZETA = 3 };
// reduces the partials of the preceding launch_dot_partials and applies stage `stage` of iteration `it`
// it_base (not null): the iteration is it + *it_base (the loop of the device-side solve counts on the device)
void launch_cg_scalar(const DeviceState& d, CgStage stage, int it, double eta, int min_it, int max_it, const LaunchCfg& lc,
                      const int* it_base = nullptr);
void launch_dot_partials(const DeviceState& d, int n, const double* x, const double* y, const LaunchCfg& lc);
enum CgUpdate { CG_UPDATE_P = 0, CG_UPDATE_X = 1, CG_UPDATE_R = 2 };
void launch_cg_update(const DeviceState& d, CgUpdate what, int n, int it, const double* src, double* dst, const LaunchCfg& lc,
                      const int* it_base = nullptr);

// ---- the LM loops on the device (kernels_lm.cu, Engine::bundle_adjust_async) ----
// control block of the device-side solve: the state run_step / povar_bundle_adjust keep on the host
enum LmMessage { LM_MSG_NONE = 0, LM_MSG_LINEARIZATION, LM_MSG_PEER_TIMEOUT, LM_MSG_FUNCTION_TOLERANCE,
                 LM_MSG_MAX_DAMPING, LM_MSG_MAX_ITERATIONS };
struct LmCtl {
  LmLoop loop;
  LmLog log;
  povar_residual_info ri;           // cost of the current state
  int32_t status;                   // what povar_bundle_adjust returns
  int32_t termination[2];
  int32_t message, message_iterations;
  int32_t lin_next;                 // the next trial starts with a linearisation (its failure flag is read with the trial)
  int32_t cg_base;                  // PCG / RIPCG: iterations of the running solve before the current loop body
  long long power_terms;
  double power_time;
  double times[5];                  // residual, linearize, prepare, reduced solve, back-substitution (s, since the last entry)
  unsigned long long t_start, t_it, t_step1;
  unsigned long long stamp[8];      // %globaltimer where the host route records its events ev_[0..7]
};
// condition handles of the graph (cudaGraphConditionalHandle values; kNoCond: none)
constexpr unsigned long long kNoCond = ~0ULL;
struct LmConds {
  unsigned long long run = kNoCond, lin = kNoCond, restore = kNoCond;
};
void launch_lm_stamp(unsigned long long* at, const LaunchCfg& lc);
// t_it = now; the IF(linearise) node of the trial body runs when ctl->lin_next
void launch_lm_top(LmCtl* ctl, const LmConds& h, const LaunchCfg& lc);
// iteration 0 of step `step` from the cost in trial_out[0..8) (stamps 0 / 1 around it); step 1 also resets ctl
void launch_lm_begin(LmCtl* ctl, const double* trial_out, const povar_options& opt, int step, povar_iteration* log,
                     int capacity, const LmConds& h, const LaunchCfg& lc);
// the decision of one trial (lm_trial_step) and its log entry
void launch_lm_decide(LmCtl* ctl, const double* trial_out, const SeriesCtl* sctl, const povar_options& opt, int step,
                      bool power, povar_iteration* log, int capacity, const LmConds& h, const LaunchCfg& lc);
// termination type and message of a step; step 1: `ok` (IF node of step 2) = no failure
void launch_lm_end_step(LmCtl* ctl, int step, int max_iter, unsigned long long ok, const LaunchCfg& lc);
void launch_lm_finish(LmCtl* ctl, int capacity, povar_solve_summary* summary, int* status, const LaunchCfg& lc);
// summary->num_iterations = min(it, max_iterations): the caller's capacity, applied after the graph
void launch_lm_clip(povar_solve_summary* summary, int max_iterations, const LaunchCfg& lc);
// CHOLESKY inside a graph: info != 0 -> an invalid step (what solve_cholesky's host read-back does)
void launch_chol_status(const int* info, SeriesCtl* ctl, const LaunchCfg& lc);
// PCG / RIPCG inside a graph: the WHILE node around 10 iterations; advance = 0 before the node (base = 0)
void launch_cg_loop(SeriesCtl* ctl, int* base, int max_it, bool advance, unsigned long long handle, const LaunchCfg& lc);

}  // namespace povar
