// Landmark-major kernels: everything that reduces over the observations of one landmark.
//
// Work decomposition of the passes over the observations (linearisation, back-substitution): landmarks with
// 1..32 observations go through the sliced-ELL walk of sell_walk.cuh -- one lane per landmark, sums in
// registers in camera order, the camera matrices staged in shared memory by the TMA unit; a landmark with more
// than 32 observations gets a warp of the k_*_long kernels (lanes stride over it, fixed-tree warp sum).  All
// reductions have a fixed order => results are bit-reproducible.
//
// Reference loops replaced (paths relative to /root/reference/src/rootba_povar/):
//   k_init_varproj      bal/bal_bundle_adjustment_helper.cpp:75-99, 220-241
//   k_cost              helper.cpp:116-196, bal/residual_info.cpp:97-117
//   k_lin_landmark      sc/landmark_block.hpp:135-225 (Jl part), 284-309 (scale_Jl_cols_*)
//   k_prep_landmark     sc/landmark_block.hpp:474-572 (Hll^-1, Hll^-1 Jl^T r)
//   k_backsub_*         sc/landmark_block.hpp:574-707
#include <cuda_runtime.h>

#include "device_math.cuh"
#include "povar_internal.h"
#include "sell_walk.cuh"

namespace povar {

namespace {

constexpr int kBlock = 256;
// minimum resident blocks per SM the register allocator has to leave room for (tuning knobs; the
// defaults are the measured optimum on B200, profiles/)
#ifdef POVAR_OCC_LIN
#define POVAR_BOUNDS_LIN __launch_bounds__(kBlock, POVAR_OCC_LIN)
#else
#define POVAR_BOUNDS_LIN __launch_bounds__(kBlock)
#endif
#ifdef POVAR_OCC_BACKSUB
#define POVAR_BOUNDS_BACKSUB __launch_bounds__(kBlock, POVAR_OCC_BACKSUB)
#else
#define POVAR_BOUNDS_BACKSUB __launch_bounds__(kBlock)
#endif

__device__ __forceinline__ void load_lm4(const double* __restrict__ X, int lm, double (&x)[4]) {
  load4_256(X + 4 * static_cast<size_t>(lm), x);
}

// one warp per landmark with more than 32 observations (DeviceIndex::long_lm)
struct TileLane {
  int tb, te;
  int lane;
  __device__ __forceinline__ TileLane(const DeviceIndex& ix, int which) {
    const int lm = __ldg(ix.long_lm + which);
    tb = __ldg(ix.lm_ptr + lm);
    te = __ldg(ix.lm_ptr + lm + 1);
    lane = threadIdx.x & 31;
  }
};

// landmark totals of per-lane accumulators
template <int NV>
__device__ __forceinline__ void tile_allreduce(double (&acc)[NV], const TileLane&, bool, int, const int*) {
  warp_allreduce<NV>(acc);
}

__device__ __forceinline__ bool is_head(const TileLane& t, bool, int, const int*, int) { return t.lane == 0; }

// ------------------------------------------------------------------------------------------
// VarPro initialisation: X_l = argmin | G X - z | by Givens row updates of a 3x3 triangular
// factor (backward stable; the reference uses bdcSvd on the stacked 4n x 3 system).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void givens_row(double (&R)[6], double (&d)[3], double g0, double g1,
                                           double g2, double z) {
  // R packed upper: [00 01 02 11 12 22]
  if (g0 != 0.0) {
    const double rot = hypot(R[0], g0);
    const double c = R[0] / rot, s = g0 / rot;
    R[0] = rot;
    double t;
    t = c * R[1] + s * g1;  g1 = -s * R[1] + c * g1;  R[1] = t;
    t = c * R[2] + s * g2;  g2 = -s * R[2] + c * g2;  R[2] = t;
    t = c * d[0] + s * z;   z = -s * d[0] + c * z;    d[0] = t;
  }
  if (g1 != 0.0) {
    const double rot = hypot(R[3], g1);
    const double c = R[3] / rot, s = g1 / rot;
    R[3] = rot;
    double t;
    t = c * R[4] + s * g2;  g2 = -s * R[4] + c * g2;  R[4] = t;
    t = c * d[1] + s * z;   z = -s * d[1] + c * z;    d[1] = t;
  }
  if (g2 != 0.0) {
    const double rot = hypot(R[5], g2);
    const double c = R[5] / rot, s = g2 / rot;
    R[5] = rot;
    const double t = c * d[2] + s * z;
    d[2] = t;
  }
}

// (one thread per landmark of `list`: the landmarks with more than 32 observations; the others go through the
// walk, InitVarprojOp below)
__global__ void __launch_bounds__(kBlock)
k_init_varproj(int n, const int* __restrict__ list, const int* __restrict__ lm_ptr, const int* __restrict__ obs_cam,
               const double2* __restrict__ obs_uv, const double* __restrict__ P, double c1,
               double c2, double* __restrict__ X) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int l = list[i];
  double R[6] = {0, 0, 0, 0, 0, 0};
  double d[3] = {0, 0, 0};
  const int e = lm_ptr[l + 1];
  for (int o = lm_ptr[l]; o < e; ++o) {
    Cam3x4 cam;
    load_cam(P, obs_cam[o], cam);
    const double2 uv = obs_uv[o];
    // rows of G = T[:, 0:3], z = -(T[:,3]) + [0 0 c2 u c2 v]   (helper.cpp:224-237)
    givens_row(R, d, c1 * (cam.r0[0] - cam.r2[0] * uv.x), c1 * (cam.r0[1] - cam.r2[1] * uv.x),
               c1 * (cam.r0[2] - cam.r2[2] * uv.x), c1 * (cam.r2[3] * uv.x - cam.r0[3]));
    givens_row(R, d, c1 * (cam.r1[0] - cam.r2[0] * uv.y), c1 * (cam.r1[1] - cam.r2[1] * uv.y),
               c1 * (cam.r1[2] - cam.r2[2] * uv.y), c1 * (cam.r2[3] * uv.y - cam.r1[3]));
    givens_row(R, d, c2 * cam.r0[0], c2 * cam.r0[1], c2 * cam.r0[2], c2 * (uv.x - cam.r0[3]));
    givens_row(R, d, c2 * cam.r1[0], c2 * cam.r1[1], c2 * cam.r1[2], c2 * (uv.y - cam.r1[3]));
  }
  // rank-deficient systems (fewer than 3 independent rows): zero the free component.  The
  // reference's SVD solve returns the minimum-norm solution there; BAL landmarks have >= 2 views.
  double x2 = R[5] != 0.0 ? d[2] / R[5] : 0.0;
  double x1 = R[3] != 0.0 ? (d[1] - R[4] * x2) / R[3] : 0.0;
  double x0 = R[0] != 0.0 ? (d[0] - R[1] * x1 - R[2] * x2) / R[0] : 0.0;
  double* out = X + 4 * static_cast<size_t>(l);
  out[0] = x0;
  out[1] = x1;
  out[2] = x2;
  out[3] = 1.0;
}

// ------------------------------------------------------------------------------------------
// cost
// ------------------------------------------------------------------------------------------
template <bool JOINT>
__global__ void __launch_bounds__(kBlock)
k_cost(int nnz, const int* __restrict__ obs_cam, const int* __restrict__ obs_lm,
       const double2* __restrict__ obs_uv, const double* __restrict__ P,
       const double* __restrict__ X, double c1, double c2, Robust rb,
       double* __restrict__ part) {
  __shared__ double smem[6 * (kBlock / 32)];
  double acc[6] = {0, 0, 0, 0, 0, 0};  // err_all rsum_all err_valid rsum_valid n_valid nonfinite
  for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < nnz; o += gridDim.x * blockDim.x) {
    Cam3x4 cam;
    load_cam(P, __ldg(obs_cam + o), cam);
    double x[4];
    load_lm4(X, __ldg(obs_lm + o), x);
    const double2 uv = obs_uv[o];
    double res_sq;
    bool valid = true, finite;
    if (JOINT) {
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, x, rb);
      res_sq = ob.res_sq();
      valid = ob.valid;
      finite = isfinite(ob.r[0]) && isfinite(ob.r[1]);
    } else {
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
      res_sq = ob.res_sq();
      finite = isfinite(ob.r[0]) && isfinite(ob.r[1]) && isfinite(ob.r[2]) && isfinite(ob.r[3]);
    }
    double err, w;
    error_weight(rb, res_sq, err, w);
    const double rn = sqrt(res_sq);
    acc[0] += err;
    acc[1] += rn;
    if (valid) {
      acc[2] += err;
      acc[3] += rn;
      acc[4] += 1.0;
    }
    if (!finite) acc[5] += 1.0;
  }
  block_reduce<6>(acc, smem);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < 6; ++k) part[blockIdx.x * 8 + k] = acc[k];
  }
}

__global__ void __launch_bounds__(kBlock)
k_cost_final(int nblocks, long long nnz, const double* __restrict__ part, CostAccum* out, double* __restrict__ outd) {
  __shared__ double smem[6 * (kBlock / 32)];
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k] += part[b * 8 + k];
  }
  block_reduce<6>(acc, smem);
  if (threadIdx.x == 0) {
    out->err_all = acc[0];
    out->rsum_all = acc[1];
    out->err_valid = acc[2];
    out->rsum_valid = acc[3];
    out->n_all = nnz;
    out->n_valid = static_cast<long long>(acc[4] + 0.5);
    out->nonfinite = acc[5] > 0.0 ? 1 : 0;
    // the same as doubles: what a sharded run sums over the ranks in place
    outd[0] = acc[0];
    outd[1] = acc[1];
    outd[2] = acc[2];
    outd[3] = acc[3];
    outd[4] = static_cast<double>(nnz);
    outd[5] = static_cast<double>(static_cast<long long>(acc[4] + 0.5));
    outd[6] = acc[5] > 0.0 ? 1.0 : 0.0;
    outd[7] = 0.0;
  }
}

__global__ void k_flag_to_double(const int* __restrict__ flags, double* __restrict__ out) {
  out[0] = flags[0] != 0 ? 1.0 : 0.0;
}

__global__ void __launch_bounds__(kBlock)
k_scalar_final(int nblocks, const double* __restrict__ part, double* out) {
  __shared__ double smem[kBlock / 32];
  double acc[1] = {0};
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) acc[0] += part[b];
  block_reduce<1>(acc, smem);
  if (threadIdx.x == 0) out[0] = acc[0];
}

// ------------------------------------------------------------------------------------------
// linearisation, landmark side: sum_i w Jl_raw^T Jl_raw, sum_i w Jl_raw^T r, column scales
// ------------------------------------------------------------------------------------------
template <bool JOINT>
__global__ void POVAR_BOUNDS_LIN
k_lin_long(DeviceIndex ix, const double* __restrict__ P, const double* __restrict__ X,
               double c1, double c2, Robust rb, double eps, int scale_jl,
               double* __restrict__ lm_hraw, double* __restrict__ lm_graw,
               double* __restrict__ lm_scale, int* __restrict__ flags,
               double* __restrict__ obs_d, double* __restrict__ obs_w,
               double* __restrict__ sell_d, double* __restrict__ sell_w) {
  constexpr int NV = JOINT ? 14 : 9;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int tile = warp; tile < ix.num_long; tile += nwarps) {
    const TileLane t(ix, tile);
    double acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.0;
    int lm = __ldg(ix.obs_lm + t.tb), o_first = -1;
    bool has_obs = false, bad = false;
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      has_obs = true;
      if (o_first < 0) o_first = o;
      lm = __ldg(ix.obs_lm + o);
      Cam3x4 cam;
      load_cam(P, __ldg(ix.obs_cam + o), cam);
      double x[4];
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      if (JOINT) {
        JointObs ob;
        ob.eval(cam, uv.x, uv.y, x, rb);
        double j0[4], j1[4];
        ob.jl_rows(cam, j0, j1);
        const double w = ob.sw * ob.sw;
        {
          // what the power-series term kernels stream instead of re-deriving it (kernels_series.cu)
          const double d0 = ob.sw * ob.iz, d1 = ob.sw * ob.d02, d2 = ob.sw * ob.d12;
          double* dp = obs_d + 3 * static_cast<size_t>(o);
          dp[0] = d0;
          dp[1] = d1;
          dp[2] = d2;
          const int slot = __ldg(ix.obs_slot + o);
          if (slot >= 0) {
            // [row][coefficient][lane]: what a warp of the landmark half reads is one line per coefficient
            double* sp = sell_d + 3 * static_cast<size_t>(slot - (slot % kSellWidth)) + (slot % kSellWidth);
            sp[0] = d0;
            sp[kSellWidth] = d1;
            sp[2 * kSellWidth] = d2;
          }
        }
        int n = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
#pragma unroll
          for (int b2 = a; b2 < 4; ++b2) acc[n++] += w * (j0[a] * j0[b2] + j1[a] * j1[b2]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) acc[10 + a] += w * (j0[a] * ob.r[0] + j1[a] * ob.r[1]);
        bad = bad || !(isfinite(ob.r[0]) && isfinite(ob.r[1]) && isfinite(ob.iz) &&
                       isfinite(ob.d02) && isfinite(ob.d12));
      } else {
        PoseObs ob;
        ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
        const double w = ob.sw * ob.sw;
        if (obs_w != nullptr) {
          obs_w[o] = w;
          const int slot = __ldg(ix.obs_slot + o);
          if (slot >= 0) sell_w[slot] = w;
        }
        int n = 0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
          for (int b2 = a; b2 < 3; ++b2) {
            acc[n++] += w * (ob.T[0][a] * ob.T[0][b2] + ob.T[1][a] * ob.T[1][b2] +
                             ob.T[2][a] * ob.T[2][b2] + ob.T[3][a] * ob.T[3][b2]);
          }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          acc[6 + a] += w * (ob.T[0][a] * ob.r[0] + ob.T[1][a] * ob.r[1] + ob.T[2][a] * ob.r[2] +
                             ob.T[3][a] * ob.r[3]);
        }
        bad = bad || !(isfinite(ob.r[0]) && isfinite(ob.r[1]) && isfinite(ob.r[2]) &&
                       isfinite(ob.r[3]));
      }
      bad = bad || !(isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]) && isfinite(x[3]));
    }
    tile_allreduce<NV>(acc, t, has_obs, lm, ix.lm_ptr);
    if (is_head(t, has_obs, lm, ix.lm_ptr, o_first)) {
      double* h = lm_hraw + 10 * static_cast<size_t>(lm);
      double* g = lm_graw + 4 * static_cast<size_t>(lm);
      double* s = lm_scale + 4 * static_cast<size_t>(lm);
      if (JOINT) {
#pragma unroll
        for (int k = 0; k < 10; ++k) h[k] = acc[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) g[k] = acc[10 + k];
        s[0] = 1.0 / (eps + sqrt(acc[0]));
        s[1] = 1.0 / (eps + sqrt(acc[4]));
        s[2] = 1.0 / (eps + sqrt(acc[7]));
        s[3] = 1.0 / (eps + sqrt(acc[9]));
      } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) h[k] = acc[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) g[k] = acc[6 + k];
        g[3] = 0.0;
        s[0] = scale_jl ? 1.0 / (eps + sqrt(acc[0])) : 1.0;
        s[1] = scale_jl ? 1.0 / (eps + sqrt(acc[3])) : 1.0;
        s[2] = scale_jl ? 1.0 / (eps + sqrt(acc[5])) : 1.0;
        s[3] = 1.0;
      }
      bool fin = true;
#pragma unroll
      for (int k = 0; k < NV; ++k) fin = fin && isfinite(acc[k]);
      bad = bad || !fin;
    }
    if (bad) atomicOr(flags, 1);
  }
}

// ------------------------------------------------------------------------------------------
// per solve, per landmark: Hll^-1 (with landmark damping), H_r = scale o (Pi) Hll^-1 Jl^T r,
// and the [X | H] record the camera-major pass gathers
// ------------------------------------------------------------------------------------------
// x, s: landmark and column scales; h (10), g (4): the raw sums of the linearisation.  Out: inv = Hll^-1 (packed),
// H = scale o (Pi) Hll^-1 (Pi^T) (scale o g), fold (10; 6 used in step 1)
template <bool JOINT>
__device__ __forceinline__ void prep_one(const double (&x)[4], const double (&s)[4], const double* h, const double* g,
                                         double lambda_lm, double (&inv)[6], double (&H)[4], double (&fold)[10]) {
  double hll[6];
  H[0] = H[1] = H[2] = H[3] = 0.0;
  if (JOINT) {
    // A = (s s^T) o hraw (4x4), Hll = Pi^T A Pi + lambda I
    double A[4][4];
    {
      int n = 0;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 4; ++b2) {
          const double v = s[a] * s[b2] * h[n++];
          A[a][b2] = v;
          A[b2][a] = v;
        }
      }
    }
    Reflector<4> pi;
    pi.make(x);
    double col[3][4];   // columns of Pi
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double e[3] = {0, 0, 0};
      e[k] = 1.0;
      pi.apply(e, col[k]);
    }
    double M[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double ac[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        ac[a] = A[a][0] * col[k][0] + A[a][1] * col[k][1] + A[a][2] * col[k][2] + A[a][3] * col[k][3];
      }
#pragma unroll
      for (int j = 0; j < 3; ++j) M[j][k] = dot4(col[j], ac);
    }
    hll[0] = M[0][0] + lambda_lm;
    hll[1] = 0.5 * (M[0][1] + M[1][0]);
    hll[2] = 0.5 * (M[0][2] + M[2][0]);
    hll[3] = M[1][1] + lambda_lm;
    hll[4] = 0.5 * (M[1][2] + M[2][1]);
    hll[5] = M[2][2] + lambda_lm;
    inv3_sym(hll, inv);
    double sg[4], g3[3], h3[3], h4[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) sg[a] = s[a] * g[a];
    pi.apply_t(sg, g3);
    sym3_mul(inv, g3, h3);
    pi.apply(h3, h4);
#pragma unroll
    for (int a = 0; a < 4; ++a) H[a] = s[a] * h4[a];
    // fold = S Pi Hll^-1 Pi^T S (4x4, symmetric): H_l = fold G_l in the power-series term
    double F[4][4];
#pragma unroll
    for (int nn = 0; nn < 4; ++nn) {
      double e4[4] = {0, 0, 0, 0}, f3[3], k3[3], k4[4];
      e4[nn] = s[nn];
      pi.apply_t(e4, f3);
      sym3_mul(inv, f3, k3);
      pi.apply(k3, k4);
#pragma unroll
      for (int a = 0; a < 4; ++a) F[a][nn] = s[a] * k4[a];
    }
    {
      int nn = 0;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 4; ++b2) fold[nn++] = 0.5 * (F[a][b2] + F[b2][a]);
      }
    }
  } else {
    hll[0] = s[0] * s[0] * h[0] + lambda_lm;
    hll[1] = s[0] * s[1] * h[1];
    hll[2] = s[0] * s[2] * h[2];
    hll[3] = s[1] * s[1] * h[3] + lambda_lm;
    hll[4] = s[1] * s[2] * h[4];
    hll[5] = s[2] * s[2] * h[5] + lambda_lm;
    inv3_sym(hll, inv);
    double sg[3], h3[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) sg[a] = s[a] * g[a];
    sym3_mul(inv, sg, h3);
#pragma unroll
    for (int a = 0; a < 3; ++a) H[a] = s[a] * h3[a];
    fold[0] = s[0] * s[0] * inv[0];
    fold[1] = s[0] * s[1] * inv[1];
    fold[2] = s[0] * s[2] * inv[2];
    fold[3] = s[1] * s[1] * inv[3];
    fold[4] = s[1] * s[2] * inv[4];
    fold[5] = s[2] * s[2] * inv[5];
    fold[6] = fold[7] = fold[8] = fold[9] = 0.0;
  }
}

// landmarks with more than 32 observations: everything by landmark (k_*_long and long_landmark_warp read it there)
template <bool JOINT>
__global__ void __launch_bounds__(kBlock)
k_prep_long(int num_long, const int* __restrict__ long_lm, const double* __restrict__ X,
            const double* __restrict__ lm_hraw, const double* __restrict__ lm_graw,
            const double* __restrict__ lm_scale, double lambda_lm, const double* __restrict__ lambda_dev,
            double* __restrict__ hll_inv, double* __restrict__ lm_rec, double* __restrict__ lm_fold) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num_long) return;
  if (lambda_dev != nullptr) lambda_lm = *lambda_dev;
  const int l = long_lm[i];
  double x[4], s[4], inv[6], H[4], fold[10];
  load_lm4(X, l, x);
  load_lm4(lm_scale, l, s);
  prep_one<JOINT>(x, s, lm_hraw + 10 * static_cast<size_t>(l), lm_graw + 4 * static_cast<size_t>(l), lambda_lm, inv,
                  H, fold);
  double* hi = hll_inv + 6 * static_cast<size_t>(l);
#pragma unroll
  for (int k = 0; k < 6; ++k) hi[k] = inv[k];
  double* fo = lm_fold + 10 * static_cast<size_t>(l);
#pragma unroll
  for (int k = 0; k < 10; ++k) fo[k] = fold[k];
  double* rec = lm_rec + kLmRec * static_cast<size_t>(l);
  rec[kLmRecX0] = x[0], rec[kLmRecX0 + 1] = x[1], rec[kLmRecX2] = x[2], rec[kLmRecX2 + 1] = x[3];
  rec[kLmRecH0] = H[0], rec[kLmRecH0 + 1] = H[1], rec[kLmRecH2] = H[2], rec[kLmRecH2 + 1] = H[3];
}

// the landmarks of the sliced-ELL set, one thread per slot: the sums of the linearisation come in and Hll^-1
// and the fold go out as lane-major planes (one coalesced line per component and slice, what the walks read);
// the [X | H] record of the camera-major passes and Hll^-1 for the camera-major kernels of PCG / CHOLESKY go
// out by landmark
template <bool JOINT>
__global__ void __launch_bounds__(kBlock)
k_prep_sell(int slots, const int* __restrict__ sell_lm, const double* __restrict__ sell_x,
            const double* __restrict__ sell_hraw, const double* __restrict__ sell_graw,
            const double* __restrict__ sell_scale, double lambda_lm, const double* __restrict__ lambda_dev,
            double* __restrict__ sell_hinv, double* __restrict__ sell_fold, double* __restrict__ hll_inv,
            double* __restrict__ lm_rec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots) return;
  if (lambda_dev != nullptr) lambda_lm = *lambda_dev;
  const int sl = i / kSellWidth, lane = i % kSellWidth;
  const int lm = sell_lm[i];
  double* ip = sell_hinv + 6 * kSellWidth * static_cast<size_t>(sl) + lane;
  double* fp = sell_fold + 10 * kSellWidth * static_cast<size_t>(sl) + lane;
  if (lm < 0) {   // padding of the last slice of a window: nothing reads it, keep it finite
#pragma unroll
    for (int k = 0; k < 6; ++k) ip[k * kSellWidth] = 0.0;
#pragma unroll
    for (int k = 0; k < 10; ++k) fp[k * kSellWidth] = 0.0;
    return;
  }
  double x[4], s[4], h[10], g[4], inv[6], H[4], fold[10];
  {
    const double* xp = sell_x + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    const double* sp = sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    const double* gp = sell_graw + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    const double* hp = sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl) + lane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      x[k] = xp[k * kSellWidth];
      s[k] = sp[k * kSellWidth];
      g[k] = gp[k * kSellWidth];
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) h[k] = (JOINT || k < 6) ? hp[k * kSellWidth] : 0.0;
  }
  prep_one<JOINT>(x, s, h, g, lambda_lm, inv, H, fold);
#pragma unroll
  for (int k = 0; k < 6; ++k) ip[k * kSellWidth] = inv[k];
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    if (JOINT || k < 6) fp[k * kSellWidth] = fold[k];
  }
  if (hll_inv != nullptr) {   // only the camera-major kernels of PCG / CHOLESKY read Hll^-1 by landmark
    double2* hi = reinterpret_cast<double2*>(hll_inv + 6 * static_cast<size_t>(lm));
    hi[0] = make_double2(inv[0], inv[1]);
    hi[1] = make_double2(inv[2], inv[3]);
    hi[2] = make_double2(inv[4], inv[5]);
  }
  static_assert(kLmRecX0 == 0 && kLmRecH0 == 2 && kLmRecX2 == 4 && kLmRecH2 == 6, "two sectors: [X0 X1 H0 H1] [X2 X3 H2 H3]");
  double* rec = lm_rec + kLmRec * static_cast<size_t>(lm);
  const unsigned long long keep = l2_keep();
  store4_256(rec, x[0], x[1], H[0], H[1], keep);
  store4_256(rec + 4, x[2], x[3], H[2], H[3], keep);
}

// landmark-level tail shared by the E0 pass: G (sum of Jl_raw^T a over the landmark) -> H
template <bool JOINT>
__device__ __forceinline__ void landmark_solve(const double* acc, const double (&x)[4],
                                               const double (&s)[4], const double (&inv)[6],
                                               double (&H)[4]) {
  if (JOINT) {
    Reflector<4> pi;
    pi.make(x);
    double sg[4], g3[3], h3[3], h4[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) sg[a] = s[a] * acc[a];
    pi.apply_t(sg, g3);
    sym3_mul(inv, g3, h3);
    pi.apply(h3, h4);
#pragma unroll
    for (int a = 0; a < 4; ++a) H[a] = s[a] * h4[a];
  } else {
    double sg[3], h3[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) sg[a] = s[a] * acc[a];
    sym3_mul(inv, sg, h3);
#pragma unroll
    for (int a = 0; a < 3; ++a) H[a] = s[a] * h3[a];
    H[3] = 0.0;
  }
}

// ------------------------------------------------------------------------------------------
// back-substitutions.  l_diff partial sums go to scalar_part[block]; k_scalar_final adds them.
// ------------------------------------------------------------------------------------------
// VarPro (landmark_block.hpp:670-707): cameras are ALREADY updated (P), P_old is the backup.
// Fresh raw Jp/Jl/res at (P, X_old); stored scaled Jl and r are those of the linearisation
// (P_old, X_old, weights, lm_scale).  `inc` is the scaled-space pose increment (SURVEY H1).
__global__ void POVAR_BOUNDS_BACKSUB
k_backsub_varpro_long(DeviceIndex ix, const double* __restrict__ P, const double* __restrict__ P_old,
                 double* __restrict__ X, const double* __restrict__ inc, double c1, double c2,
                 Robust rb, const double* __restrict__ lm_scale, double* __restrict__ scalar_part) {
  __shared__ double smem[kBlock / 32];
  const Robust none = {NORM_NONE, 1.0};
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  double ld[1] = {0.0};
  for (int tile = warp; tile < ix.num_long; tile += nwarps) {
    const TileLane t(ix, tile);
    double acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.0;
    int lm = __ldg(ix.obs_lm + t.tb), o_first = -1;
    bool has_obs = false;
    double x[4] = {0, 0, 0, 0};
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      has_obs = true;
      if (o_first < 0) o_first = o;
      lm = __ldg(ix.obs_lm + o);
      Cam3x4 cam;
      load_cam(P, __ldg(ix.obs_cam + o), cam);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, x, c1, c2, none);   // helper.cpp:382-454: no robust weight
      int n = 0;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 3; ++b2) {
          acc[n++] += ob.T[0][a] * ob.T[0][b2] + ob.T[1][a] * ob.T[1][b2] + ob.T[2][a] * ob.T[2][b2] +
                      ob.T[3][a] * ob.T[3][b2];
        }
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        acc[6 + a] += ob.T[0][a] * ob.r[0] + ob.T[1][a] * ob.r[1] + ob.T[2][a] * ob.r[2] +
                      ob.T[3][a] * ob.r[3];
      }
    }
    tile_allreduce<9>(acc, t, has_obs, lm, ix.lm_ptr);
    double hll[6], inv[6], tmp[3], il[3];
#pragma unroll
    for (int k = 0; k < 6; ++k) hll[k] = acc[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) tmp[k] = acc[6 + k];
    inv3_sym(hll, inv);
    sym3_mul(inv, tmp, il);
#pragma unroll
    for (int k = 0; k < 3; ++k) il[k] = -il[k];
    double s[4];
    load_lm4(lm_scale, lm, s);
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      const int c = __ldg(ix.obs_cam + o);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      double i0[4], i1[4], i2[4], jp[4];
      const double* ic = inc + 12 * static_cast<size_t>(c);
      load4(ic, i0);
      load4(ic + 4, i1);
      load4(ic + 8, i2);
      pose_jp_mul(x, uv.x, uv.y, c1, c2, i0, i1, i2, jp);   // fresh, unscaled, unweighted Jp
      Cam3x4 cam_old;
      load_cam(P_old, c, cam_old);
      PoseObs old;
      old.eval(cam_old, uv.x, uv.y, x, c1, c2, rb);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double jl = old.sw * (old.T[q][0] * s[0] * il[0] + old.T[q][1] * s[1] * il[1] +
                                    old.T[q][2] * s[2] * il[2]);
        const double ji = jp[q] + jl;
        ld[0] -= ji * (0.5 * ji + old.sw * old.r[q]);
      }
    }
    __syncwarp();
    if (is_head(t, has_obs, lm, ix.lm_ptr, o_first)) {
      double* xo = X + 4 * static_cast<size_t>(lm);
      xo[0] += il[0];
      xo[1] += il[1];
      xo[2] += il[2];
    }
  }
  block_reduce<1>(ld, smem);
  if (threadIdx.x == 0) scalar_part[blockIdx.x] = ld[0];
}

// PoBA (landmark_block.hpp:625-656): stored scaled Jp, Jl, r at the linearisation point, which is
// the current state; y = pose_scale o inc.
__global__ void __launch_bounds__(kBlock)
k_backsub_poba_long(DeviceIndex ix, const double* __restrict__ P, double* __restrict__ X,
               const double* __restrict__ y, double c1, double c2, Robust rb,
               const double* __restrict__ lm_scale, const double* __restrict__ hll_inv,
               double* __restrict__ scalar_part) {
  __shared__ double smem[kBlock / 32];
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  double ld[1] = {0.0};
  for (int tile = warp; tile < ix.num_long; tile += nwarps) {
    const TileLane t(ix, tile);
    double acc[3] = {0, 0, 0};
    int lm = __ldg(ix.obs_lm + t.tb), o_first = -1;
    bool has_obs = false;
    double x[4] = {0, 0, 0, 0};
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      has_obs = true;
      if (o_first < 0) o_first = o;
      lm = __ldg(ix.obs_lm + o);
      const int c = __ldg(ix.obs_cam + o);
      Cam3x4 cam;
      load_cam(P, c, cam);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
      double y0[4], y1[4], y2[4], a[4];
      const double* yc = y + 12 * static_cast<size_t>(c);
      load4(yc, y0);
      load4(yc + 4, y1);
      load4(yc + 8, y2);
      pose_jp_mul(x, uv.x, uv.y, c1, c2, y0, y1, y2, a);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        double sum = 0.0;
#pragma unroll
        for (int q = 0; q < 4; ++q) sum += ob.T[q][k] * (ob.sw * ob.r[q] + ob.sw * a[q]);
        acc[k] += ob.sw * sum;
      }
    }
    tile_allreduce<3>(acc, t, has_obs, lm, ix.lm_ptr);
    double s[4], inv[6], st[3], il[3];
    load_lm4(lm_scale, lm, s);
    {
      const double* hi = hll_inv + 6 * static_cast<size_t>(lm);
#pragma unroll
      for (int k = 0; k < 6; ++k) inv[k] = hi[k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) st[k] = s[k] * acc[k];
    sym3_mul(inv, st, il);
#pragma unroll
    for (int k = 0; k < 3; ++k) il[k] = -il[k];
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      const int c = __ldg(ix.obs_cam + o);
      Cam3x4 cam;
      load_cam(P, c, cam);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
      double y0[4], y1[4], y2[4], a[4];
      const double* yc = y + 12 * static_cast<size_t>(c);
      load4(yc, y0);
      load4(yc + 4, y1);
      load4(yc + 8, y2);
      pose_jp_mul(x, uv.x, uv.y, c1, c2, y0, y1, y2, a);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double jl = ob.sw * (ob.T[q][0] * s[0] * il[0] + ob.T[q][1] * s[1] * il[1] +
                                   ob.T[q][2] * s[2] * il[2]);
        const double ji = ob.sw * a[q] + jl;
        ld[0] -= ji * (0.5 * ji + ob.sw * ob.r[q]);
      }
    }
    __syncwarp();
    if (is_head(t, has_obs, lm, ix.lm_ptr, o_first)) {
      double* xo = X + 4 * static_cast<size_t>(lm);
      xo[0] += s[0] * il[0];   // "scale only after computing model cost change", :653
      xo[1] += s[1] * il[1];
      xo[2] += s[2] * il[2];
    }
  }
  block_reduce<1>(ld, smem);
  if (threadIdx.x == 0) scalar_part[blockIdx.x] = ld[0];
}

// joint (landmark_block.hpp:574-623): y = pose_scale o (Pi_c inc11)
__global__ void POVAR_BOUNDS_BACKSUB
k_backsub_joint_long(DeviceIndex ix, const double* __restrict__ P, double* __restrict__ X,
                const double* __restrict__ y, Robust rb, const double* __restrict__ lm_scale,
                const double* __restrict__ hll_inv, double* __restrict__ scalar_part) {
  __shared__ double smem[kBlock / 32];
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  double ld[1] = {0.0};
  for (int tile = warp; tile < ix.num_long; tile += nwarps) {
    const TileLane t(ix, tile);
    double acc[4] = {0, 0, 0, 0};
    int lm = __ldg(ix.obs_lm + t.tb), o_first = -1;
    bool has_obs = false;
    double x[4] = {0, 0, 0, 0};
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      has_obs = true;
      if (o_first < 0) o_first = o;
      lm = __ldg(ix.obs_lm + o);
      const int c = __ldg(ix.obs_cam + o);
      Cam3x4 cam;
      load_cam(P, c, cam);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, x, rb);
      double y0[4], y1[4], y2[4], a[2], j0[4], j1[4];
      const double* yc = y + 12 * static_cast<size_t>(c);
      load4(yc, y0);
      load4(yc + 4, y1);
      load4(yc + 8, y2);
      ob.jp_mul(x, y0, y1, y2, a);
      ob.jl_rows(cam, j0, j1);
      const double e0 = ob.sw * ob.r[0] + ob.sw * a[0], e1 = ob.sw * ob.r[1] + ob.sw * a[1];
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[k] += ob.sw * (j0[k] * e0 + j1[k] * e1);
    }
    tile_allreduce<4>(acc, t, has_obs, lm, ix.lm_ptr);
    load_lm4(X, lm, x);
    double s[4], inv[6];
    load_lm4(lm_scale, lm, s);
    {
      const double* hi = hll_inv + 6 * static_cast<size_t>(lm);
#pragma unroll
      for (int k = 0; k < 6; ++k) inv[k] = hi[k];
    }
    Reflector<4> pi;
    pi.make(x);
    double st[4], t3[3], i3[3], i4[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) st[k] = s[k] * acc[k];
    pi.apply_t(st, t3);
    sym3_mul(inv, t3, i3);
#pragma unroll
    for (int k = 0; k < 3; ++k) i3[k] = -i3[k];
    pi.apply(i3, i4);
    for (int o = t.tb + t.lane; o < t.te; o += 32) {
      const int c = __ldg(ix.obs_cam + o);
      Cam3x4 cam;
      load_cam(P, c, cam);
      load_lm4(X, lm, x);
      const double2 uv = ix.obs_uv[o];
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, x, rb);
      double y0[4], y1[4], y2[4], a[2], j0[4], j1[4];
      const double* yc = y + 12 * static_cast<size_t>(c);
      load4(yc, y0);
      load4(yc + 4, y1);
      load4(yc + 8, y2);
      ob.jp_mul(x, y0, y1, y2, a);
      ob.jl_rows(cam, j0, j1);
      double l0 = 0.0, l1 = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        l0 += j0[k] * s[k] * i4[k];
        l1 += j1[k] * s[k] * i4[k];
      }
      const double ji0 = ob.sw * a[0] + ob.sw * l0, ji1 = ob.sw * a[1] + ob.sw * l1;
      ld[0] -= ji0 * (0.5 * ji0 + ob.sw * ob.r[0]) + ji1 * (0.5 * ji1 + ob.sw * ob.r[1]);
    }
    __syncwarp();
    if (is_head(t, has_obs, lm, ix.lm_ptr, o_first)) {
      double* xo = X + 4 * static_cast<size_t>(lm);
#pragma unroll
      for (int k = 0; k < 4; ++k) xo[k] += s[k] * i4[k];   // :621-622
    }
  }
  block_reduce<1>(ld, smem);
  if (threadIdx.x == 0) scalar_part[blockIdx.x] = ld[0];
}

// ------------------------------------------------------------------------------------------
// The same passes for the landmarks of the sliced-ELL set (1..32 observations): operations of k_sell_walk.
// A lane owns a landmark, meets its observations in camera order and keeps the sums in registers; the camera
// data come from the staged table -- [P | pad] (kCamTab1 doubles) or [A | B | pad] (kCamTab2 doubles), packed
// from the 12-vectors per camera right before the walk (k_pack_cam_tab).
// The model decrease of a back-substitution, l_diff = -sum_i ji (ji / 2 + e_i) with ji = a_i + Jl_i dl, needs the
// landmark increment dl, which is only known after the landmark's sums: the tile kernels walk the
// observations twice.  Here the square is expanded,
//   sum_i ji (ji / 2 + e_i) = sum_i (a_i^2 / 2 + a_i e_i) + dl^T sum_i Jl_i^T (a_i + e_i) + dl^T (sum_i Jl_i^T Jl_i) dl / 2,
// the first two sums are made in the one walk and the third is the landmark's Jl^T Jl block of the
// linearisation (lm_hraw): one walk, same value up to rounding.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void rec_cam(const double2* __restrict__ rec, Cam3x4& m) {
  const double2 a0 = rec[0], a1 = rec[1], b0 = rec[2], b1 = rec[3], c0 = rec[4], c1 = rec[5];
  m.r0[0] = a0.x; m.r0[1] = a0.y; m.r0[2] = a1.x; m.r0[3] = a1.y;
  m.r1[0] = b0.x; m.r1[1] = b0.y; m.r1[2] = b1.x; m.r1[3] = b1.y;
  m.r2[0] = c0.x; m.r2[1] = c0.y; m.r2[2] = c1.x; m.r2[3] = c1.y;
}
__device__ __forceinline__ void rec_vec12(const double2* __restrict__ rec, double (&y0)[4], double (&y1)[4],
                                          double (&y2)[4]) {
  const double2 a0 = rec[0], a1 = rec[1], b0 = rec[2], b1 = rec[3], c0 = rec[4], c1 = rec[5];
  y0[0] = a0.x; y0[1] = a0.y; y0[2] = a1.x; y0[3] = a1.y;
  y1[0] = b0.x; y1[1] = b0.y; y1[2] = b1.x; y1[3] = b1.y;
  y2[0] = c0.x; y2[1] = c0.y; y2[2] = c1.x; y2[3] = c1.y;
}

// table[c] = [A_c (12) | pad]  or  [A_c (12) | B_c (12) | pad]
__global__ void __launch_bounds__(kBlock)
k_pack_cam_tab(int C, int stride, const double* __restrict__ A, const double* __restrict__ B,
               double* __restrict__ table) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= C * 14) return;
  const int c = idx / 14, k = idx % 14;
  double* r = table + static_cast<size_t>(stride) * c;
  if (k < 12) {
    r[k] = A[12 * static_cast<size_t>(c) + k];
    if (B != nullptr) r[12 + k] = B[12 * static_cast<size_t>(c) + k];
  } else {
    r[(B != nullptr ? 24 : 12) + (k - 12)] = 0.0;
  }
}

// what every one of these walks shares: the stream, the landmark of the lane, the l_diff partial of the block
struct WalkBase {
  static constexpr int kStage = kStagePose;
  static constexpr int kWarpsPerSm = 16;   // 100 - 128 registers per lane
  __device__ __forceinline__ bool skip() const { return false; }
  template <class Lane>
  __device__ __forceinline__ void init(Lane& st) const {
    st.lm1 = -2;   // nothing fetched yet
  }
  __device__ __forceinline__ void issue(const DeviceIndex& ix, int row, unsigned char* stage,
                                        unsigned long long* bar) const {
    issue_cam_uv(ix, row, stage, bar);
  }
  __device__ __forceinline__ static double2 uv_of(const unsigned char* stage, int lane) {
    return reinterpret_cast<const double2*>(stage + 128)[lane];
  }
  // The landmark of this lane in slice `sl` and its coordinates (x0 for an idle lane).  The gather X[lm] is
  // two dependent trips to memory per slice; it is taken off the critical path by running ahead: the index
  // two slices ahead and the coordinates one slice ahead travel while the current slice is walked.
  template <class Lane>
  __device__ __forceinline__ static void open_landmark(Lane& st, const DeviceIndex& ix, const double* __restrict__ X,
                                                       int sl, int lane, int last, double x0) {
    const int* lmp = ix.sell_lm + kSellWidth * static_cast<size_t>(sl) + lane;
    if (st.lm1 == -2) {   // first slice of the warp (every lane starts with -2)
      st.lm1 = __ldcs(lmp);
      st.lm2 = sl < last ? __ldcs(lmp + kSellWidth) : -1;
      fetch(X, st.lm1, x0, st.x1);
    }
    st.lm = st.lm1;
#pragma unroll
    for (int k = 0; k < 4; ++k) st.x[k] = st.x1[k];
    st.lm1 = st.lm2;
    fetch(X, st.lm1, x0, st.x1);
    st.lm2 = sl + 2 <= last ? __ldcs(lmp + 2 * kSellWidth) : -1;
  }
  __device__ __forceinline__ static void fetch(const double* __restrict__ X, int lm, double x0, double (&x)[4]) {
    if (lm >= 0) {
      load_lm4(X, lm, x);
    } else {
      x[0] = x0;
      x[1] = x[2] = x[3] = 0.0;
    }
  }
  __device__ __forceinline__ static void block_sum_to(double v, double* __restrict__ out) {
    __shared__ double smem[32];
    double ld[1] = {v};
    block_reduce<1>(ld, smem);
    if (threadIdx.x == 0) out[blockIdx.x] = ld[0];
  }
};

// VarPro initialisation (k_init_varproj) for the sliced-ELL landmarks: the same Givens row updates, in camera order
struct InitVarprojOp : WalkBase {
  static constexpr int kRec = kCamTab1;
  double c1, c2;
  double* X;

  struct Lane {
    int lm, lm1;   // (lm1: WalkBase::init's marker, unused: nothing is gathered per landmark)
    double R[6], d[3];
  };

  __device__ __forceinline__ void open(Lane& st, const DeviceIndex& ix, int sl, int lane, int) const {
    st.lm = __ldcs(ix.sell_lm + kSellWidth * static_cast<size_t>(sl) + lane);
#pragma unroll
    for (int k = 0; k < 6; ++k) st.R[k] = 0.0;
    st.d[0] = st.d[1] = st.d[2] = 0.0;
  }

  __device__ __forceinline__ void obs(Lane& st, const double2* __restrict__ rec, const unsigned char* stage, int lane,
                                      int) const {
    Cam3x4 cam;
    rec_cam(rec, cam);
    const double2 uv = uv_of(stage, lane);
    // rows of G = T[:, 0:3], z = -(T[:,3]) + [0 0 c2 u c2 v]   (helper.cpp:224-237)
    givens_row(st.R, st.d, c1 * (cam.r0[0] - cam.r2[0] * uv.x), c1 * (cam.r0[1] - cam.r2[1] * uv.x),
               c1 * (cam.r0[2] - cam.r2[2] * uv.x), c1 * (cam.r2[3] * uv.x - cam.r0[3]));
    givens_row(st.R, st.d, c1 * (cam.r1[0] - cam.r2[0] * uv.y), c1 * (cam.r1[1] - cam.r2[1] * uv.y),
               c1 * (cam.r1[2] - cam.r2[2] * uv.y), c1 * (cam.r2[3] * uv.y - cam.r1[3]));
    givens_row(st.R, st.d, c2 * cam.r0[0], c2 * cam.r0[1], c2 * cam.r0[2], c2 * (uv.x - cam.r0[3]));
    givens_row(st.R, st.d, c2 * cam.r1[0], c2 * cam.r1[1], c2 * cam.r1[2], c2 * (uv.y - cam.r1[3]));
  }

  __device__ __forceinline__ void close(Lane& st, const DeviceIndex&, int, int) const {
    if (st.lm < 0) return;
    const double x2 = st.R[5] != 0.0 ? st.d[2] / st.R[5] : 0.0;
    const double x1 = st.R[3] != 0.0 ? (st.d[1] - st.R[4] * x2) / st.R[3] : 0.0;
    const double x0 = st.R[0] != 0.0 ? (st.d[0] - st.R[1] * x1 - st.R[2] * x2) / st.R[0] : 0.0;
    double2* out = reinterpret_cast<double2*>(X + 4 * static_cast<size_t>(st.lm));
    out[0] = make_double2(x0, x1);
    out[1] = make_double2(x2, 1.0);
  }

  __device__ __forceinline__ void finish(Lane&, const DeviceIndex&, const CamWindow&, const double*) const {}
};

// k_lin_long for the sliced-ELL landmarks: sum_i w Jl_raw^T Jl_raw, sum_i w Jl_raw^T r, column scales
template <bool JOINT>
struct LinLandmarkOp : WalkBase {
  static constexpr int kRec = kCamTab1;
  static constexpr int kStage = kStageLin;   // camera indices, (u, v), rows of the term kernel's copy
  static constexpr int NV = JOINT ? 14 : 9;
  const double* X;
  double c1, c2;
  Robust rb;
  double eps;
  int scale_jl;
  double* sell_hraw;   // [slice][10][32] (6 planes used in step 1)
  double* sell_graw;   // [slice][4][32]
  double* sell_scale;  // [slice][4][32]
  double* sell_x;      // [slice][4][32] the landmarks of the linearisation point, for the term kernels
  double* lm_scale;    // the scales by landmark too: the camera-major kernels of PCG / CHOLESKY gather them
  int* flags;
  double* sell_d;   // step 2: what the term kernels stream, [row][3][32]
  double* sell_w;   // step 1 with HUBER: [row][32]

  struct Lane {
    int lm, lm1, lm2, row0;
    bool bad;
    double x[4], x1[4], acc[NV];
  };

  __device__ __forceinline__ void issue(const DeviceIndex& ix, int row, unsigned char* stage,
                                        unsigned long long* bar) const {
    const size_t slot = kSellWidth * static_cast<size_t>(row);
    mbar_expect_tx(bar, kStageLin);
    bulk_stream_g2s(stage, ix.sell_cam + slot, 128u, bar);
    bulk_stream_g2s(stage + 128, ix.sell_uv + slot, 512u, bar);
    bulk_stream_g2s(stage + 640, ix.sell_row_e0 + slot, 32u, bar);
  }

  __device__ __forceinline__ void open(Lane& st, const DeviceIndex& ix, int sl, int lane, int last) const {
    open_landmark(st, ix, X, sl, lane, last, 0.0);
    st.row0 = __ldg(ix.slice_ptr + sl);
    st.bad = false;
#pragma unroll
    for (int k = 0; k < NV; ++k) st.acc[k] = 0.0;
  }

  __device__ __forceinline__ void obs(Lane& st, const double2* __restrict__ rec, const unsigned char* stage, int lane,
                                      int row) const {
    Cam3x4 cam;
    rec_cam(rec, cam);
    const double2 uv = uv_of(stage, lane);
    if (JOINT) {
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, st.x, rb);
      double j0[4], j1[4];
      ob.jl_rows(cam, j0, j1);
      const double w = ob.sw * ob.sw;
      // where the term kernel reads this observation (its copy has other rows inside a slice)
      const int row_e0 = st.row0 + stage[640 + lane];
      double* sp = sell_d + 3 * kSellWidth * static_cast<size_t>(row_e0) + lane;
      sp[0] = ob.sw * ob.iz;
      sp[kSellWidth] = ob.sw * ob.d02;
      sp[2 * kSellWidth] = ob.sw * ob.d12;
      int n = 0;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 4; ++b2) st.acc[n++] += w * (j0[a] * j0[b2] + j1[a] * j1[b2]);
      }
#pragma unroll
      for (int a = 0; a < 4; ++a) st.acc[10 + a] += w * (j0[a] * ob.r[0] + j1[a] * ob.r[1]);
      st.bad = st.bad || !(isfinite(ob.r[0]) && isfinite(ob.r[1]) && isfinite(ob.iz) && isfinite(ob.d02) &&
                           isfinite(ob.d12));
    } else {
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, st.x, c1, c2, rb);
      const double w = ob.sw * ob.sw;
      if (sell_w != nullptr) sell_w[kSellWidth * static_cast<size_t>(st.row0 + stage[640 + lane]) + lane] = w;
      int n = 0;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 3; ++b2) {
          st.acc[n++] += w * (ob.T[0][a] * ob.T[0][b2] + ob.T[1][a] * ob.T[1][b2] + ob.T[2][a] * ob.T[2][b2] +
                              ob.T[3][a] * ob.T[3][b2]);
        }
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        st.acc[6 + a] += w * (ob.T[0][a] * ob.r[0] + ob.T[1][a] * ob.r[1] + ob.T[2][a] * ob.r[2] +
                              ob.T[3][a] * ob.r[3]);
      }
      st.bad = st.bad || !(isfinite(ob.r[0]) && isfinite(ob.r[1]) && isfinite(ob.r[2]) && isfinite(ob.r[3]));
    }
  }

  // one coalesced line per component and slice (idle lanes write zeros: x = 0, sums = 0, scale = 1 / eps)
  __device__ __forceinline__ void close(Lane& st, const DeviceIndex&, int sl, int lane) const {
    double* h = sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl) + lane;
    double* g = sell_graw + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    double* sp = sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    double* xp = sell_x + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    double s[4];
    if (JOINT) {
#pragma unroll
      for (int k = 0; k < 10; ++k) h[k * kSellWidth] = st.acc[k];
#pragma unroll
      for (int k = 0; k < 4; ++k) g[k * kSellWidth] = st.acc[10 + k];
      s[0] = 1.0 / (eps + sqrt(st.acc[0]));
      s[1] = 1.0 / (eps + sqrt(st.acc[4]));
      s[2] = 1.0 / (eps + sqrt(st.acc[7]));
      s[3] = 1.0 / (eps + sqrt(st.acc[9]));
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) h[k * kSellWidth] = st.acc[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) g[k * kSellWidth] = st.acc[6 + k];
      g[3 * kSellWidth] = 0.0;
      s[0] = scale_jl ? 1.0 / (eps + sqrt(st.acc[0])) : 1.0;
      s[1] = scale_jl ? 1.0 / (eps + sqrt(st.acc[3])) : 1.0;
      s[2] = scale_jl ? 1.0 / (eps + sqrt(st.acc[5])) : 1.0;
      s[3] = 1.0;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      sp[k * kSellWidth] = s[k];
      xp[k * kSellWidth] = st.x[k];
    }
    if (st.lm < 0) return;
    double2* so = reinterpret_cast<double2*>(lm_scale + 4 * static_cast<size_t>(st.lm));
    so[0] = make_double2(s[0], s[1]);
    so[1] = make_double2(s[2], s[3]);
    bool fin = isfinite(st.x[0]) && isfinite(st.x[1]) && isfinite(st.x[2]) && isfinite(st.x[3]);
#pragma unroll
    for (int k = 0; k < NV; ++k) fin = fin && isfinite(st.acc[k]);
    if (st.bad || !fin) atomicOr(flags, 1);
  }

  __device__ __forceinline__ void finish(Lane&, const DeviceIndex&, const CamWindow&, const double*) const {}
};

// VarPro back-substitution, first walk (table [P_new]): the closed-form landmark step at the new cameras,
//   il = -(sum_i T^T T)^-1 sum_i T^T r   (landmark_block.hpp:670-690, no robust weight, helper.cpp:382-454),
// kept in lm_step; X is updated by the second walk, which still needs the old landmark
struct BacksubVarproStepOp : WalkBase {
  static constexpr int kRec = kCamTab1;
  const double* X;
  double c1, c2;
  double* sell_step;   // [slice][4][32]

  struct Lane {
    int lm, lm1, lm2;
    double x[4], x1[4], acc[9];
  };

  __device__ __forceinline__ void open(Lane& st, const DeviceIndex& ix, int sl, int lane, int last) const {
    open_landmark(st, ix, X, sl, lane, last, 0.0);
#pragma unroll
    for (int k = 0; k < 9; ++k) st.acc[k] = 0.0;
  }

  __device__ __forceinline__ void obs(Lane& st, const double2* __restrict__ rec, const unsigned char* stage, int lane,
                                      int) const {
    Cam3x4 cam;
    rec_cam(rec, cam);
    const double2 uv = uv_of(stage, lane);
    const Robust none = {NORM_NONE, 1.0};
    PoseObs ob;
    ob.eval(cam, uv.x, uv.y, st.x, c1, c2, none);
    int n = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int b2 = a; b2 < 3; ++b2) {
        st.acc[n++] += ob.T[0][a] * ob.T[0][b2] + ob.T[1][a] * ob.T[1][b2] + ob.T[2][a] * ob.T[2][b2] +
                       ob.T[3][a] * ob.T[3][b2];
      }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      st.acc[6 + a] += ob.T[0][a] * ob.r[0] + ob.T[1][a] * ob.r[1] + ob.T[2][a] * ob.r[2] + ob.T[3][a] * ob.r[3];
    }
  }

  __device__ __forceinline__ void close(Lane& st, const DeviceIndex&, int sl, int lane) const {
    double hll[6], inv[6], tmp[3], il[3];
#pragma unroll
    for (int k = 0; k < 6; ++k) hll[k] = st.acc[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) tmp[k] = st.acc[6 + k];
    inv3_sym(hll, inv);
    sym3_mul(inv, tmp, il);
    double* out = sell_step + 4 * kSellWidth * static_cast<size_t>(sl) + lane;   // (idle lanes: never read)
    out[0] = -il[0];
    out[kSellWidth] = -il[1];
    out[2 * kSellWidth] = -il[2];
  }

  __device__ __forceinline__ void finish(Lane&, const DeviceIndex&, const CamWindow&, const double*) const {}
};

// VarPro back-substitution, second walk (table [P_old | inc]): the model decrease with the Jacobians and
// residuals of the linearisation point and the fresh Jp (landmark_block.hpp:691-707), then X += il
struct BacksubVarproDiffOp : WalkBase {
  static constexpr int kRec = kCamTab2;
  double* X;
  double c1, c2;
  Robust rb;
  const double* sell_scale;
  const double* sell_hraw;
  const double* sell_step;
  double* scalar_part;

  struct Lane {
    int lm, lm1, lm2;
    double ld;
    double x[4], x1[4], A, B[3];
  };

  __device__ __forceinline__ void init(Lane& st) const {
    WalkBase::init(st);
    st.ld = 0.0;
  }

  __device__ __forceinline__ void open(Lane& st, const DeviceIndex& ix, int sl, int lane, int last) const {
    open_landmark(st, ix, X, sl, lane, last, 0.0);
    // what close() reads, towards L2: 6 + 3 + 3 planes of 256 bytes = 24 lines
    if (lane < 12) prefetch_l2(sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl) + 16 * lane);
    else if (lane < 18) prefetch_l2(sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + 16 * (lane - 12));
    else if (lane < 24) prefetch_l2(sell_step + 4 * kSellWidth * static_cast<size_t>(sl) + 16 * (lane - 18));
    st.A = 0.0;
    st.B[0] = st.B[1] = st.B[2] = 0.0;
  }

  __device__ __forceinline__ void obs(Lane& st, const double2* __restrict__ rec, const unsigned char* stage, int lane,
                                      int) const {
    Cam3x4 cam_old;
    rec_cam(rec, cam_old);
    double i0[4], i1[4], i2[4], jp[4];
    rec_vec12(rec + 6, i0, i1, i2);
    const double2 uv = uv_of(stage, lane);
    pose_jp_mul(st.x, uv.x, uv.y, c1, c2, i0, i1, i2, jp);   // fresh, unscaled, unweighted Jp
    PoseObs old;
    old.eval(cam_old, uv.x, uv.y, st.x, c1, c2, rb);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double e = old.sw * old.r[q];
      st.A += jp[q] * (0.5 * jp[q] + e);
      const double t = old.sw * (jp[q] + e);
      st.B[0] += old.T[q][0] * t;
      st.B[1] += old.T[q][1] * t;
      st.B[2] += old.T[q][2] * t;
    }
  }

  __device__ __forceinline__ void close(Lane& st, const DeviceIndex&, int sl, int lane) const {
    if (st.lm < 0) return;
    double il[3], d[3], hd[3], hs[6];
    const double* sp = sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    const double* ip = sell_step + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
    const double* hp = sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl) + lane;
#pragma unroll
    for (int k = 0; k < 6; ++k) hs[k] = __ldcs(hp + k * kSellWidth);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      il[k] = __ldcs(ip + k * kSellWidth);
      d[k] = __ldcs(sp + k * kSellWidth) * il[k];
    }
    sym3_mul(hs, d, hd);
    st.ld -= st.A + (d[0] * st.B[0] + d[1] * st.B[1] + d[2] * st.B[2]) +
             0.5 * (d[0] * hd[0] + d[1] * hd[1] + d[2] * hd[2]);
    double2* xo = reinterpret_cast<double2*>(X + 4 * static_cast<size_t>(st.lm));
    xo[0] = make_double2(st.x[0] + il[0], st.x[1] + il[1]);
    xo[1] = make_double2(st.x[2] + il[2], st.x[3]);
  }

  __device__ __forceinline__ void finish(Lane& st, const DeviceIndex&, const CamWindow&, const double*) const {
    block_sum_to(st.ld, scalar_part);
  }
};

// PoBA (landmark_block.hpp:625-656) and joint (:574-623) back-substitution (table [P | y]): stored scaled
// Jacobians and residuals at the linearisation point, which is the current state
template <bool JOINT>
struct BacksubLinPointOp : WalkBase {
  static constexpr int kRec = kCamTab2;
  static constexpr int NA = JOINT ? 4 : 3;
  double* X;
  double c1, c2;
  Robust rb;
  const double* sell_scale;
  const double* sell_hinv;   // [slice][6][32] Hll^-1 of the last solve
  const double* sell_hraw;
  double* scalar_part;

  struct Lane {
    int lm, lm1, lm2;
    double ld;
    double x[4], x1[4], S0, acc[NA];
  };

  __device__ __forceinline__ void init(Lane& st) const {
    WalkBase::init(st);
    st.ld = 0.0;
  }

  __device__ __forceinline__ void open(Lane& st, const DeviceIndex& ix, int sl, int lane, int last) const {
    open_landmark(st, ix, X, sl, lane, last, 1.0);   // x0 = 1 keeps the reflector of an idle lane well defined
    // what close() reads, towards L2: 10 + 4 + 6 planes of 256 bytes = 40 lines, two per lane
    {
      const double* hp = sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl);
      if (lane < 20) prefetch_l2(hp + 16 * lane);
      else if (lane < 28) prefetch_l2(sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + 16 * (lane - 20));
      if (lane < 12) prefetch_l2(sell_hinv + 6 * kSellWidth * static_cast<size_t>(sl) + 16 * lane);
    }
    st.S0 = 0.0;
#pragma unroll
    for (int k = 0; k < NA; ++k) st.acc[k] = 0.0;
  }

  __device__ __forceinline__ void obs(Lane& st, const double2* __restrict__ rec, const unsigned char* stage, int lane,
                                      int) const {
    Cam3x4 cam;
    rec_cam(rec, cam);
    double y0[4], y1[4], y2[4];
    rec_vec12(rec + 6, y0, y1, y2);
    const double2 uv = uv_of(stage, lane);
    if (JOINT) {
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, st.x, rb);
      double a[2], j0[4], j1[4];
      ob.jp_mul(st.x, y0, y1, y2, a);
      ob.jl_rows(cam, j0, j1);
      const double ea0 = ob.sw * a[0], ea1 = ob.sw * a[1], er0 = ob.sw * ob.r[0], er1 = ob.sw * ob.r[1];
      st.S0 += ea0 * (0.5 * ea0 + er0) + ea1 * (0.5 * ea1 + er1);
      const double e0 = er0 + ea0, e1 = er1 + ea1;
#pragma unroll
      for (int k = 0; k < 4; ++k) st.acc[k] += ob.sw * (j0[k] * e0 + j1[k] * e1);
    } else {
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, st.x, c1, c2, rb);
      double a[4];
      pose_jp_mul(st.x, uv.x, uv.y, c1, c2, y0, y1, y2, a);
      double e[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double ea = ob.sw * a[q], er = ob.sw * ob.r[q];
        st.S0 += ea * (0.5 * ea + er);
        e[q] = er + ea;
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        st.acc[k] += ob.sw * (ob.T[0][k] * e[0] + ob.T[1][k] * e[1] + ob.T[2][k] * e[2] + ob.T[3][k] * e[3]);
      }
    }
  }

  __device__ __forceinline__ void close(Lane& st, const DeviceIndex&, int sl, int lane) const {
    if (st.lm < 0) return;
    double s[4], inv[6], h[10];
    {
      const double* sp = sell_scale + 4 * kSellWidth * static_cast<size_t>(sl) + lane;
      const double* ip = sell_hinv + 6 * kSellWidth * static_cast<size_t>(sl) + lane;
      const double* hp = sell_hraw + 10 * kSellWidth * static_cast<size_t>(sl) + lane;
#pragma unroll
      for (int k = 0; k < 4; ++k) s[k] = __ldcs(sp + k * kSellWidth);
#pragma unroll
      for (int k = 0; k < 6; ++k) inv[k] = __ldcs(ip + k * kSellWidth);
#pragma unroll
      for (int k = 0; k < 10; ++k) h[k] = (JOINT || k < 6) ? __ldcs(hp + k * kSellWidth) : 0.0;
    }
    double dl[4];   // the landmark increment in raw coordinates
    if (JOINT) {
      Reflector<4> pi;
      pi.make(st.x);
      double sg[4], t3[3], i3[3], i4[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) sg[k] = s[k] * st.acc[k];
      pi.apply_t(sg, t3);
      sym3_mul(inv, t3, i3);
#pragma unroll
      for (int k = 0; k < 3; ++k) i3[k] = -i3[k];
      pi.apply(i3, i4);
#pragma unroll
      for (int k = 0; k < 4; ++k) dl[k] = s[k] * i4[k];
      // dl^T H dl with the packed symmetric 4x4 of the linearisation
      double hd[4];
      hd[0] = h[0] * dl[0] + h[1] * dl[1] + h[2] * dl[2] + h[3] * dl[3];
      hd[1] = h[1] * dl[0] + h[4] * dl[1] + h[5] * dl[2] + h[6] * dl[3];
      hd[2] = h[2] * dl[0] + h[5] * dl[1] + h[7] * dl[2] + h[8] * dl[3];
      hd[3] = h[3] * dl[0] + h[6] * dl[1] + h[8] * dl[2] + h[9] * dl[3];
      double da = 0.0;
#pragma unroll
      for (int k = 0; k < NA; ++k) da += dl[k] * st.acc[k];
      st.ld -= st.S0 + da + 0.5 * dot4(dl, hd);
    } else {
      double sg[3], il[3], hd[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) sg[k] = s[k] * st.acc[k];
      sym3_mul(inv, sg, il);
#pragma unroll
      for (int k = 0; k < 3; ++k) dl[k] = -s[k] * il[k];
      dl[3] = 0.0;
      const double hs[6] = {h[0], h[1], h[2], h[3], h[4], h[5]};
      const double d3[3] = {dl[0], dl[1], dl[2]};
      sym3_mul(hs, d3, hd);
      st.ld -= st.S0 + (dl[0] * st.acc[0] + dl[1] * st.acc[1] + dl[2] * st.acc[2]) +
               0.5 * (dl[0] * hd[0] + dl[1] * hd[1] + dl[2] * hd[2]);
    }
    double2* xo = reinterpret_cast<double2*>(X + 4 * static_cast<size_t>(st.lm));
    xo[0] = make_double2(st.x[0] + dl[0], st.x[1] + dl[1]);
    xo[1] = make_double2(st.x[2] + dl[2], st.x[3] + dl[3]);
  }

  __device__ __forceinline__ void finish(Lane& st, const DeviceIndex&, const CamWindow&, const double*) const {
    block_sum_to(st.ld, scalar_part);
  }
};

// create_homogeneous_landmark, landmark part (bal_bundle_adjustment.cpp:546-549): the 4th entry is
// already 1 in step-1 storage, written explicitly for clarity
__global__ void k_to_homogeneous(int L, double* __restrict__ X) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < L) X[4 * static_cast<size_t>(l) + 3] = 1.0;
}

// X_h <- X_h / X_h[3]  (bal_bundle_adjustment.cpp:703-705)
__global__ void k_normalize_lms(int L, double* __restrict__ X) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  double* x = X + 4 * static_cast<size_t>(l);
  const double w = x[3];
  x[0] = x[0] / w;
  x[1] = x[1] / w;
  x[2] = x[2] / w;
  x[3] = w / w;
}

// blocks of the k_*_long kernels: one warp per landmark with more than 32 observations
inline int long_grid(const DeviceState& d) {
  const int warps_per_block = kBlock / 32;
  long long blocks = (static_cast<long long>(d.ix.num_long) + warps_per_block - 1) / warps_per_block;
  const long long cap = static_cast<long long>(sm_count()) * 8;
  if (blocks > cap) blocks = cap;
  return static_cast<int>(blocks);
}

inline void count(const LaunchCfg& lc, int n = 1) {
  if (lc.launch_counter) *lc.launch_counter += n;
}

}  // namespace

int cost_blocks(const DeviceState& d) {
  long long blocks = (static_cast<long long>(d.ix.nnz) + kBlock - 1) / kBlock;
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

// l_diff partials: [blocks of the long kernel | blocks of the walk]
int scalar_blocks(const DeviceState& d) { return long_grid(d) + d.plan[4].blocks + d.plan[3].blocks; }

namespace {

// table of a once-per-trial walk: [A | pad] (B == nullptr) or [A | B | pad] per camera
void pack_cam_tab(const DeviceState& d, const double* A, const double* B, const LaunchCfg& lc) {
  const int n = d.ix.C * 14;
  k_pack_cam_tab<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(d.ix.C, B != nullptr ? kCamTab2 : kCamTab1, A, B,
                                                                     d.cam_tab);
  count(lc);
}

// sum of the l_diff partials of the long kernel (`long_blocks`) and of the walk (`walked`: it ran)
void finish_l_diff(const DeviceState& d, int long_blocks, bool walked, const LaunchCfg& lc) {
  const int walk_blocks = walked ? d.plan[4].blocks : 0;   // written behind the long kernel's partials
  k_scalar_final<<<1, kBlock, 0, lc.stream>>>(long_blocks + walk_blocks, d.scalar_part, d.trial_out + 8);
  count(lc);
}

}  // namespace

void launch_init_varproj(const DeviceState& d, const ModelParams& mp, const LaunchCfg& lc) {
  if (d.plan[3].blocks > 0) {
    pack_cam_tab(d, d.P, nullptr, lc);
    const InitVarprojOp op{{}, mp.c1, mp.c2, d.X};
    if (launch_sell_walk(d.ix, d.plan[3], d.debug_window_cams, d.cam_tab, op, lc.stream)) count(lc);
  }
  if (d.ix.num_long > 0) {
    k_init_varproj<<<(d.ix.num_long + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(
        d.ix.num_long, d.ix.long_lm, d.ix.lm_ptr, d.ix.obs_cam, d.ix.obs_uv, d.P, mp.c1, mp.c2, d.X);
    count(lc);
  }
}

void launch_flag_to_double(const DeviceState& d, const LaunchCfg& lc) {
  k_flag_to_double<<<1, 1, 0, lc.stream>>>(d.flags, d.trial_out + 9);
  count(lc);
}

void launch_cost(const DeviceState& d, const ModelParams& mp, bool joint, const LaunchCfg& lc) {
  const int blocks = cost_blocks(d);
  const Robust rb = {mp.robust_norm, mp.huber};
  if (joint) {
    k_cost<true><<<blocks, kBlock, 0, lc.stream>>>(d.ix.nnz, d.ix.obs_cam, d.ix.obs_lm, d.ix.obs_uv, d.P,
                                                   d.X, mp.c1, mp.c2, rb, d.cost_part);
  } else {
    k_cost<false><<<blocks, kBlock, 0, lc.stream>>>(d.ix.nnz, d.ix.obs_cam, d.ix.obs_lm, d.ix.obs_uv, d.P,
                                                    d.X, mp.c1, mp.c2, rb, d.cost_part);
  }
  k_cost_final<<<1, kBlock, 0, lc.stream>>>(blocks, d.ix.nnz, d.cost_part, d.cost_out, d.trial_out);
  count(lc, 2);
}

void launch_lin_landmark(const DeviceState& d, const ModelParams& mp, bool joint, bool scale_jl,
                         const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  double* sw = mp.robust_norm == NORM_HUBER ? d.sell_w : nullptr;
  if (d.plan[3].blocks > 0) {
    pack_cam_tab(d, d.P, nullptr, lc);
    if (joint) {
      const LinLandmarkOp<true> op{{},          d.X,         mp.c1,        mp.c2,    rb,         mp.jacobi_eps, 1,
                                   d.sell_hraw, d.sell_graw, d.sell_scale, d.sell_x, d.lm_scale, d.flags,       d.sell_d,
                                   nullptr};
      if (launch_sell_walk(d.ix, d.plan[3], d.debug_window_cams, d.cam_tab, op, lc.stream)) count(lc);
    } else {
      const LinLandmarkOp<false> op{{},          d.X,         mp.c1,        mp.c2,    rb,         mp.jacobi_eps,
                                    scale_jl ? 1 : 0, d.sell_hraw, d.sell_graw, d.sell_scale, d.sell_x, d.lm_scale,
                                    d.flags,     nullptr,     sw};
      if (launch_sell_walk(d.ix, d.plan[3], d.debug_window_cams, d.cam_tab, op, lc.stream)) count(lc);
    }
  }
  const int blocks = long_grid(d);
  if (blocks == 0) return;
  if (joint) {
    k_lin_long<true><<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.X, mp.c1, mp.c2, rb, mp.jacobi_eps, 1, d.lm_hraw,
                                                       d.lm_graw, d.lm_scale, d.flags, d.obs_d, nullptr, d.sell_d,
                                                       nullptr);
  } else {
    k_lin_long<false><<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.X, mp.c1, mp.c2, rb, mp.jacobi_eps,
                                                        scale_jl ? 1 : 0, d.lm_hraw, d.lm_graw, d.lm_scale, d.flags,
                                                        nullptr, mp.robust_norm == NORM_HUBER ? d.obs_w : nullptr,
                                                        nullptr, d.sell_w);
  }
  count(lc);
}

void launch_prep_landmark(const DeviceState& d, bool joint, double lambda_lm, bool hinv_by_landmark,
                          const LaunchCfg& lc, const double* lambda_dev) {
  const int slots = kSellWidth * d.ix.num_slices;
  double* hinv_out = hinv_by_landmark ? d.hll_inv : nullptr;
  if (slots > 0) {
    const int blocks = (slots + kBlock - 1) / kBlock;
    if (joint) {
      k_prep_sell<true><<<blocks, kBlock, 0, lc.stream>>>(slots, d.ix.sell_lm, d.sell_x, d.sell_hraw, d.sell_graw,
                                                          d.sell_scale, lambda_lm, lambda_dev, d.sell_hinv, d.sell_fold, hinv_out,
                                                          d.lm_rec);
    } else {
      k_prep_sell<false><<<blocks, kBlock, 0, lc.stream>>>(slots, d.ix.sell_lm, d.sell_x, d.sell_hraw, d.sell_graw,
                                                           d.sell_scale, lambda_lm, lambda_dev, d.sell_hinv, d.sell_fold, hinv_out,
                                                           d.lm_rec);
    }
    count(lc);
  }
  if (d.ix.num_long > 0) {
    const int blocks = (d.ix.num_long + kBlock - 1) / kBlock;
    if (joint) {
      k_prep_long<true><<<blocks, kBlock, 0, lc.stream>>>(d.ix.num_long, d.ix.long_lm, d.X, d.lm_hraw, d.lm_graw,
                                                          d.lm_scale, lambda_lm, lambda_dev, d.hll_inv, d.lm_rec, d.lm_fold);
    } else {
      k_prep_long<false><<<blocks, kBlock, 0, lc.stream>>>(d.ix.num_long, d.ix.long_lm, d.X, d.lm_hraw, d.lm_graw,
                                                           d.lm_scale, lambda_lm, lambda_dev, d.hll_inv, d.lm_rec, d.lm_fold);
    }
    count(lc);
  }
}

// d.P: the updated cameras, d.P_bak: those of the linearisation point
void launch_backsub_varpro(const DeviceState& d, const ModelParams& mp, const double* inc,
                           const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  const int blocks = long_grid(d);
  if (blocks > 0) {
    k_backsub_varpro_long<<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.P_bak, d.X, inc, mp.c1, mp.c2, rb,
                                                            d.lm_scale, d.scalar_part);
    count(lc);
  }
  bool walked = false;
  if (d.plan[3].blocks > 0) {
    pack_cam_tab(d, d.P, nullptr, lc);
    const BacksubVarproStepOp step{{}, d.X, mp.c1, mp.c2, d.sell_step};
    if (launch_sell_walk(d.ix, d.plan[3], d.debug_window_cams, d.cam_tab, step, lc.stream)) count(lc);
    pack_cam_tab(d, d.P_bak, inc, lc);
    const BacksubVarproDiffOp diff{{}, d.X, mp.c1, mp.c2, rb, d.sell_scale, d.sell_hraw, d.sell_step, d.scalar_part + blocks};
    walked = launch_sell_walk(d.ix, d.plan[4], d.debug_window_cams, d.cam_tab, diff, lc.stream);
    if (walked) count(lc);
  }
  finish_l_diff(d, blocks, walked, lc);
}

void launch_backsub_poba(const DeviceState& d, const ModelParams& mp, const double* y,
                         const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  const int blocks = long_grid(d);
  if (blocks > 0) {
    k_backsub_poba_long<<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.X, y, mp.c1, mp.c2, rb, d.lm_scale, d.hll_inv,
                                                          d.scalar_part);
    count(lc);
  }
  bool walked = false;
  if (d.plan[4].blocks > 0) {
    pack_cam_tab(d, d.P, y, lc);
    const BacksubLinPointOp<false> op{{}, d.X, mp.c1, mp.c2, rb, d.sell_scale, d.sell_hinv, d.sell_hraw, d.scalar_part + blocks};
    walked = launch_sell_walk(d.ix, d.plan[4], d.debug_window_cams, d.cam_tab, op, lc.stream);
    if (walked) count(lc);
  }
  finish_l_diff(d, blocks, walked, lc);
}

void launch_backsub_joint(const DeviceState& d, const ModelParams& mp, const double* y,
                          const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  const int blocks = long_grid(d);
  if (blocks > 0) {
    k_backsub_joint_long<<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.X, y, rb, d.lm_scale, d.hll_inv,
                                                           d.scalar_part);
    count(lc);
  }
  bool walked = false;
  if (d.plan[4].blocks > 0) {
    pack_cam_tab(d, d.P, y, lc);
    const BacksubLinPointOp<true> op{{}, d.X, mp.c1, mp.c2, rb, d.sell_scale, d.sell_hinv, d.sell_hraw, d.scalar_part + blocks};
    walked = launch_sell_walk(d.ix, d.plan[4], d.debug_window_cams, d.cam_tab, op, lc.stream);
    if (walked) count(lc);
  }
  finish_l_diff(d, blocks, walked, lc);
}

void launch_to_homogeneous(const DeviceState& d, const LaunchCfg& lc) {
  const int blocks = (d.ix.L + kBlock - 1) / kBlock;
  if (blocks == 0) return;
  k_to_homogeneous<<<blocks, kBlock, 0, lc.stream>>>(d.ix.L, d.X);
  count(lc);
}

void launch_normalize_joint(const DeviceState& d, const LaunchCfg& lc) {
  const int blocks = (d.ix.L + kBlock - 1) / kBlock;
  if (blocks == 0) return;
  k_normalize_lms<<<blocks, kBlock, 0, lc.stream>>>(d.ix.L, d.X);
  count(lc);
}

}  // namespace povar
