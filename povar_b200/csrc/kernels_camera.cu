// Camera-major kernels: everything that reduces over the observations of one camera, plus the
// per-camera dense work (12x12 / 11x11 blocks) and the power-series bookkeeping.
//
// The reference scatters per-landmark results into per-camera vectors and blocks under one
// std::mutex per camera (sc/landmark_block.hpp:531-537, sc/linearization_power_varproj.hpp:393-397),
// which makes it non-reproducible with more than one thread (SURVEY F10).  Here the observation
// list is also kept camera-major (CSC, built once); a work ITEM is a fixed run of CSC entries of a
// single camera, one warp reduces an item with a fixed tree, and items are summed per camera in
// index order => bit-reproducible, no atomics.
//
// Reference loops replaced (paths relative to /root/reference/src/rootba_povar/):
//   k_kron          sc/landmark_block.hpp:272-282, 658-668 (Jp diag), :498/:530/:563 (Jp^T Jp)
//   k_cam_scale     solver/linearizor_power_varproj.cpp:66-70, 101-105
//   k_cam_binv      sc/linearization_power_varproj.hpp:91-121, 141-154
//   k_passB         sc/linearization_power_varproj.hpp:364-453 second half (Jp^T Jl ...), and the
//                   b part of sc/landmark_block.hpp:474-572
//   k_finish_b / k_term / k_series_*   sc/linearization_power_varproj.hpp:191-360
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>

#include "device_math.cuh"
#include "povar_internal.h"

namespace povar {

namespace {

constexpr int kBlock = 256;

inline void count(const LaunchCfg& lc, int n = 1) {
  if (lc.launch_counter) *lc.launch_counter += n;
}

inline int item_grid(const DeviceState& d) {
  const int warps_per_block = kBlock / 32;
  long long blocks = (static_cast<long long>(d.ix.num_items) + warps_per_block - 1) / warps_per_block;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

__device__ __forceinline__ void load_rec(const double* __restrict__ rec, int lm, double (&x)[4],
                                         double (&h)[4]) {
  const double* p = rec + kLmRec * static_cast<size_t>(lm);
  double a[4], b[4];   // [X0 X1 H0 H1], [X2 X3 H2 H3]
  const unsigned long long keep = l2_keep();
  load4_256(p, a, keep);
  load4_256(p + 4, b, keep);
  x[0] = a[0], x[1] = a[1], x[2] = b[0], x[3] = b[1];
  h[0] = a[2], h[1] = a[3], h[2] = b[2], h[3] = b[3];
}

// ------------------------------------------------------------------------------------------
// sum_i E_i (x) (X_i X_i^T) per camera: 6 x 10 unique entries.  E_i is the 3x3 symmetric matrix
// with Jp_raw^T W Jp_raw = E (x) X X^T (both observation models have Jp_raw = K (x) X^T).
// ------------------------------------------------------------------------------------------
// KIND 0 (KRON_HPP):   E_i = W K_i^T K_i            -> Jp^T Jp
// KIND 1 (KRON_SDIAG): E_i = W^2 K_i^T N_i K_i,  N_i = Jl_i Hll^-1 Jl_i^T (scaled, tangent-projected
//                      in step 2)                  -> diagonal blocks of sum_l Hpl Hll^-1 Hlp
// factors of one camera-major entry e: E[6] (packed symmetric 3x3) and Y[10] = packed X X^T
template <bool JOINT, int KIND>
__device__ __forceinline__ void kron_factors(int e, int lm, double2 uv, const Cam3x4& cam,
                                             const double* __restrict__ X, double c1, double c2, const Robust& rb,
                                             const double* __restrict__ lm_scale,
                                             const double* __restrict__ hll_inv, double* __restrict__ csc_d,
                                             double* __restrict__ csc_w, double (&E)[6], double (&Y)[10]) {
  double x[4];
  load4_256(X + 4 * static_cast<size_t>(lm), x);
  if (KIND == KRON_SDIAG) {
    double sl[4], inv[6];
    load4_256(lm_scale + 4 * static_cast<size_t>(lm), sl);
    {
      const double* hi = hll_inv + 6 * static_cast<size_t>(lm);
#pragma unroll
      for (int k = 0; k < 6; ++k) inv[k] = hi[k];
    }
    if (JOINT) {
      JointObs ob;
      ob.eval(cam, uv.x, uv.y, x, rb);
      double j0[4], j1[4];
      ob.jl_rows(cam, j0, j1);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        j0[k] *= sl[k];
        j1[k] *= sl[k];
      }
      Reflector<4> pi;
      pi.make(x);
      double t0[3], t1[3], v0[3], v1[3];
      pi.apply_t(j0, t0);             // rows of Jl_t = (Jl_raw o scale) Pi_l
      pi.apply_t(j1, t1);
      sym3_mul(inv, t0, v0);
      sym3_mul(inv, t1, v1);
      const double n00 = t0[0] * v0[0] + t0[1] * v0[1] + t0[2] * v0[2];
      const double n01 = t0[0] * v1[0] + t0[1] * v1[1] + t0[2] * v1[2];
      const double n11 = t1[0] * v1[0] + t1[1] * v1[1] + t1[2] * v1[2];
      const double w2 = ob.sw * ob.sw * ob.sw * ob.sw;
      // E = w^2 d^T N d with d = [[iz 0 d02],[0 iz d12]]
      const double a0 = n00 * ob.d02 + n01 * ob.d12, a1 = n01 * ob.d02 + n11 * ob.d12;
      E[0] = w2 * ob.iz * ob.iz * n00;
      E[1] = w2 * ob.iz * ob.iz * n01;
      E[2] = w2 * ob.iz * a0;
      E[3] = w2 * ob.iz * ob.iz * n11;
      E[4] = w2 * ob.iz * a1;
      E[5] = w2 * (ob.d02 * a0 + ob.d12 * a1);
    } else {
      PoseObs ob;
      ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
      double Z[4][3], V[4][3], N[4][4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int k = 0; k < 3; ++k) Z[q][k] = ob.T[q][k] * sl[k];
        sym3_mul(inv, Z[q], V[q]);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int r = 0; r < 4; ++r) N[q][r] = Z[q][0] * V[r][0] + Z[q][1] * V[r][1] + Z[q][2] * V[r][2];
      }
      // K rows: c1 (1 0 -u), c1 (0 1 -v), c2 (1 0 0), c2 (0 1 0);  E = w^2 K^T N K
      const double K[4][3] = {{c1, 0.0, -c1 * uv.x}, {0.0, c1, -c1 * uv.y}, {c2, 0.0, 0.0}, {0.0, c2, 0.0}};
      double G[4][3];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          G[q][k] = N[q][0] * K[0][k] + N[q][1] * K[1][k] + N[q][2] * K[2][k] + N[q][3] * K[3][k];
        }
      }
      const double w2 = ob.sw * ob.sw * ob.sw * ob.sw;
      int n = 0;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b2 = a; b2 < 3; ++b2) {
          E[n++] = w2 * (K[0][a] * G[0][b2] + K[1][a] * G[1][b2] + K[2][a] * G[2][b2] + K[3][a] * G[3][b2]);
        }
      }
    }
  } else if (JOINT) {
    JointObs ob;
    ob.eval(cam, uv.x, uv.y, x, rb);
    const double w = ob.sw * ob.sw;
    if (csc_d != nullptr) {
      double* dp = csc_d + 3 * static_cast<size_t>(e);
      dp[0] = ob.sw * ob.iz;
      dp[1] = ob.sw * ob.d02;
      dp[2] = ob.sw * ob.d12;
    }
    E[0] = w * ob.iz * ob.iz;
    E[1] = 0.0;
    E[2] = w * ob.iz * ob.d02;
    E[3] = E[0];
    E[4] = w * ob.iz * ob.d12;
    E[5] = w * (ob.d02 * ob.d02 + ob.d12 * ob.d12);
  } else {
    PoseObs ob;
    ob.eval(cam, uv.x, uv.y, x, c1, c2, rb);
    const double w = ob.sw * ob.sw;
    if (csc_w != nullptr) csc_w[e] = w;
    const double a = c1 * c1, bq = c2 * c2;
    E[0] = w * (a + bq);
    E[1] = 0.0;
    E[2] = -w * a * uv.x;
    E[3] = E[0];
    E[4] = -w * a * uv.y;
    E[5] = w * a * (uv.x * uv.x + uv.y * uv.y);
  }
  {
    int n = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = i; j < 4; ++j) Y[n++] = x[i] * x[j];
    }
  }
}

// The sums on the FP64 tensor cores.  Per camera the 6 x 10 block is a contraction over the
// observations, sum_i E_i (x) Y_i = [E_1 .. E_n] [Y_1 .. Y_n]^T: each lane makes the factors of one entry,
// the warp transposes them through shared memory into DMMA fragments (m8n8k4: A = E^T, 8 x 4 entries with
// rows 6..7 zero; B = Y, 4 entries x 8, two column tiles for the 10 entries of X X^T) and eight k-steps
// consume the 32 entries.  Four accumulator registers per lane instead of 60 (a one-lane-one-entry
// kernel ran at one block per SM), and no 60-value warp reduction at the end.
// The staging rows are 64 bytes, so plain rows put the 16-byte stores of a quarter warp on two bank groups (4-way
// conflict) and the 8-byte fragment reads of a half warp on half the banks (2-way): 290 shared-memory wavefronts
// per 32 entries, which is what bounded the kernel (l1tex 95 %).  The four 16-byte chunks of row R are therefore
// stored at chunk position q ^ swz(R), swz(R) = 2 * bit1(R) + bit2(R): stores and fragment reads are both
// conflict-free (96 wavefronts).
__device__ __forceinline__ void dmma_m8n8k4(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
}

constexpr int kKronWarps = 4;   // warps per block of k_kron_mma: 6 KB of staging each

template <bool JOINT, int KIND>
__global__ void __launch_bounds__(32 * kKronWarps, KIND == KRON_HPP ? 5 : 4)
k_kron_mma(DeviceIndex ix, const double* __restrict__ P, const double* __restrict__ X, double c1,
           double c2, Robust rb, const double* __restrict__ lm_scale, const double* __restrict__ hll_inv,
           double* __restrict__ item_kron, double* __restrict__ csc_d, double* __restrict__ csc_w) {
  __shared__ __align__(16) double stage[kKronWarps][3][32][8];   // [E | Y 0..7 | Y 8..9] per entry
  const int wib = threadIdx.x >> 5;
  const int warp = blockIdx.x * kKronWarps + wib;
  const int lane = threadIdx.x & 31;
  if (warp >= ix.num_items) return;
  const int c = __ldg(ix.item_cam + warp);
  const int eb = __ldg(ix.item_ptr + warp), ee = __ldg(ix.item_ptr + warp + 1);
  Cam3x4 cam;
  load_cam(P, c, cam);
  double (*sE)[8] = stage[wib][0];
  double (*sY0)[8] = stage[wib][1];
  double (*sY1)[8] = stage[wib][2];
  const int wz = 2 * ((lane >> 1) & 1) + ((lane >> 2) & 1);   // swz(row) of the row this lane writes
  // the padding never changes
  *reinterpret_cast<double2*>(&sE[lane][2 * (3 ^ wz)]) = make_double2(0.0, 0.0);
#pragma unroll
  for (int q = 1; q < 4; ++q) *reinterpret_cast<double2*>(&sY1[lane][2 * (q ^ wz)]) = make_double2(0.0, 0.0);
  double d0[2] = {0.0, 0.0}, d1[2] = {0.0, 0.0};
  const int fr = lane >> 2, fk = lane & 3;   // fragment row (A) / column (B), k index inside a step
  // column fr of row 4 j + fk sits at chunk (fr >> 1) ^ swz(4 j + fk), swz(4 j + fk) = 2 * (fk >> 1) + (j & 1)
  const int rq = (fr >> 1) ^ (2 * (fk >> 1)), ro = fr & 1;
  // landmark index and image point of a lane's entry: loaded one trip ahead of the gather that needs them
  int lm = eb + lane < ee ? __ldg(ix.csc_lm + eb + lane) : 0;
  double2 uv = eb + lane < ee ? ix.csc_uv[eb + lane] : make_double2(0.0, 0.0);
  for (int e0 = eb; e0 < ee; e0 += 32) {
    const int e = e0 + lane;
    double E[6], Y[10];
    const int lm_now = lm;
    const double2 uv_now = uv;
    if (e + 32 < ee) {
      lm = __ldg(ix.csc_lm + e + 32);
      uv = ix.csc_uv[e + 32];
    }
    if (e < ee) {
      kron_factors<JOINT, KIND>(e, lm_now, uv_now, cam, X, c1, c2, rb, lm_scale, hll_inv, csc_d, csc_w, E, Y);
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) E[k] = 0.0;
#pragma unroll
      for (int k = 0; k < 10; ++k) Y[k] = 0.0;
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      *reinterpret_cast<double2*>(&sE[lane][2 * (q ^ wz)]) = make_double2(E[2 * q], E[2 * q + 1]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      *reinterpret_cast<double2*>(&sY0[lane][2 * (q ^ wz)]) = make_double2(Y[2 * q], Y[2 * q + 1]);
    }
    *reinterpret_cast<double2*>(&sY1[lane][2 * wz]) = make_double2(Y[8], Y[9]);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = 2 * (rq ^ (j & 1)) + ro;
      const double a = sE[4 * j + fk][col];
      dmma_m8n8k4(d0, a, sY0[4 * j + fk][col]);
      dmma_m8n8k4(d1, a, sY1[4 * j + fk][col]);
    }
    __syncwarp();
  }
  // C fragment: row fr = entry of E, columns 2 fk, 2 fk + 1 of the tile
  if (fr < 6) {
    double* out = item_kron + kKron * static_cast<size_t>(warp) + 10 * fr;
    out[2 * fk] = d0[0];
    out[2 * fk + 1] = d0[1];
    if (fk == 0) {
      out[8] = d1[0];
      out[9] = d1[1];
    }
  }
}

// out[c*width + k] = sum over the items of camera c, in item order
__global__ void __launch_bounds__(kBlock)
k_reduce_items(int C, int width, const int* __restrict__ cam_item_ptr,
               const double* __restrict__ item_vals, double* __restrict__ out,
               const SeriesCtl* __restrict__ ctl) {
  if (ctl != nullptr && ctl->done) return;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(C) * width) return;
  const int c = static_cast<int>(idx / width), k = static_cast<int>(idx % width);
  double sum = 0.0;
  const int ie = cam_item_ptr[c + 1];
  for (int it = cam_item_ptr[c]; it < ie; ++it) sum += item_vals[static_cast<size_t>(it) * width + k];
  out[idx] = sum;
}

__device__ __forceinline__ int e_index(int a, int b) {   // a <= b, 3x3 packed
  return a * 3 - (a * (a - 1)) / 2 + (b - a);
}

// M[(a,j),(b,k)] of the 12x12 matrix sum_i E_i (x) X X^T
__device__ __forceinline__ double kron_entry(const double* __restrict__ kr, int row, int col) {
  int a = row >> 2, j = row & 3, b = col >> 2, k = col & 3;
  if (a > b) {
    const int t = a;
    a = b;
    b = t;
  }
  if (j > k) {
    const int t = j;
    j = k;
    k = t;
  }
  return kr[e_index(a, b) * 10 + sym4_index(j, k)];
}

// pose_scale = 1 / (eps + sqrt(diag(Jp^T Jp)))
__global__ void __launch_bounds__(kBlock)
k_cam_scale(int C, const double* __restrict__ kron, double eps, double* __restrict__ pose_scale) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= C * 12) return;
  const int c = idx / 12, r = idx % 12;
  const double d2 = kron_entry(kron + kKron * static_cast<size_t>(c), r, r);
  pose_scale[idx] = 1.0 / (eps + sqrt(d2));
}

// ------------------------------------------------------------------------------------------
// per camera: B = (s s^T) o Jp^T Jp + lambda I  (step 2: tangent-space projection first),
// B^-1 by Cholesky solves of the identity.  One thread per camera, matrix in local memory.
// ------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ bool chol_inverse(double (&A)[D][D], double (&Inv)[D][D]) {
  // lower Cholesky in place (reads the lower triangle).  Like Eigen's unblocked LLT
  // (external/eigen/Eigen/src/Cholesky/LLT.h) the factorisation STOPS at the first pivot <= 0 and
  // leaves the remaining columns untouched; the reference never checks info(), so the solves below
  // then run on the half-factored triangle (finite garbage, not NaN).  Kept for parity.
  bool ok = true;
  for (int j = 0; j < D && ok; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
    if (!(d > 0.0)) {
      ok = false;
      break;
    }
    const double l = sqrt(d);
    A[j][j] = l;
    const double il = 1.0 / l;
    for (int i = j + 1; i < D; ++i) {
      double v = A[i][j];
      for (int k = 0; k < j; ++k) v -= A[i][k] * A[j][k];
      A[i][j] = v * il;
    }
  }
  // solve L L^T x = e_c for every column
  for (int c = 0; c < D; ++c) {
    double yv[D];
    for (int i = 0; i < D; ++i) {
      double v = (i == c) ? 1.0 : 0.0;
      for (int k = 0; k < i; ++k) v -= A[i][k] * yv[k];
      yv[i] = v / A[i][i];
    }
    for (int i = D - 1; i >= 0; --i) {
      double v = yv[i];
      for (int k = i + 1; k < D; ++k) v -= A[k][i] * Inv[k][c];
      Inv[i][c] = v / A[i][i];
    }
  }
  return ok;
}

// The same computation with sixteen lanes per camera and the block in shared memory: lane i owns row i
// during assembly and factorisation, lane c solves column c of the inverse.  Every entry is produced by
// the same sequence of operations as in the one-thread version below (k_cam_binv, kept for A/B runs
// with POVAR_CAM_BINV=v1), including Eigen's stop-at-the-first-bad-pivot behaviour.
// MODE 0: R = proj((s s^T) o kron) + lambda I -> Bmat, R^-1 -> Binv           (prepare_Hb_*)
// MODE 1: R = Bmat - proj((s s^T) o kron)               , R^-1 -> Binv(=Mprec) (block-Jacobi
//         preconditioner of the reduced camera system, cg/preconditioner.hpp:78-124; kron then holds
//         the diagonal blocks of sum_l Hpl Hll^-1 Hlp)
template <bool JOINT, int MODE>
__global__ void __launch_bounds__(kBlock)
k_cam_binv16(int C, const double* __restrict__ P, const double* __restrict__ kron,
             const double* __restrict__ pose_scale, double lambda, const double* __restrict__ lambda_dev,
             double* __restrict__ Bmat, double* __restrict__ Binv) {
  constexpr int D = JOINT ? 11 : 12;
  if (MODE == 0 && lambda_dev != nullptr) lambda = *lambda_dev;
  constexpr int kCams = kBlock / 16;
  __shared__ double As[kCams][12][13];
  __shared__ double Us[kCams][12];
  const int lane16 = threadIdx.x & 15;
  const int slot = threadIdx.x >> 4;
  const int c_raw = blockIdx.x * kCams + slot;
  const bool live = c_raw < C;
  const int c = live ? c_raw : C - 1;   // idle half-warps shadow the last camera (no stores)
  double (*A)[13] = As[slot];
  const double* kr = kron + kKron * static_cast<size_t>(c);
  const double* s = pose_scale + 12 * static_cast<size_t>(c);
  const int i = lane16;
  if (i < 12) {
    const double si = s[i];
#pragma unroll
    for (int j = 0; j < 12; ++j) A[i][j] = si * s[j] * kron_entry(kr, i, j);
  }
  __syncwarp();
  if (JOINT) {
    // Pi^T A Pi = (H S A S H)[1:,1:]  with S the 0<->p exchange and H = I - tau w w^T
    double pv[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) pv[k] = P[12 * static_cast<size_t>(c) + k];
    Reflector<12> pi;
    pi.make(pv);
    const int p = pi.p;
    if (p != 0 && i < 12) {
      const double t = A[0][i];
      A[0][i] = A[p][i];
      A[p][i] = t;
    }
    __syncwarp();
    if (p != 0 && i < 12) {
      const double t = A[i][0];
      A[i][0] = A[i][p];
      A[i][p] = t;
    }
    __syncwarp();
    double row[12];
    if (i < 12) {
      double v = 0.0;
#pragma unroll
      for (int j = 0; j < 12; ++j) {
        row[j] = A[i][j];
        v += row[j] * pi.w[j];
      }
      Us[slot][i] = v;
    }
    __syncwarp();
    double u[12], alpha = 0.0;
#pragma unroll
    for (int k = 0; k < 12; ++k) u[k] = Us[slot][k];
#pragma unroll
    for (int k = 0; k < 12; ++k) alpha += pi.w[k] * u[k];
    const double tau = pi.tau;
    if (i >= 1 && i < 12) {
      double wi = 0.0, ui = 0.0;
#pragma unroll
      for (int k = 0; k < 12; ++k) {   // static indexing keeps w / u in registers
        wi = (k == i) ? pi.w[k] : wi;
        ui = (k == i) ? u[k] : ui;
      }
#pragma unroll
      for (int j = 1; j < 12; ++j) {
        A[i - 1][j - 1] = row[j] - tau * (wi * u[j] + ui * pi.w[j]) + tau * tau * alpha * wi * pi.w[j];
      }
    }
    __syncwarp();
  }
  double* bm = Bmat + 144 * static_cast<size_t>(c);
  if (i < D) {
    if (MODE == 0) {
      A[i][i] += lambda;
      if (live) {
#pragma unroll
        for (int j = 0; j < D; ++j) bm[i * D + j] = A[i][j];
      }
    } else {
#pragma unroll
      for (int j = 0; j < D; ++j) A[i][j] = bm[i * D + j] - A[i][j];
    }
  }
  __syncwarp();
  // lower Cholesky in place, column by column; rows below the pivot in parallel
  bool ok = true;
  for (int j = 0; j < D; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
    if (!(d > 0.0)) ok = false;
    __syncwarp();
    if (ok) {
      const double l = sqrt(d);
      const double il = 1.0 / l;
      if (i > j && i < D) {
        double v = A[i][j];
        for (int k = 0; k < j; ++k) v -= A[i][k] * A[j][k];
        A[i][j] = v * il;
      }
      if (i == j) A[j][j] = l;
    }
    __syncwarp();
  }
  // lane cc solves L L^T x = e_cc
  if (i < D) {
    const int cc = i;
    double yv[D], x[D];
#pragma unroll
    for (int r = 0; r < D; ++r) {
      double v = (r == cc) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < r; ++k) v -= A[r][k] * yv[k];
      yv[r] = v / A[r][r];
    }
#pragma unroll
    for (int r = D - 1; r >= 0; --r) {
      double v = yv[r];
#pragma unroll
      for (int k = r + 1; k < D; ++k) v -= A[k][r] * x[k];
      x[r] = v / A[r][r];
    }
    if (live) {
      double* bi = Binv + 144 * static_cast<size_t>(c);
#pragma unroll
      for (int r = 0; r < D; ++r) bi[r * D + cc] = x[r];
    }
  }
}

// ------------------------------------------------------------------------------------------
// camera half of b:  raw_c = sum_i (Jp_raw^T W t_i), t_i = r_i - Jl_i H_l.  Output per item; k_reduce_items adds
// the items of a camera.  (The camera half of the E0 products is k_passB_e0_v2, kernels_series.cu.)
// ------------------------------------------------------------------------------------------
template <bool JOINT>
__global__ void __launch_bounds__(kBlock, 2)
k_passB(DeviceIndex ix, const double* __restrict__ P, const double* __restrict__ lm_rec, double c1,
        double c2, Robust rb, double* __restrict__ item_part) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= ix.num_items) return;
  const int c = __ldg(ix.item_cam + warp);
  const int eb = __ldg(ix.item_ptr + warp), ee = __ldg(ix.item_ptr + warp + 1);
  Cam3x4 cam;
  load_cam(P, c, cam);
  double acc[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) acc[k] = 0.0;
  // the landmark index and the image point of the next entry are loaded before the record of this one is used:
  // one memory latency per entry on the critical path instead of two (the kernel waits on the gather)
  int e = eb + lane;
  int lm = e < ee ? __ldg(ix.csc_lm + e) : 0;
  double2 uv = e < ee ? ix.csc_uv[e] : make_double2(0.0, 0.0);
  for (; e < ee; e += 32) {
    double x[4], H[4], m[3];
    load_rec(lm_rec, lm, x, H);
    const double2 uv_now = uv;
    if (e + 32 < ee) {
      lm = __ldg(ix.csc_lm + e + 32);
      uv = ix.csc_uv[e + 32];
    }
    if (JOINT) {
      JointObs ob;
      ob.eval(cam, uv_now.x, uv_now.y, x, rb);
      double j0[4], j1[4], t[2];
      ob.jl_rows(cam, j0, j1);
      const double l0 = dot4(j0, H), l1 = dot4(j1, H);
      const double w = ob.sw * ob.sw;
      t[0] = w * (ob.r[0] - l0);
      t[1] = w * (ob.r[1] - l1);
      ob.jpT_coef(t, m);
    } else {
      PoseObs ob;
      ob.eval(cam, uv_now.x, uv_now.y, x, c1, c2, rb);
      const double w = ob.sw * ob.sw;
      double t[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double l = ob.T[q][0] * H[0] + ob.T[q][1] * H[1] + ob.T[q][2] * H[2];
        t[q] = w * (ob.r[q] - l);
      }
      pose_jpT_coef(t, uv_now.x, uv_now.y, c1, c2, m);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[4 * k + j] += m[k] * x[j];
    }
  }
  warp_allreduce<12>(acc);
  if (lane == 0) {
    double* out = item_part + 12 * static_cast<size_t>(warp);
#pragma unroll
    for (int k = 0; k < 12; ++k) out[k] = acc[k];
  }
}

// ------------------------------------------------------------------------------------------
// per-camera vector plumbing.  D = 12 (step 1) or 11 (step 2, tangent space of vec(P)).
// ------------------------------------------------------------------------------------------
// e (D) from the raw 12-vector of the camera pass:  s o raw   or   Pi^T (s o raw)
template <bool JOINT>
__device__ __forceinline__ void raw_to_reduced(const double* __restrict__ raw,
                                               const double* __restrict__ s,
                                               const double* __restrict__ Pc, double* e) {
  double v[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) v[i] = s[i] * raw[i];
  if (JOINT) {
    double pv[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) pv[i] = Pc[i];
    Reflector<12> pi;
    pi.make(pv);
    pi.apply_t(v, e);
  } else {
#pragma unroll
    for (int i = 0; i < 12; ++i) e[i] = v[i];
  }
}

// y (12) gathered by the passes:  s o x   or   s o (Pi x)
// y values only (12): s o x  or  s o (Pi x)
template <bool JOINT>
__device__ __forceinline__ void reduced_to_y_values(const double* x, const double* __restrict__ s,
                                                    const double* __restrict__ Pc, double (&yv)[12]) {
  if (JOINT) {
    double pv[12], full[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) pv[i] = Pc[i];
    Reflector<12> pi;
    pi.make(pv);
    pi.apply(x, full);
#pragma unroll
    for (int i = 0; i < 12; ++i) yv[i] = s[i] * full[i];
  } else {
#pragma unroll
    for (int i = 0; i < 12; ++i) yv[i] = s[i] * x[i];
  }
}

// `rec` is the camera's record of the landmark-major E0 pass (CamRec<JOINT>): y is stored there too
template <bool JOINT>
__device__ __forceinline__ void reduced_to_y(const double* x, const double* __restrict__ s,
                                             const double* __restrict__ Pc, double* __restrict__ y,
                                             double* __restrict__ rec) {
  double yv[12];
  if (JOINT) {
    double pv[12], full[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) pv[i] = Pc[i];
    Reflector<12> pi;
    pi.make(pv);
    pi.apply(x, full);
#pragma unroll
    for (int i = 0; i < 12; ++i) yv[i] = s[i] * full[i];
  } else {
#pragma unroll
    for (int i = 0; i < 12; ++i) yv[i] = s[i] * x[i];
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) y[i] = yv[i];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int j = 0; j < 4; ++j) rec[CamRec::y_index(k, j)] = yv[4 * k + j];
  }
}

// b = reduced(raw);  accum = tmp = B^-1 (-b);  y = y(tmp)     (solve_*: "accum = right_mul_b_inv(-b_p)")
template <bool JOINT>
__global__ void __launch_bounds__(128)
k_finish_b(int C, const double* __restrict__ raw, const double* __restrict__ pose_scale,
           const double* __restrict__ P, const double* __restrict__ Binv, double* __restrict__ b,
           double* __restrict__ tmp, double* __restrict__ acc, double* __restrict__ y,
           double* __restrict__ cam_rec, double* __restrict__ norm_part) {
  constexpr int D = JOINT ? 11 : 12;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double* s = pose_scale + 12 * static_cast<size_t>(c);
  const double* Pc = P + 12 * static_cast<size_t>(c);
  double e[12];
  raw_to_reduced<JOINT>(raw + 12 * static_cast<size_t>(c), s, Pc, e);
  const double* bi = Binv + 144 * static_cast<size_t>(c);
  double x0[12];
  double n2 = 0.0;
  for (int i = 0; i < D; ++i) {
    b[static_cast<size_t>(c) * D + i] = e[i];
    double v = 0.0;
    for (int j = 0; j < D; ++j) v += bi[i * D + j] * (-e[j]);
    x0[i] = v;
    n2 += v * v;
    tmp[static_cast<size_t>(c) * D + i] = v;
    acc[static_cast<size_t>(c) * D + i] = v;
  }
  reduced_to_y<JOINT>(x0, s, Pc, y + 12 * static_cast<size_t>(c),
                      cam_rec + CamRec::stride(JOINT) * static_cast<size_t>(c));
  norm_part[2 * c] = n2;
  norm_part[2 * c + 1] = n2;
}

// one power-series term, camera side:  tmp = B^-1 reduced(raw);  accum += tmp;  y = y(tmp)
template <bool JOINT>
__global__ void __launch_bounds__(128)
k_term(int C, const double* __restrict__ raw, const double* __restrict__ pose_scale,
       const double* __restrict__ P, const double* __restrict__ Binv, double* __restrict__ tmp,
       double* __restrict__ acc, double* __restrict__ y, double* __restrict__ cam_rec,
       double* __restrict__ norm_part, const SeriesCtl* __restrict__ ctl) {
  if (ctl->done) return;
  constexpr int D = JOINT ? 11 : 12;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double* s = pose_scale + 12 * static_cast<size_t>(c);
  const double* Pc = P + 12 * static_cast<size_t>(c);
  double e[12];
  raw_to_reduced<JOINT>(raw + 12 * static_cast<size_t>(c), s, Pc, e);
  const double* bi = Binv + 144 * static_cast<size_t>(c);
  double t[12];
  double nt = 0.0, na = 0.0;
  for (int i = 0; i < D; ++i) {
    double v = 0.0;
    for (int j = 0; j < D; ++j) v += bi[i * D + j] * e[j];
    t[i] = v;
    nt += v * v;
    const double a = acc[static_cast<size_t>(c) * D + i] + v;
    acc[static_cast<size_t>(c) * D + i] = a;
    na += a * a;
    tmp[static_cast<size_t>(c) * D + i] = v;
  }
  reduced_to_y<JOINT>(t, s, Pc, y + 12 * static_cast<size_t>(c),
                      cam_rec + CamRec::stride(JOINT) * static_cast<size_t>(c));
  norm_part[2 * c] = nt;
  norm_part[2 * c + 1] = na;
}

// ordered sum of the per-camera partial norms; single block
__device__ __forceinline__ void sum_norm_parts(int C, const double* __restrict__ norm_part,
                                               double* smem, double& s0, double& s1) {
  double acc[2] = {0.0, 0.0};
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    acc[0] += __ldcg(norm_part + 2 * c);       // written by other blocks of the same launch (k_term16)
    acc[1] += __ldcg(norm_part + 2 * c + 1);
  }
  block_reduce<2>(acc, smem);
  s0 = acc[0];
  s1 = acc[1];
}

// convergence test after term i (linearization_power_varproj.hpp:205-229), one thread
__device__ __forceinline__ void series_decide(double s0, double s1, int term, double eta,
                                              double r_tolerance, SeriesCtl* ctl) {
  const double it_norm = sqrt(s0), acc_norm = sqrt(s1);
  ctl->last_tmp_norm = it_norm;
  ctl->last_acc_norm = acc_norm;
  ctl->nonfinite = isfinite(s1) ? 0 : 1;
  bool stop = false;
  if (eta > 0) {
    const double zeta = term * it_norm / acc_norm;
    if (zeta < eta) stop = true;
  }
  if (!stop && r_tolerance > 0 && it_norm / ctl->norm0 < r_tolerance) stop = true;
  if (stop) {
    ctl->done = 1;
    ctl->iterations = term;
  }
}

// Peer exchange, low-latency protocol: a double travels as ONE 16-byte store of two 8-byte words
// {lo | number << 32, hi | number << 32}; the receiver polls the slot until both words carry the number of the
// exchange it waits for.  PTX guarantees single-copy atomicity per ELEMENT of a vector access, so each
// {value half, tag} pair is one 64-bit element: a reader sees a half either with its own tag or not at all,
// and a slot whose two tags match holds one value.  No fence, no separate flag: the latency of an exchange is
// one NVLink store.
__device__ __forceinline__ void st_tagged(double* slot, double v, unsigned int epoch) {
  const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(v));
  const unsigned long long tag = static_cast<unsigned long long>(epoch) << 32;
  const unsigned long long a = (bits & 0xffffffffULL) | tag, b = (bits >> 32) | tag;
  asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(slot), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ bool ld_tagged(const double* slot, unsigned int epoch, double& v) {
  unsigned long long a, b;
  asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(slot) : "memory");
  v = __longlong_as_double(static_cast<long long>((b << 32) | (a & 0xffffffffULL)));
  return static_cast<unsigned int>(a >> 32) == epoch && static_cast<unsigned int>(b >> 32) == epoch;
}
// number of the exchange a kernel is about to perform: one more than the buffer has seen (written by the last
// block of the previous exchanging kernel on this stream)
__device__ __forceinline__ unsigned int next_exchange_number(const PeerExchange& px) {
  return *reinterpret_cast<volatile const unsigned int*>(px.count) + 1u;
}
__device__ __forceinline__ long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return static_cast<long long>(t);
}
constexpr long long kPeerSpinNs = 4000000000LL;   // give up after 4 s: a peer died; fail the solve

// one power-series term, camera side, sixteen lanes per camera (lane i owns row i of B^-1 -- the
// 144 loads of the block are the expensive part -- and everything else is recomputed per lane in the
// order of k_term, so the two kernels give identical bits):
//   [kTermFused, kTermPeer] raw = sum of the camera's item partials (k_reduce_items);
//   [kTermPeer] the all-reduce over the landmark shards, fused: every lane stores its camera sum, tagged
//       with the exchange number, into every rank's receive buffer (NVLink peer stores), then polls its
//       own buffer for the peers' values and adds them in rank order -- every rank gets the same bits,
//       no NCCL launch, no separate reduction kernel, no fence;
//   tmp = B^-1 reduced(raw);  accum += tmp;  y = y(tmp);  per-camera norms;  then the LAST block to
//   finish applies the convergence test (series_decide).  Block = 256 threads = 16 cameras.
template <bool JOINT, int MODE>
__global__ void __launch_bounds__(kBlock)
k_term16(int C, const double* __restrict__ raw_in, const int* __restrict__ cam_item_ptr,
         const double* __restrict__ item_part, const double* __restrict__ pose_scale,
         const double* __restrict__ P, const double* __restrict__ Binv, double* __restrict__ tmp,
         double* __restrict__ acc, double* __restrict__ y, double* __restrict__ cam_rec,
         double* __restrict__ norm_part, int term, double eta, double r_tolerance, SeriesCtl* ctl,
         PeerExchange px, SeriesLoop loop) {
  if (ctl->done) return;
  if (term <= 0) term = ctl->term + 1;   // inside the loop of the series graph (the last block advances the count)
  constexpr int D = JOINT ? 11 : 12;
  __shared__ double smem[2 * (kBlock / 32)];
  __shared__ int is_last;
  const int lane16 = threadIdx.x & 15;
  const int base = (threadIdx.x & 31) & ~15;   // first lane of this half-warp
  // Peer mode: a block waits for the sums its cameras get from the other ranks, i.e. for the peers'
  // block with the same number.  Numbers are handed out in dispatch order (a counter, as in a
  // decoupled look-back scan), so on every rank the lowest-numbered unfinished block is running and
  // has already sent: the exchange makes progress even when the grid is larger than one wave.
  unsigned int bid = blockIdx.x;
  unsigned int epoch = 0;
  if (MODE == kTermPeer) {
    epoch = next_exchange_number(px);   // before this block's ticket: the last block advances the count
    __shared__ unsigned int s_bid;
    if (threadIdx.x == 0) s_bid = atomicAdd(&ctl->next_block, 1u);
    __syncthreads();
    bid = s_bid;
  }
  const int c_raw = static_cast<int>((bid * blockDim.x + threadIdx.x) >> 4);
  const bool live = c_raw < C;
  const int c = live ? c_raw : C - 1;          // idle half-warps shadow the last camera (no stores)
  // Everything that does not depend on the camera sums is requested first: these loads are in flight
  // while the item partials are added and (sharded) while the peers' sums travel.
  const double* s = pose_scale + 12 * static_cast<size_t>(c);
  const double* Pc = P + 12 * static_cast<size_t>(c);
  double sreg[12], preg[12], brow[12], aold[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    sreg[k] = s[k];
    preg[k] = JOINT ? Pc[k] : 0.0;
  }
  {
    const double* bi = Binv + 144 * static_cast<size_t>(c) + (lane16 < D ? lane16 : 0) * D;
#pragma unroll
    for (int j = 0; j < D; ++j) brow[j] = bi[j];
#pragma unroll
    for (int i = 0; i < D; ++i) aold[i] = acc[static_cast<size_t>(c) * D + i];
  }
  double raw[12];
  if (MODE != kTermRaw) {
    double mine = 0.0;
    if (lane16 < 12) {
      const int ie = cam_item_ptr[c + 1];
      for (int it = cam_item_ptr[c]; it < ie; ++it) mine += item_part[static_cast<size_t>(it) * 12 + lane16];
    }
    if (MODE == kTermPeer) {
      // slots are 16 bytes (2 doubles wide): [parity][source rank][stride], the first 12*C of a rank used here
      const int par = static_cast<int>(epoch & 1u);
      const size_t vec = static_cast<size_t>(px.stride);
      const size_t mine_at = 2 * ((static_cast<size_t>(par) * px.world + px.rank) * vec + 12 * static_cast<size_t>(c) + lane16);
      if (live && lane16 < 12) {
#pragma unroll
        for (int r = 0; r < kMaxPeers; ++r) {
          if (r < px.world) st_tagged(px.recv[r] + mine_at, mine, epoch);
        }
      }
      // collect the ranks' sums (all polls of a round are in flight together), then add them in rank
      // order: the same bits on every rank
      double sum = 0.0;
      if (live && lane16 < 12) {
        const double* rb = px.recv[px.rank] + 2 * (static_cast<size_t>(par) * px.world * vec + 12 * static_cast<size_t>(c) + lane16);
        double v[kMaxPeers];
        unsigned int pending = (1u << px.world) - 1u;
        long long t0 = 0;
        unsigned int spins = 0;
#pragma unroll
        for (int r = 0; r < kMaxPeers; ++r) v[r] = 0.0;
        while (pending != 0u) {
#pragma unroll
          for (int r = 0; r < kMaxPeers; ++r) {
            if ((pending >> r) & 1u) {
              double got;
              if (ld_tagged(rb + 2 * r * vec, epoch, got)) {
                v[r] = got;
                pending &= ~(1u << r);
              }
            }
          }
          if ((++spins & 1023u) == 0) {
            const long long now = global_ns();
            if (t0 == 0) t0 = now;
            if (now - t0 > kPeerSpinNs) {
              atomicExch(&ctl->peer_timeout, 1);
              break;
            }
          }
        }
#pragma unroll
        for (int r = 0; r < kMaxPeers; ++r) {
          if (r < px.world) sum += v[r];
        }
      }
      __syncwarp();
      mine = sum;
    }
#pragma unroll
    for (int k = 0; k < 12; ++k) raw[k] = __shfl_sync(kFullMask, mine, base + k);
  } else {
#pragma unroll
    for (int k = 0; k < 12; ++k) raw[k] = raw_in[12 * static_cast<size_t>(c) + k];
  }
  double e[12];
  raw_to_reduced<JOINT>(raw, sreg, preg, e);
  double ti = 0.0;
  if (lane16 < D) {
#pragma unroll
    for (int j = 0; j < D; ++j) ti += brow[j] * e[j];
  }
  double t[12];
  double nt = 0.0, na = 0.0;
#pragma unroll
  for (int i = 0; i < 12; ++i) t[i] = __shfl_sync(kFullMask, ti, base + i);
#pragma unroll
  for (int i = 0; i < D; ++i) {
    nt += t[i] * t[i];
    const double a = aold[i] + t[i];
    na += a * a;
  }
  __syncwarp();   // every lane has read accum before lane i overwrites entry i
  if (live && lane16 < D) {
    double mine_old = 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) mine_old = (i == lane16) ? aold[i] : mine_old;
    acc[static_cast<size_t>(c) * D + lane16] = mine_old + ti;
    tmp[static_cast<size_t>(c) * D + lane16] = ti;
  }
  double yv[12];
  reduced_to_y_values<JOINT>(t, sreg, preg, yv);
  if (live && lane16 < 12) {
    double mine = 0.0;
#pragma unroll
    for (int i = 0; i < 12; ++i) mine = (i == lane16) ? yv[i] : mine;
    y[12 * static_cast<size_t>(c) + lane16] = mine;
    cam_rec[CamRec::stride(JOINT) * static_cast<size_t>(c) + CamRec::y_index(lane16 >> 2, lane16 & 3)] = mine;
  }
  if (live && lane16 == 0) {
    norm_part[2 * c] = nt;
    norm_part[2 * c + 1] = na;
  }
  // last block to arrive applies the convergence test (linearization_power_varproj.hpp:205-229)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(&ctl->ticket, 1u);
    is_last = (prev == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double s0, s1;
  sum_norm_parts(C, norm_part, smem, s0, s1);
  if (threadIdx.x == 0) {
    ctl->ticket = 0;
    ctl->next_block = 0;
    ctl->term = term;
    if (MODE == kTermPeer) *px.count = epoch;   // this exchange happened (skipped terms never get here)
    series_decide(s0, s1, term, eta, r_tolerance, ctl);
    if (loop.active) {
      cudaGraphSetConditional(static_cast<cudaGraphConditionalHandle>(loop.handle),
                              (ctl->done || term >= loop.max_terms) ? 0u : 1u);
    }
  }
}

__global__ void __launch_bounds__(kBlock)
k_series_start(int C, const double* __restrict__ norm_part, double r_tolerance, int max_terms,
               SeriesCtl* ctl, SeriesLoop loop) {
  __shared__ double smem[2 * (kBlock / 32)];
  double s0, s1;
  sum_norm_parts(C, norm_part, smem, s0, s1);
  if (threadIdx.x == 0) {
    ctl->done = max_terms > 0 ? 0 : 1;
    ctl->iterations = max_terms > 0 ? max_terms : 0;   // "Maximum number of iterations reached."
    ctl->nonfinite = isfinite(s1) ? 0 : 1;
    ctl->norm0 = r_tolerance > 0 ? sqrt(s0) : 0.0;
    ctl->last_tmp_norm = sqrt(s0);
    ctl->last_acc_norm = sqrt(s1);
    ctl->term = 0;
    if (loop.active) {
      cudaGraphSetConditional(static_cast<cudaGraphConditionalHandle>(loop.handle), max_terms > 0 ? 1u : 0u);
    }
  }
}

// out = reduced(raw)   (E0 x for callers outside the series: tests, PCG)
template <bool JOINT>
__global__ void __launch_bounds__(128)
k_e0_finish(int C, const double* __restrict__ raw, const double* __restrict__ pose_scale,
            const double* __restrict__ P, double* __restrict__ out) {
  constexpr int D = JOINT ? 11 : 12;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double e[12];
  raw_to_reduced<JOINT>(raw + 12 * static_cast<size_t>(c), pose_scale + 12 * static_cast<size_t>(c),
                        P + 12 * static_cast<size_t>(c), e);
  for (int i = 0; i < D; ++i) out[static_cast<size_t>(c) * D + i] = e[i];
}

template <bool JOINT>
__global__ void __launch_bounds__(128)
k_make_y(int C, const double* __restrict__ x, const double* __restrict__ pose_scale,
         const double* __restrict__ P, double* __restrict__ y, double* __restrict__ cam_rec) {
  constexpr int D = JOINT ? 11 : 12;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double xv[12];
  for (int i = 0; i < D; ++i) xv[i] = x[static_cast<size_t>(c) * D + i];
  reduced_to_y<JOINT>(xv, pose_scale + 12 * static_cast<size_t>(c), P + 12 * static_cast<size_t>(c),
                      y + 12 * static_cast<size_t>(c),
                      cam_rec + CamRec::stride(JOINT) * static_cast<size_t>(c));
}

// P += reshape(v)   (Camera::inc_pose_pOSE / inc_pose_projective_space, bal_problem.hpp:132-163)
__global__ void __launch_bounds__(kBlock)
k_cam_add(int n, const double* __restrict__ v, const double* __restrict__ scale, double* __restrict__ P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  P[i] += scale != nullptr ? v[i] * scale[i] : v[i];
}

// P <- P / |P|_F   (space_matrix.normalize(), bal_bundle_adjustment.cpp:550-552, 700-702)
__global__ void __launch_bounds__(128)
k_normalize_cams(int C, double* __restrict__ P) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double* p = P + 12 * static_cast<size_t>(c);
  double n2 = 0.0;
  for (int i = 0; i < 12; ++i) n2 += p[i] * p[i];
  const double n = sqrt(n2);
  for (int i = 0; i < 12; ++i) p[i] = p[i] / n;
}

// out_c = blocks_c * x_c  (D x D blocks with leading dimension D, stored 144 apart)
__global__ void __launch_bounds__(128)
k_block_matvec(int C, int D, const double* __restrict__ blocks, const double* __restrict__ x,
               double* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double* bm = blocks + 144 * static_cast<size_t>(c);
  for (int i = 0; i < D; ++i) {
    double v = 0.0;
    for (int j = 0; j < D; ++j) v += bm[i * D + j] * x[static_cast<size_t>(c) * D + j];
    out[static_cast<size_t>(c) * D + i] = v;
  }
}

}  // namespace

void launch_kron(const DeviceState& d, const ModelParams& mp, bool joint, KronKind kind,
                 const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  const int blocks = (d.ix.num_items + kKronWarps - 1) / kKronWarps;
  const int threads = 32 * kKronWarps;
  if (blocks == 0) return;
  double* cw = (!joint && kind == KRON_HPP && mp.robust_norm == NORM_HUBER) ? d.csc_w : nullptr;
  double* cd = (joint && kind == KRON_HPP) ? d.csc_d : nullptr;
#define POVAR_KRON_LAUNCH(K, J, KIND)                                                                     \
  K<J, KIND><<<blocks, threads, 0, lc.stream>>>(d.ix, d.P, d.X, mp.c1, mp.c2, rb, d.lm_scale, d.hll_inv, \
                                                d.item_kron, cd, cw)
  if (kind == KRON_HPP) {
    if (joint) POVAR_KRON_LAUNCH(k_kron_mma, true, KRON_HPP);
    else POVAR_KRON_LAUNCH(k_kron_mma, false, KRON_HPP);
  } else {
    if (joint) POVAR_KRON_LAUNCH(k_kron_mma, true, KRON_SDIAG);
    else POVAR_KRON_LAUNCH(k_kron_mma, false, KRON_SDIAG);
  }
#undef POVAR_KRON_LAUNCH
  count(lc);
}

void launch_reduce_items(const DeviceState& d, const double* item_vals, int width, double* out,
                         bool in_series, const LaunchCfg& lc) {
  const long long n = static_cast<long long>(d.ix.C) * width;
  const int blocks = static_cast<int>((n + kBlock - 1) / kBlock);
  k_reduce_items<<<blocks, kBlock, 0, lc.stream>>>(d.ix.C, width, d.ix.cam_item_ptr, item_vals, out,
                                                   in_series ? d.ctl : nullptr);
  count(lc);
}

void launch_cam_scale(const DeviceState& d, const ModelParams& mp, const LaunchCfg& lc) {
  const int blocks = (d.ix.C * 12 + kBlock - 1) / kBlock;
  k_cam_scale<<<blocks, kBlock, 0, lc.stream>>>(d.ix.C, d.kron, mp.jacobi_eps, d.pose_scale);
  count(lc);
}

void launch_cam_binv(const DeviceState& d, bool joint, double lambda, const LaunchCfg& lc, const double* lambda_dev) {
  const int blocks16 = (d.ix.C + kBlock / 16 - 1) / (kBlock / 16);
  if (joint) {
    k_cam_binv16<true, 0><<<blocks16, kBlock, 0, lc.stream>>>(d.ix.C, d.P, d.kron, d.pose_scale, lambda, lambda_dev, d.Bmat, d.Binv);
  } else {
    k_cam_binv16<false, 0><<<blocks16, kBlock, 0, lc.stream>>>(d.ix.C, d.P, d.kron, d.pose_scale, lambda, lambda_dev, d.Bmat, d.Binv);
  }
  count(lc);
}

void launch_cam_precond(const DeviceState& d, bool joint, const double* kron_sdiag, const LaunchCfg& lc) {
  const int blocks16 = (d.ix.C + kBlock / 16 - 1) / (kBlock / 16);
  if (joint) {
    k_cam_binv16<true, 1><<<blocks16, kBlock, 0, lc.stream>>>(d.ix.C, d.P, kron_sdiag, d.pose_scale, 0.0, nullptr, d.Bmat, d.Mprec);
  } else {
    k_cam_binv16<false, 1><<<blocks16, kBlock, 0, lc.stream>>>(d.ix.C, d.P, kron_sdiag, d.pose_scale, 0.0, nullptr, d.Bmat, d.Mprec);
  }
  count(lc);
}

// b: the camera-major pass with r_i - Jl_i H_l per observation (prepare_Hb_*); the E0 products use
// k_passB_e0_v2 (kernels_series.cu)
void launch_passB(const DeviceState& d, const ModelParams& mp, bool joint, const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  const int blocks = item_grid(d);
  if (joint) {
    k_passB<true><<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.lm_rec, mp.c1, mp.c2, rb, d.item_part);
  } else {
    k_passB<false><<<blocks, kBlock, 0, lc.stream>>>(d.ix, d.P, d.lm_rec, mp.c1, mp.c2, rb, d.item_part);
  }
  count(lc);
}

void launch_finish_b(const DeviceState& d, bool joint, const LaunchCfg& lc) {
  const int blocks = (d.ix.C + 127) / 128;
  if (joint) {
    k_finish_b<true><<<blocks, 128, 0, lc.stream>>>(d.ix.C, d.cam_raw, d.pose_scale, d.P, d.Binv, d.b,
                                                    d.vec_tmp, d.vec_acc, d.vec_y, d.cam_rec, d.norm_part);
  } else {
    k_finish_b<false><<<blocks, 128, 0, lc.stream>>>(d.ix.C, d.cam_raw, d.pose_scale, d.P, d.Binv, d.b,
                                                     d.vec_tmp, d.vec_acc, d.vec_y, d.cam_rec, d.norm_part);
  }
  count(lc);
}

void launch_series_start(const DeviceState& d, double r_tolerance, int max_terms, const LaunchCfg& lc,
                         const SeriesLoop& loop) {
  k_series_start<<<1, kBlock, 0, lc.stream>>>(d.ix.C, d.norm_part, r_tolerance, max_terms, d.ctl, loop);
  count(lc);
}

// The same exchange for any vector of up to px.stride doubles (cost scalars, l_diff, flags, b, the Kronecker
// sums): element i is pushed to every rank and collected from every rank by one thread; a thread only waits
// for the thread with the same index on the other ranks, which pushes before it polls, so the one-wave
// grid-stride launch cannot deadlock.
__global__ void __launch_bounds__(kBlock)
k_peer_allreduce(double* __restrict__ buf, size_t n, PeerExchange px, SeriesCtl* ctl, int skip_when_done) {
  if (skip_when_done && ctl->done) return;   // every rank holds the same flag: nobody exchanges
  const unsigned int epoch = next_exchange_number(px);
  const int par = static_cast<int>(epoch & 1u);
  const size_t stride = static_cast<size_t>(px.stride);
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const double mine = buf[i];
    const size_t at = 2 * ((static_cast<size_t>(par) * px.world + px.rank) * stride + i);
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) {
      if (r < px.world) st_tagged(px.recv[r] + at, mine, epoch);
    }
    const double* rb = px.recv[px.rank] + 2 * (static_cast<size_t>(par) * px.world * stride + i);
    double v[kMaxPeers];
    unsigned int pending = (1u << px.world) - 1u;
    long long t0 = 0;
    unsigned int spins = 0;
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) v[r] = 0.0;
    while (pending != 0u) {
#pragma unroll
      for (int r = 0; r < kMaxPeers; ++r) {
        if ((pending >> r) & 1u) {
          double got;
          if (ld_tagged(rb + 2 * r * stride, epoch, got)) {
            v[r] = got;
            pending &= ~(1u << r);
          }
        }
      }
      if ((++spins & 1023u) == 0) {
        const long long now = global_ns();
        if (t0 == 0) t0 = now;
        if (now - t0 > kPeerSpinNs) {
          atomicExch(&ctl->peer_timeout, 1);
          break;
        }
      }
    }
    double sum = 0.0;
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) {
      if (r < px.world) sum += v[r];
    }
    // a peer that never answered: poison the result so that the caller's finiteness checks trip
    buf[i] = pending != 0u ? __longlong_as_double(0x7ff8000000000000LL) : sum;
  }
  // the last block to finish advances the exchange count (every block has read it by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int prev = atomicAdd(px.count + 1, 1u);
    if (prev == gridDim.x - 1) {
      px.count[1] = 0;
      px.count[0] = epoch;
    }
  }
}

void launch_peer_allreduce(const DeviceState& d, double* buf, size_t n, const PeerExchange& px,
                           const LaunchCfg& lc, bool skip_when_done) {
  if (n == 0) return;
  size_t blocks = (n + kBlock - 1) / kBlock;
  if (blocks > static_cast<size_t>(sm_count()) * 2) blocks = static_cast<size_t>(sm_count()) * 2;   // one wave, always resident
  k_peer_allreduce<<<static_cast<int>(blocks), kBlock, 0, lc.stream>>>(buf, n, px, d.ctl, skip_when_done ? 1 : 0);
  count(lc);
}

void launch_series_term(const DeviceState& d, bool joint, int term, double eta, double r_tolerance,
                        TermMode mode, const PeerExchange* px, const LaunchCfg& lc, const SeriesLoop& loop) {
  const int blocks = (d.ix.C + 15) / 16;
  const PeerExchange none{};
  const PeerExchange& pe = (mode == kTermPeer && px != nullptr) ? *px : none;
#define POVAR_TERM(J, M)                                                                              \
  k_term16<J, M><<<blocks, kBlock, 0, lc.stream>>>(d.ix.C, d.cam_raw, d.ix.cam_item_ptr, d.item_part,  \
                                                   d.pose_scale, d.P, d.Binv, d.vec_tmp, d.vec_acc,    \
                                                   d.vec_y, d.cam_rec, d.norm_part, term, eta,         \
                                                   r_tolerance, d.ctl, pe, loop)
  if (joint) {
    if (mode == kTermPeer) POVAR_TERM(true, kTermPeer);
    else if (mode == kTermFused) POVAR_TERM(true, kTermFused);
    else POVAR_TERM(true, kTermRaw);
  } else {
    if (mode == kTermPeer) POVAR_TERM(false, kTermPeer);
    else if (mode == kTermFused) POVAR_TERM(false, kTermFused);
    else POVAR_TERM(false, kTermRaw);
  }
#undef POVAR_TERM
  count(lc);
}

void launch_e0_finish(const DeviceState& d, bool joint, double* out, const LaunchCfg& lc) {
  const int blocks = (d.ix.C + 127) / 128;
  if (joint) {
    k_e0_finish<true><<<blocks, 128, 0, lc.stream>>>(d.ix.C, d.cam_raw, d.pose_scale, d.P, out);
  } else {
    k_e0_finish<false><<<blocks, 128, 0, lc.stream>>>(d.ix.C, d.cam_raw, d.pose_scale, d.P, out);
  }
  count(lc);
}

void launch_make_y(const DeviceState& d, bool joint, const double* x, double* y, const LaunchCfg& lc) {
  const int blocks = (d.ix.C + 127) / 128;
  if (joint) {
    k_make_y<true><<<blocks, 128, 0, lc.stream>>>(d.ix.C, x, d.pose_scale, d.P, y, d.cam_rec);
  } else {
    k_make_y<false><<<blocks, 128, 0, lc.stream>>>(d.ix.C, x, d.pose_scale, d.P, y, d.cam_rec);
  }
  count(lc);
}

void launch_cam_update_pose(const DeviceState& d, const double* inc, const LaunchCfg& lc) {
  const int n = d.ix.C * 12;
  k_cam_add<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(n, inc, d.pose_scale, d.P);
  count(lc);
}

void launch_cam_update_joint(const DeviceState& d, const double* y, const LaunchCfg& lc) {
  const int n = d.ix.C * 12;
  k_cam_add<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(n, y, nullptr, d.P);
  count(lc);
}

void launch_normalize_cams(const DeviceState& d, const LaunchCfg& lc) {
  k_normalize_cams<<<(d.ix.C + 127) / 128, 128, 0, lc.stream>>>(d.ix.C, d.P);
  count(lc);
}

void launch_block_matvec(const DeviceState& d, int dim, const double* blocks, const double* x,
                         double* out, const LaunchCfg& lc) {
  k_block_matvec<<<(d.ix.C + 127) / 128, 128, 0, lc.stream>>>(d.ix.C, dim, blocks, x, out);
  count(lc);
}

}  // namespace povar
