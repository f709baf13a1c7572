// CHOLESKY, step 1: the explicit reduced camera system and its direct solve, hand-written.
//
// Replaces get_Hb_pOSE / add_Hb_pOSE (/root/reference/src/rootba_povar/sc/linearization_sc.hpp:419-438,
// sc/landmark_block.hpp:360-412: scatter-adds of pairwise 12x12 blocks into a hash map under C^2 mutexes) and
// solve_direct_pOSE (sc/linearization_sc.hpp:236-245: Eigen::SimplicialLLT).  The solution of S x = -b is
// unique, so neither the ordering nor the blocking of the factorisation changes the result beyond rounding.
//
//   assembly   S = blockdiag(B) - sum_l Hpl Hll^-1 Hlp, lower block triangle, WITHOUT atomics: one thread block
//              per block row (camera i) walks the camera's observations in landmark order; warp w owns the
//              block columns j = w (mod warps), so every 12x12 block is updated by exactly one warp in a fixed
//              order -- two runs give the same bits (the reference's own order depends on its thread count).
//   factorise  right-looking blocked LL^T on 64x64 tiles: the diagonal tile is factorised and its factor inverted
//              inside one thread block (shared memory); the panel below it is multiplied by that inverse and the
//              trailing matrix updated by one FP64 tensor-core tile kernel (mma.sync.m8n8k4.f64, DMMA in SASS):
//              C -= A B^T on 64x64x64 tiles staged in shared memory.  The only dense factorisation of the path
//              that profiles as a contraction (DESIGN.md 4).
//   solve      forward / backward substitution tile row by tile row with the stored inverses of the diagonal
//              factors.
// Two storages of S and its factor, one set of kernels: the kernels take an addressing policy.
//   dense        the whole matrix, row-major, leading dimension n_pad = 12 C rounded up to 64 (identity on the
//                padding), cameras in their own order;
//   tile-sparse  only the 64x64 tiles of the factor that can be non-zero (CholPattern, host/chol_symbolic.cpp),
//                each stored contiguously (ld = 64) in slot order, cameras in the fill-reducing order perm; the
//                panel and the update walk the stored tiles of a column, the backward substitution those of a row.
// The dense instantiations compute what they computed before the policies existed, bit for bit.
#include <cuda_runtime.h>

#include <cassert>

#include "device_math.cuh"
#include "povar_internal.h"

namespace povar {

namespace {

constexpr int kNB = 64;        // tile edge
constexpr int kKC = 32;        // k-chunk of a tile product staged in shared memory
constexpr int kPad = 4;        // row padding of the staged chunks (doubles): conflict-free fragment loads

inline void count(const LaunchCfg& lc, int n = 1) {
  if (lc.launch_counter) *lc.launch_counter += n;
}

__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
}

// ---- assembly ------------------------------------------------------------------------------------
// Wk = w Z^T K (3x3): Z = Jl_raw o lm_scale, K the 4x3 coefficient matrix of Jp_raw (Jp_raw = K (x) Xt^T)
__device__ __forceinline__ void pose_wk(const Cam3x4& cam, double u, double v, const double (&x)[4],
                                        const double (&sl)[4], double c1, double c2, const Robust& rb,
                                        double (&Wk)[3][3]) {
  PoseObs ob;
  ob.eval(cam, u, v, x, c1, c2, rb);
  const double w = ob.sw * ob.sw;
  const double K[4][3] = {{c1, 0.0, -c1 * u}, {0.0, c1, -c1 * v}, {c2, 0.0, 0.0}, {0.0, c2, 0.0}};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      Wk[a][k] = w * sl[a] * (ob.T[0][a] * K[0][k] + ob.T[1][a] * K[1][k] + ob.T[2][a] * K[2][k] +
                              ob.T[3][a] * K[3][k]);
    }
  }
}

constexpr int kRowWarps = 8;

// ---- addressing policies --------------------------------------------------------------------------
// element (R, C) and element (r, cc) of the 12x12 block (ci, cj), cj <= ci in camera order, of S; stores(..): whether
// the assembly writes that element of the block at all
struct DenseS {
  double* S;
  long long ld;
  __device__ bool stores(int, int, int, int) const { return true; }
  __device__ double* elem(long long R, long long C) const { return S + R * ld + C; }
  __device__ double* block(int ci, int cj, int r, int cc) const {
    return S + (static_cast<long long>(ci) * 12 + r) * ld + (static_cast<long long>(cj) * 12 + cc);
  }
};
// rows of camera c at 12 perm[c] ..; a block that lands in the upper triangle of that order is stored transposed.
// Only the lower triangle of a diagonal block is written: rows 12 p .. 12 p + 11 of a camera can straddle two tiles,
// and the upper part of its block would then fall into tile (I, I + 1), which is not stored.
struct TiledS {
  double* tiles;
  const int* slot;
  const int* perm;
  int T;
  __device__ bool stores(int ci, int cj, int r, int cc) const { return ci != cj || cc <= r; }
  __device__ double* elem(long long R, long long C) const {
    const int s = slot[(R >> 6) * T + (C >> 6)];
    assert(s >= 0);   // every tile the assembly writes is in the pattern of the factor
    return tiles + static_cast<size_t>(s) * (kNB * kNB) + (R & 63) * kNB + (C & 63);
  }
  __device__ double* block(int ci, int cj, int r, int cc) const {
    const long long pi = perm[ci], pj = perm[cj];
    return pi >= pj ? elem(pi * 12 + r, pj * 12 + cc) : elem(pj * 12 + cc, pi * 12 + r);
  }
};

// tiles of the factor: tile(I, J); below(k, i) the i-th stored tile row under the diagonal of column k; left(k, i)
// the i-th stored tile column left of the diagonal of row k; pair(k, ..) the tiles (ti, tj), tj <= ti, the update
// of column k writes from this thread block
struct DenseTiles {
  double* S;
  long long ld;
  __device__ double* tile(int I, int J) const {
    return S + (static_cast<long long>(I) * kNB) * ld + static_cast<long long>(J) * kNB;
  }
  __device__ int below(int k, int i) const { return k + 1 + i; }
  __device__ int left(int, int i) const { return i; }
  __device__ bool pair(int k, int& ti, int& tj) const {
    ti = k + 1 + static_cast<int>(blockIdx.x);
    tj = k + 1 + static_cast<int>(blockIdx.y);
    return tj <= ti;
  }
};
struct SparseTiles {
  double* tiles;
  const int* slot;
  const int* col_ptr;
  const int* col_row;
  const int* row_ptr;
  const int* row_col;
  int T;
  static constexpr long long ld = kNB;
  __device__ double* tile(int I, int J) const {
    return tiles + static_cast<size_t>(slot[static_cast<long long>(I) * T + J]) * (kNB * kNB);
  }
  __device__ int below(int k, int i) const { return col_row[col_ptr[k] + 1 + i]; }
  __device__ int left(int k, int i) const { return row_col[row_ptr[k] + i]; }
  // blockIdx.x = i (i + 1) / 2 + j, j <= i, over the stored tiles below the diagonal of column k
  __device__ bool pair(int k, int& ti, int& tj) const {
    const long long p = blockIdx.x;
    int i = static_cast<int>((sqrt(8.0 * static_cast<double>(p) + 1.0) - 1.0) * 0.5);
    while (static_cast<long long>(i + 1) * (i + 2) / 2 <= p) ++i;
    while (static_cast<long long>(i) * (i + 1) / 2 > p) --i;
    const int j = static_cast<int>(p - static_cast<long long>(i) * (i + 1) / 2);
    ti = below(k, i);
    tj = below(k, j);
    return true;
  }
};

// block row i of S (lower triangle): S_ij -= (s_i s_j^T) o [(Wk_i^T Hll^-1 Wk_j) (x) (Xt Xt^T)] summed over the
// landmarks l seen by both cameras, in the order of camera i's observation list (landmarks ascending)
template <class Addr>
__global__ void __launch_bounds__(32 * kRowWarps)
k_schur_rows(DeviceIndex ix, const double* __restrict__ P, const double* __restrict__ X, double c1, double c2,
             Robust rb, const double* __restrict__ lm_scale, const double* __restrict__ hll_inv,
             const double* __restrict__ pose_scale, const double* __restrict__ Bmat, Addr S) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int ci = blockIdx.x; ci < ix.C; ci += gridDim.x) {
    Cam3x4 cam_i;
    load_cam(P, ci, cam_i);
    const double* si = pose_scale + 12 * static_cast<size_t>(ci);
    const int eb = ix.cam_ptr[ci], ee = ix.cam_ptr[ci + 1];
    for (int e = eb; e < ee; ++e) {
      const int l = ix.csc_lm[e];
      const double2 uvi = ix.csc_uv[e];
      const int ob = ix.lm_ptr[l], oe = ix.lm_ptr[l + 1];
      double x[4], sl[4], inv[6];
      load4(X + 4 * static_cast<size_t>(l), x);
      load4(lm_scale + 4 * static_cast<size_t>(l), sl);
#pragma unroll
      for (int k = 0; k < 6; ++k) inv[k] = hll_inv[6 * static_cast<size_t>(l) + k];
      double Wi[3][3], HWi[3][3];
      pose_wk(cam_i, uvi.x, uvi.y, x, sl, c1, c2, rb, Wi);
#pragma unroll
      for (int k = 0; k < 3; ++k) {   // HWi = Hll^-1 Wi, column by column
        const double col[3] = {Wi[0][k], Wi[1][k], Wi[2][k]};
        double out[3];
        sym3_mul(inv, col, out);
        HWi[0][k] = out[0];
        HWi[1][k] = out[1];
        HWi[2][k] = out[2];
      }
      for (int j = ob; j < oe; ++j) {
        const int cj = ix.obs_cam[j];
        if (cj > ci) break;                       // lower triangle; cameras ascend inside a landmark
        if (cj % kRowWarps != warp) continue;     // this warp's block columns
        Cam3x4 cam_j;
        load_cam(P, cj, cam_j);
        const double2 uvj = ix.obs_uv[j];
        double Wj[3][3], Q[3][3];
        pose_wk(cam_j, uvj.x, uvj.y, x, sl, c1, c2, rb, Wj);
#pragma unroll
        for (int a = 0; a < 3; ++a) {             // Q = Wi^T Hll^-1 Wj = HWi^T Wj
#pragma unroll
          for (int b2 = 0; b2 < 3; ++b2) Q[a][b2] = HWi[0][a] * Wj[0][b2] + HWi[1][a] * Wj[1][b2] + HWi[2][a] * Wj[2][b2];
        }
        const double* sj = pose_scale + 12 * static_cast<size_t>(cj);
        for (int t = lane; t < 144; t += 32) {
          const int r = t / 12, cc = t % 12;
          if (!S.stores(ci, cj, r, cc)) continue;
          double q = 0.0;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b2 = 0; b2 < 3; ++b2) q = (a == (r >> 2) && b2 == (cc >> 2)) ? Q[a][b2] : q;
          }
          const double val = si[r] * sj[cc] * q * x[r & 3] * x[cc & 3];
          double* dst = S.block(ci, cj, r, cc);
          *dst -= val;
        }
      }
    }
    // the diagonal block: + Bmat_i (which holds (s s^T) o Jp^T Jp + lambda I); warp (ci mod warps) owns it
    __syncwarp();
    if (ci % kRowWarps == warp) {
      for (int t = lane; t < 144; t += 32) {
        const int r = t / 12, cc = t % 12;
        if (S.stores(ci, ci, r, cc)) *S.block(ci, ci, r, cc) += Bmat[144 * static_cast<size_t>(ci) + t];
      }
    }
  }
}

// identity on the padding rows
template <class Addr>
__global__ void k_pad_identity(int n, int n_pad, Addr S) {
  const int i = n + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) *S.elem(i, i) = 1.0;
}

// ---- factorisation --------------------------------------------------------------------------------
// diagonal tile k: A = L L^T in shared memory (lower part read), L written back with a zero upper part,
// L^-1 written to linv[k].  info != 0: a pivot was not positive (the matrix is not positive definite).
template <class Tiles>
__global__ void __launch_bounds__(256)
k_potrf_tile(Tiles S, int k, double* __restrict__ linv, int* __restrict__ info) {
  __shared__ double A[kNB][kNB + 1];
  __shared__ int bad;
  double* tile = S.tile(k, k);
  const long long ld = S.ld;
  if (*info != 0) return;   // an earlier tile was not positive definite
  if (threadIdx.x == 0) bad = 0;
  for (int t = threadIdx.x; t < kNB * kNB; t += blockDim.x) {
    const int r = t / kNB, c = t % kNB;
    A[r][c] = c <= r ? tile[static_cast<long long>(r) * ld + c] : 0.0;
  }
  __syncthreads();
  for (int j = 0; j < kNB; ++j) {
    const double d = A[j][j];
    if (!(d > 0.0)) {           // also catches NaN
      if (threadIdx.x == 0) bad = 1;
      break;                    // uniform: every thread reads the same A[j][j]
    }
    const double sq = sqrt(d);
    __syncthreads();
    for (int r = j + threadIdx.x; r < kNB; r += blockDim.x) A[r][j] = (r == j) ? sq : A[r][j] / sq;
    __syncthreads();
    // trailing update of the lower triangle: A[r][c] -= A[r][j] A[c][j], j < c <= r
    const int m = kNB - 1 - j;
    for (int t = threadIdx.x; t < m * m; t += blockDim.x) {
      const int r = j + 1 + t / m, c = j + 1 + t % m;
      if (c <= r) A[r][c] -= A[r][j] * A[c][j];
    }
    __syncthreads();
  }
  __syncthreads();
  if (bad) {
    if (threadIdx.x == 0) atomicExch(info, k + 1);
    return;
  }
  // L^-1: column c by forward substitution (thread c), straight into linv[k] (a thread reads back only what it
  // wrote itself)
  double* li = linv + static_cast<size_t>(k) * kNB * kNB;
  if (threadIdx.x < kNB) {
    const int c = threadIdx.x;
    for (int r = 0; r < kNB; ++r) {
      if (r < c) {
        li[r * kNB + c] = 0.0;
        continue;
      }
      double v = (r == c) ? 1.0 : 0.0;
      for (int m2 = c; m2 < r; ++m2) v -= A[r][m2] * li[m2 * kNB + c];
      li[r * kNB + c] = v / A[r][r];
    }
  }
  for (int t = threadIdx.x; t < kNB * kNB; t += blockDim.x) {
    const int r = t / kNB, c = t % kNB;
    tile[static_cast<long long>(r) * ld + c] = A[r][c];
  }
}

// One 64x64 tile product on the FP64 tensor cores, 256 threads: warp w owns rows 8 w .. 8 w + 7 of the tile and
// all eight 8-column fragments.
//   kUpdate:  C(ti, tj) -= A(ti, k) A(tj, k)^T   for k < tj <= ti   (trailing update; dense: grid = (m, m), upper
//                                                                      skipped; tile-sparse: one block per pair)
//   kPanel:   A(ti, k)  = A(ti, k) Linv_k^T      for ti > k          (the panel below the diagonal tile)
enum TileMode { kUpdate = 0, kPanel = 1 };

template <int MODE, class Tiles>
__global__ void __launch_bounds__(256)
k_tile_gemm(Tiles S, int k, const double* __restrict__ linv, const int* __restrict__ info) {
  if (*info != 0) return;
  __shared__ double sA[kNB][kKC + kPad];
  __shared__ double sB[kNB][kKC + kPad];
  const long long ld = S.ld;
  int ti = 0, tj = k;
  if (MODE == kUpdate) {
    if (!S.pair(k, ti, tj)) return;
  } else {
    ti = S.below(k, static_cast<int>(blockIdx.x));
  }
  const double* Ap = S.tile(ti, k);
  const double* Bp = MODE == kUpdate ? S.tile(tj, k) : linv + static_cast<size_t>(k) * kNB * kNB;
  const long long ldb = MODE == kUpdate ? ld : kNB;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;
  double acc[8][2];
#pragma unroll
  for (int n = 0; n < 8; ++n) acc[n][0] = acc[n][1] = 0.0;
  for (int k0 = 0; k0 < kNB; k0 += kKC) {
    __syncthreads();
    for (int t = threadIdx.x; t < kNB * kKC; t += blockDim.x) {
      const int r = t / kKC, c = t % kKC;
      sA[r][c] = Ap[static_cast<long long>(r) * ld + k0 + c];
      sB[r][c] = Bp[static_cast<long long>(r) * ldb + k0 + c];
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kKC; kk += 4) {
      const double a = sA[8 * warp + fr][kk + fk];
#pragma unroll
      for (int n = 0; n < 8; ++n) dmma(acc[n], a, sB[8 * n + fr][kk + fk]);   // B^T: col-major fragment = rows of B
    }
  }
  // C fragment: row fr, columns 2 fk, 2 fk + 1 of the 8x8 tile
  double* Cp = MODE == kUpdate ? S.tile(ti, tj) : S.tile(ti, k);
  if (MODE == kPanel) __syncthreads();   // every warp has read the tile it is about to overwrite
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    double2* dst = reinterpret_cast<double2*>(Cp + static_cast<long long>(8 * warp + fr) * ld + 8 * n + 2 * fk);
    if (MODE == kUpdate) {
      double2 c = *dst;
      c.x -= acc[n][0];
      c.y -= acc[n][1];
      *dst = c;
    } else {
      *dst = make_double2(acc[n][0], acc[n][1]);
    }
  }
}

// ---- substitution ---------------------------------------------------------------------------------
// x_k = Linv_k r_k (forward) or Linv_k^T r_k (backward), in place; 64 threads
template <bool TRANS>
__global__ void __launch_bounds__(kNB)
k_solve_diag(int k, const double* __restrict__ linv, double* __restrict__ r, const int* __restrict__ info) {
  if (*info != 0) return;
  __shared__ double v[kNB];
  const double* li = linv + static_cast<size_t>(k) * kNB * kNB;
  const int i = threadIdx.x;
  v[i] = r[static_cast<size_t>(k) * kNB + i];
  __syncthreads();
  double s = 0.0;
  if (TRANS) {
    for (int m = i; m < kNB; ++m) s += li[m * kNB + i] * v[m];
  } else {
    for (int m = 0; m <= i; ++m) s += li[i * kNB + m] * v[m];
  }
  r[static_cast<size_t>(k) * kNB + i] = s;
}

// forward: r_i -= L(i, k) x_k for the rows of the stored tiles below tile row k (one thread per row; `rows` =
// 64 x those tiles)
template <class Tiles>
__global__ void __launch_bounds__(256)
k_solve_fwd_update(Tiles S, int k, int rows, double* __restrict__ r, const int* __restrict__ info) {
  if (*info != 0) return;
  __shared__ double xk[kNB];
  if (threadIdx.x < kNB) xk[threadIdx.x] = r[static_cast<size_t>(k) * kNB + threadIdx.x];
  __syncthreads();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows) return;
  const int ti = S.below(k, idx / kNB), rr = idx % kNB;
  const double* a = S.tile(ti, k) + static_cast<long long>(rr) * S.ld;
  double s = 0.0;
#pragma unroll 8
  for (int m = 0; m < kNB; ++m) s += a[m] * xk[m];
  r[static_cast<size_t>(ti) * kNB + rr] -= s;
}

// backward: r_j -= L(k, j)^T x_k for the columns of the stored tiles left of tile column k (one thread per column;
// `cols` = 64 x those tiles)
template <class Tiles>
__global__ void __launch_bounds__(256)
k_solve_bwd_update(Tiles S, int k, int cols, double* __restrict__ r, const int* __restrict__ info) {
  if (*info != 0) return;
  __shared__ double xk[kNB];
  if (threadIdx.x < kNB) xk[threadIdx.x] = r[static_cast<size_t>(k) * kNB + threadIdx.x];
  __syncthreads();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cols) return;
  const int tj = S.left(k, idx / kNB), cc = idx % kNB;
  const double* a = S.tile(k, tj) + cc;
  const long long ld = S.ld;
  double s = 0.0;
#pragma unroll 8
  for (int m = 0; m < kNB; ++m) s += a[static_cast<long long>(m) * ld] * xk[m];
  r[static_cast<size_t>(tj) * kNB + cc] -= s;
}

// the right-hand side into the factor order and the solution back
__global__ void k_perm_gather_neg(int n, const int* __restrict__ perm, const double* __restrict__ b,
                                  double* __restrict__ r) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) r[12 * static_cast<size_t>(perm[i / 12]) + i % 12] = -b[i];
}
__global__ void k_perm_scatter(int n, const int* __restrict__ perm, const double* __restrict__ r,
                               double* __restrict__ x) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = r[12 * static_cast<size_t>(perm[i / 12]) + i % 12];
}

}  // namespace

int chol_padded(int n) { return (n + kNB - 1) / kNB * kNB; }

void launch_schur_lower(const DeviceState& d, const ModelParams& mp, double* S, int n_pad, const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  int blocks = d.ix.C;
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  const DenseS a{S, n_pad};
  k_schur_rows<<<blocks, 32 * kRowWarps, 0, lc.stream>>>(d.ix, d.P, d.X, mp.c1, mp.c2, rb, d.lm_scale, d.hll_inv,
                                                         d.pose_scale, d.Bmat, a);
  const int n = 12 * d.ix.C;
  if (n_pad > n) k_pad_identity<<<1, kNB, 0, lc.stream>>>(n, n_pad, a);
  count(lc, n_pad > n ? 2 : 1);
}

void launch_schur_tiles(const DeviceState& d, const ModelParams& mp, const CholTilesDev& s, int n_pad,
                        const LaunchCfg& lc) {
  const Robust rb = {mp.robust_norm, mp.huber};
  int blocks = d.ix.C;
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  const TiledS a{s.tiles, s.slot, s.perm, s.T};
  k_schur_rows<<<blocks, 32 * kRowWarps, 0, lc.stream>>>(d.ix, d.P, d.X, mp.c1, mp.c2, rb, d.lm_scale, d.hll_inv,
                                                         d.pose_scale, d.Bmat, a);
  const int n = 12 * d.ix.C;
  if (n_pad > n) k_pad_identity<<<1, kNB, 0, lc.stream>>>(n, n_pad, a);
  count(lc, n_pad > n ? 2 : 1);
}

// A = L L^T (lower, in place), L^-1 of the diagonal tiles in linv [n_pad / 64][64][64]; *info = 1 + the first
// tile with a non-positive pivot, 0 if the matrix is positive definite
void launch_cholesky_factor(double* S, int n_pad, double* linv, int* info, const LaunchCfg& lc) {
  const int T = n_pad / kNB;
  const DenseTiles a{S, n_pad};
  cudaMemsetAsync(info, 0, sizeof(int), lc.stream);
  int launches = 0;
  for (int k = 0; k < T; ++k) {
    k_potrf_tile<<<1, 256, 0, lc.stream>>>(a, k, linv, info);
    ++launches;
    const int m = T - 1 - k;
    if (m > 0) {
      k_tile_gemm<kPanel><<<dim3(m, 1), 256, 0, lc.stream>>>(a, k, linv, info);
      k_tile_gemm<kUpdate><<<dim3(m, m), 256, 0, lc.stream>>>(a, k, linv, info);
      launches += 2;
    }
  }
  count(lc, launches);
}

// r <- (L L^T)^-1 r, r has n_pad entries
void launch_cholesky_solve(const double* S, int n_pad, const double* linv, double* r, const int* info,
                           const LaunchCfg& lc) {
  const int T = n_pad / kNB;
  const DenseTiles a{const_cast<double*>(S), n_pad};
  int launches = 0;
  for (int k = 0; k < T; ++k) {
    k_solve_diag<false><<<1, kNB, 0, lc.stream>>>(k, linv, r, info);
    ++launches;
    const int rows = n_pad - (k + 1) * kNB;
    if (rows > 0) {
      k_solve_fwd_update<<<(rows + 255) / 256, 256, 0, lc.stream>>>(a, k, rows, r, info);
      ++launches;
    }
  }
  for (int k = T - 1; k >= 0; --k) {
    k_solve_diag<true><<<1, kNB, 0, lc.stream>>>(k, linv, r, info);
    ++launches;
    const int cols = k * kNB;
    if (cols > 0) {
      k_solve_bwd_update<<<(cols + 255) / 256, 256, 0, lc.stream>>>(a, k, cols, r, info);
      ++launches;
    }
  }
  count(lc, launches);
}

namespace {
SparseTiles sparse_tiles(const CholTilesDev& s) {
  return SparseTiles{s.tiles, s.slot, s.col_ptr, s.col_row, s.row_ptr, s.row_col, s.T};
}
}  // namespace

// the same factorisation over the stored tiles only: column k's panel and the pairs of its stored tiles; *info as
// above, tiles numbered in the factor order
void launch_cholesky_factor_tiles(const CholPattern& p, const CholTilesDev& s, double* linv, int* info,
                                  const LaunchCfg& lc) {
  const SparseTiles a = sparse_tiles(s);
  cudaMemsetAsync(info, 0, sizeof(int), lc.stream);
  int launches = 0;
  for (int k = 0; k < p.T; ++k) {
    k_potrf_tile<<<1, 256, 0, lc.stream>>>(a, k, linv, info);
    ++launches;
    const long long m = p.col_ptr[k + 1] - p.col_ptr[k] - 1;
    if (m > 0) {
      k_tile_gemm<kPanel><<<dim3(static_cast<unsigned>(m), 1), 256, 0, lc.stream>>>(a, k, linv, info);
      k_tile_gemm<kUpdate><<<dim3(static_cast<unsigned>(m * (m + 1) / 2), 1), 256, 0, lc.stream>>>(a, k, linv, info);
      launches += 2;
    }
  }
  count(lc, launches);
}

// forward substitution down the column lists, backward up the row lists
void launch_cholesky_solve_tiles(const CholPattern& p, const CholTilesDev& s, const double* linv, double* r,
                                 const int* info, const LaunchCfg& lc) {
  const SparseTiles a = sparse_tiles(s);
  int launches = 0;
  for (int k = 0; k < p.T; ++k) {
    k_solve_diag<false><<<1, kNB, 0, lc.stream>>>(k, linv, r, info);
    ++launches;
    const int rows = (p.col_ptr[k + 1] - p.col_ptr[k] - 1) * kNB;
    if (rows > 0) {
      k_solve_fwd_update<<<(rows + 255) / 256, 256, 0, lc.stream>>>(a, k, rows, r, info);
      ++launches;
    }
  }
  for (int k = p.T - 1; k >= 0; --k) {
    k_solve_diag<true><<<1, kNB, 0, lc.stream>>>(k, linv, r, info);
    ++launches;
    const int cols = (p.row_ptr[k + 1] - p.row_ptr[k] - 1) * kNB;
    if (cols > 0) {
      k_solve_bwd_update<<<(cols + 255) / 256, 256, 0, lc.stream>>>(a, k, cols, r, info);
      ++launches;
    }
  }
  count(lc, launches);
}

void launch_perm_gather_neg(int C, const int* perm, const double* b, double* r, const LaunchCfg& lc) {
  const int n = 12 * C;
  k_perm_gather_neg<<<(n + 255) / 256, 256, 0, lc.stream>>>(n, perm, b, r);
  count(lc);
}

void launch_perm_scatter(int C, const int* perm, const double* r, double* x, const LaunchCfg& lc) {
  const int n = 12 * C;
  k_perm_scatter<<<(n + 255) / 256, 256, 0, lc.stream>>>(n, perm, r, x);
  count(lc);
}

}  // namespace povar
