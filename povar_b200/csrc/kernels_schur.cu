// Kernels of the explicit-Schur-complement solvers: PCG / RIPCG vector algebra (CHOLESKY: kernels_chol.cu).
//
// The reference forms S = Hpp - sum_l Hpl Hll^-1 Hlp as a hash map of 12x12 (11x11) blocks
// (sc/landmark_block.hpp:360-472, cg/block_sparse_matrix.hpp:152-345) and multiplies with it.  On the
// GPU PCG/RIPCG apply S implicitly,  S p = B p - E0 p,  with the same matrix-free E0 product as the
// power series (kernels_landmark.cu / kernels_camera.cu); only the block-Jacobi preconditioner needs
// the diagonal blocks of S (k_kron<KRON_SDIAG>).
#include <cuda_runtime.h>

#include "device_math.cuh"
#include "povar_internal.h"

namespace povar {

namespace {

constexpr int kBlock = 256;

inline void count(const LaunchCfg& lc, int n = 1) {
  if (lc.launch_counter) *lc.launch_counter += n;
}

__global__ void __launch_bounds__(kBlock)
k_axpby(int n, double a, const double* __restrict__ x, double b, const double* __restrict__ y,
        double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = (y != nullptr) ? a * x[i] + b * y[i] : a * x[i];
}

// two-stage deterministic dot product: per-block partials, then one block of k_cg_scalar adds them in order
__global__ void __launch_bounds__(kBlock)
k_dot_part(int n, const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ part) {
  __shared__ double smem[kBlock / 32];
  double acc[1] = {0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) acc[0] += x[i] * y[i];
  block_reduce<1>(acc, smem);
  if (threadIdx.x == 0) part[blockIdx.x] = acc[0];
}

// ---- conjugate gradients on the device (cg/conjugate_gradient.hpp:114-489): the scalar recurrences and every
// termination test of the reference's loop, one thread, after the ordered sum of the dot-product partials
__global__ void __launch_bounds__(kBlock)
k_cg_scalar(int nblocks, const double* __restrict__ part, int stage, int it, const int* __restrict__ it_base, double eta,
            int min_it, int max_it, CgState* cg, SeriesCtl* ctl) {
  if (stage != CG_BEGIN && ctl->done) return;
  if (it_base != nullptr) it += *it_base;
  __shared__ double smem[kBlock / 32];
  double acc[1] = {0.0};
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) acc[0] += part[b];
  block_reduce<1>(acc, smem);
  if (threadIdx.x != 0) return;
  const double v = acc[0];
  auto stop = [&]() {
    ctl->done = 1;
    ctl->iterations = it;
  };
  if (stage == CG_BEGIN) {            // |b|; x0 = 0, r = b, Q0 = -x.(b + r) = 0
    cg->norm_b = sqrt(v);
    cg->rho = 1.0;
    cg->last_rho = 1.0;
    cg->alpha = 0.0;
    cg->beta = 0.0;
    cg->q0 = 0.0;
    ctl->nonfinite = 0;
    ctl->peer_timeout = 0;
    ctl->iterations = 0;
    ctl->done = cg->norm_b == 0.0 ? 1 : 0;
  } else if (stage == CG_RHO) {       // rho = r.z; beta = rho / last_rho
    cg->last_rho = cg->rho;
    cg->rho = v;
    if (v == 0.0 || isinf(v)) {       // LINEAR_SOLVER_FAILURE
      stop();
      return;
    }
    if (it == 1) {
      cg->beta = 0.0;
    } else {
      const double beta = v / cg->last_rho;
      cg->beta = beta;
      if (beta == 0.0 || isinf(beta)) stop();
    }
  } else if (stage == CG_PQ) {        // alpha = rho / p.q
    if (v <= 0 || isinf(v)) {         // "Matrix is indefinite"
      stop();
      return;
    }
    const double alpha = cg->rho / v;
    cg->alpha = alpha;
    if (isinf(alpha)) stop();
  } else {                            // Q1 = -x.(b + r); zeta = it (Q1 - Q0) / Q1
    const double q1 = -1.0 * v;
    const double zeta = it * (q1 - cg->q0) / q1;
    if (zeta < eta && it >= min_it) { // LINEAR_SOLVER_SUCCESS
      stop();
      return;
    }
    cg->q0 = q1;
    // the residual-based test never fires: tol_r = r_tolerance * |b| < 0 (pso.r_tolerance = -1)
    if (it >= max_it) stop();
  }
}

// p = z (+ beta p);  x += alpha p;  r -= alpha q  -- with the device's scalars, nothing after termination
__global__ void __launch_bounds__(kBlock)
k_cg_update(int n, int what, int it, const int* __restrict__ it_base, const double* __restrict__ src,
            double* __restrict__ dst, const CgState* __restrict__ cg, const SeriesCtl* __restrict__ ctl) {
  if (ctl->done) return;
  if (it_base != nullptr) it += *it_base;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (what == CG_UPDATE_P) {
    dst[i] = it == 1 ? src[i] : 1.0 * src[i] + cg->beta * dst[i];
  } else if (what == CG_UPDATE_X) {
    dst[i] = 1.0 * dst[i] + cg->alpha * src[i];
  } else {
    dst[i] = 1.0 * dst[i] + (-cg->alpha) * src[i];
  }
}

__global__ void __launch_bounds__(kBlock)
k_finite_check(int n, const double* __restrict__ x, SeriesCtl* ctl) {
  bool bad = false;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    bad = bad || !isfinite(x[i]);
  }
  if (bad) atomicExch(&ctl->nonfinite, 1);
}

}  // namespace

void launch_axpby(const DeviceState& d, int n, double a, const double* x, double b, const double* y,
                  double* out, const LaunchCfg& lc) {
  (void)d;
  k_axpby<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(n, a, x, b, y, out);
  count(lc);
}

void launch_dot_partials(const DeviceState& d, int n, const double* x, const double* y, const LaunchCfg& lc) {
  int blocks = (n + kBlock - 1) / kBlock;
  const int cap = scalar_blocks(d);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_dot_part<<<blocks, kBlock, 0, lc.stream>>>(n, x, y, d.scalar_part);
  count(lc);
}

void launch_cg_scalar(const DeviceState& d, CgStage stage, int it, double eta, int min_it, int max_it,
                      const LaunchCfg& lc, const int* it_base) {
  int blocks = (d.ix.C * 12 + kBlock - 1) / kBlock;   // as launch_dot_partials for a camera-sized vector
  const int cap = scalar_blocks(d);
  if (blocks > cap) blocks = cap;
  k_cg_scalar<<<1, kBlock, 0, lc.stream>>>(blocks, d.scalar_part, static_cast<int>(stage), it, it_base, eta, min_it, max_it, d.cg,
                                           d.ctl);
  count(lc);
}

void launch_cg_update(const DeviceState& d, CgUpdate what, int n, int it, const double* src, double* dst,
                      const LaunchCfg& lc, const int* it_base) {
  k_cg_update<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(n, static_cast<int>(what), it, it_base, src, dst, d.cg,
                                                                   d.ctl);
  count(lc);
}

void launch_finite_check(const DeviceState& d, int n, const double* x, const LaunchCfg& lc) {
  int blocks = (n + kBlock - 1) / kBlock;
  if (blocks > sm_count() * 4) blocks = sm_count() * 4;
  k_finite_check<<<blocks, kBlock, 0, lc.stream>>>(n, x, d.ctl);
  count(lc);
}

}  // namespace povar
