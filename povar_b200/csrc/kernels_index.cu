// Device-side construction of the per-observation index arrays from the canonical landmark-major
// list (lm_ptr, obs_cam, obs_uv):  obs_lm, the camera-major copy (csc_lm, csc_uv) and the sliced-ELL
// copies (sell_cam, sell_uv, obs_slot; sell_cam_e0, sell_uv_e0, sell_row_e0).  The host only derives the small tables (tiles, items, slice
// table) -- scattering 5 M observations into three orders is a few hundred milliseconds of cache
// misses on one host core and well under a millisecond here.
//
// Canonical order = the reference's: landmark index, then camera index ascending
// (/root/reference/src/rootba_povar/bal/bal_problem.hpp:226); the camera-major order is the STABLE
// sort of it by camera (landmarks ascending inside a camera), made with a stable LSD radix sort.
#include <cuda_runtime.h>

#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "povar_internal.h"

namespace povar {

namespace {

constexpr int kBlock = 256;

__global__ void __launch_bounds__(kBlock)
k_obs_lm(int L, const int* __restrict__ lm_ptr, int* __restrict__ obs_lm) {
  // one warp per 32 landmarks would do; degrees are small, a thread per landmark is enough
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const int e = lm_ptr[l + 1];
  for (int o = lm_ptr[l]; o < e; ++o) obs_lm[o] = l;
}

// Validation of the canonical list and the per-camera counts, one thread per landmark (povar_create used to spend
// 9 of its 18 ms on this pass on the host).  out[0..C): observations per camera, out[C]: 1 = a camera index out
// of range, 2 = the cameras of a landmark are not strictly ascending.  SMEM: the counts of a block's landmarks
// go through a shared-memory histogram (integer sums: the result does not depend on the order).
template <bool SMEM>
__global__ void __launch_bounds__(kBlock)
k_validate_obs(int L, int C, const int* __restrict__ lm_ptr, const int* __restrict__ obs_cam, int* __restrict__ out) {
  extern __shared__ int hist[];
  if (SMEM) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) hist[c] = 0;
    __syncthreads();
  }
  int bad = 0;
  for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < L; l += gridDim.x * blockDim.x) {
    const int e = lm_ptr[l + 1];
    int prev = -1;
    for (int o = lm_ptr[l]; o < e; ++o) {
      const int c = obs_cam[o];
      if (static_cast<unsigned>(c) >= static_cast<unsigned>(C)) {
        bad |= 1;
        continue;
      }
      if (c <= prev) bad |= 2;
      prev = c;
      atomicAdd(SMEM ? &hist[c] : &out[c], 1);
    }
  }
  if (bad) atomicOr(&out[C], bad);
  if (SMEM) {
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const int n = hist[c];
      if (n != 0) atomicAdd(&out[c], n);
    }
  }
}

__global__ void __launch_bounds__(kBlock) k_iota(int n, int* __restrict__ v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = i;
}

__global__ void __launch_bounds__(kBlock)
k_csc_gather(int nnz, const int* __restrict__ perm, const int* __restrict__ obs_lm,
             const double2* __restrict__ obs_uv, int* __restrict__ csc_lm, double2* __restrict__ csc_uv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const int o = perm[e];
  csc_lm[e] = obs_lm[o];
  csc_uv[e] = obs_uv[o];
}

// first slot of every landmark in the sliced-ELL order (-1: not in the set)
__global__ void __launch_bounds__(kBlock)
k_lm_slot(int groups, const int* __restrict__ slice_ptr, const int* __restrict__ sell_lm,
          int* __restrict__ lm_slot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= groups) return;
  const int lm = sell_lm[i];
  if (lm >= 0) lm_slot[lm] = kSellWidth * slice_ptr[i / kSellWidth] + (i % kSellWidth);
}

// Row of every observation inside its slice.  A lane of the landmark-major walks (sell_walk.cuh) reads the record
// of its observation's camera from shared memory with LDS.128; the eight lanes of a quarter warp are served
// together, and two of them collide when their records start in the same bank group, i.e. (records are an odd
// number of 16-byte units) when their cameras are congruent mod 8.  With the k-th observation of every landmark in
// row k the eight cameras of a quarter are as good as random: 2.55 wavefronts per quarter instead of 1, and the
// walks are bound by exactly that.  The order of a landmark's observations is free -- it only fixes the order of
// its sums -- so one thread per quarter warp places the observations of its eight landmarks greedily: each goes to
// a free row (of this landmark) whose fullest class it does not raise, else where the fewest lanes of the quarter
// have a camera of the same class (2.59 -> 1.9 wavefronts per quarter on random cameras).
// Deterministic (a function of the layout alone); rows beyond a landmark's degree are padding wherever they end up.
__global__ void __launch_bounds__(128)
k_sell_rows(int quarters, const int* __restrict__ slice_ptr, const int* __restrict__ sell_lm,
            const int* __restrict__ lm_ptr, const int* __restrict__ obs_cam, unsigned char* __restrict__ obs_row) {
  // per row: eight 4-bit counters, one per camera class; a column of shared memory per thread (indexed by row at
  // run time: in registers it would live in local memory)
  __shared__ unsigned int hist_s[32][128];
  __shared__ unsigned char rmax_s[32][128];   // the fullest class of each row (kept beside the counters: the
                                              // search below looks at it once per row and observation)
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= quarters) return;
  const int sl = q >> 2;
  const int len = slice_ptr[sl + 1] - slice_ptr[sl];   // 1..32 rows
  unsigned int (*hist)[128] = reinterpret_cast<unsigned int (*)[128]>(&hist_s[0][threadIdx.x]);
  unsigned char (*rmax)[128] = reinterpret_cast<unsigned char (*)[128]>(&rmax_s[0][threadIdx.x]);
  for (int r = 0; r < len; ++r) {
    hist[r][0] = 0u;
    rmax[r][0] = 0;
  }
  auto row_max = [](unsigned int h) {
    unsigned int m = 0u;
#pragma unroll
    for (int g = 0; g < 8; ++g) m = max(m, (h >> (4 * g)) & 0xfu);
    return m;
  };
  // one greedy pass, then two in which every landmark is taken out and placed again knowing all the others
  for (int sweep = 0; sweep < 3; ++sweep) {
    for (int j = 0; j < 8; ++j) {
      const int lm = sell_lm[kSellWidth * sl + 8 * (q & 3) + j];
      if (lm < 0) continue;
      const int ob = lm_ptr[lm], oe = lm_ptr[lm + 1];
      if (sweep > 0) {
        for (int o = ob; o < oe; ++o) {
          const int r = obs_row[o];
          const unsigned int h = hist[r][0] - (1u << (4 * (obs_cam[o] & 7)));
          hist[r][0] = h;
          rmax[r][0] = static_cast<unsigned char>(row_max(h));
        }
      }
      unsigned int used = 0u;
      for (int o = ob; o < oe; ++o) {
        const int shift = 4 * (obs_cam[o] & 7);
        int best = 0;
        unsigned int best_key = 0xffffu;
        for (int r = 0; r < len; ++r) {
          if ((used >> r) & 1u) continue;
          // what the row costs is its fullest class: first the rows where this observation does not raise it
          const unsigned int cnt = (hist[r][0] >> shift) & 0xfu;
          const unsigned int key = (cnt + 1u > rmax[r][0] ? 16u : 0u) + cnt;
          if (key < best_key) {
            best_key = key;
            best = r;
          }
        }
        used |= 1u << best;
        const unsigned int h = hist[best][0] + (1u << shift);
        hist[best][0] = h;
        rmax[best][0] = static_cast<unsigned char>(max(static_cast<unsigned int>(rmax[best][0]), (h >> shift) & 0xfu));
        obs_row[o] = static_cast<unsigned char>(best);
      }
    }
  }
}

__global__ void __launch_bounds__(kBlock)
k_sell_fill(int nnz, const int* __restrict__ lm_ptr, const int* __restrict__ obs_lm,
            const int* __restrict__ obs_cam, const double2* __restrict__ obs_uv,
            const int* __restrict__ lm_slot, const unsigned char* __restrict__ obs_row,
            int* __restrict__ sell_cam, double2* __restrict__ sell_uv, int* __restrict__ sell_cam_e0,
            double2* __restrict__ sell_uv_e0, unsigned char* __restrict__ sell_row_e0,
            int* __restrict__ obs_slot) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= nnz) return;
  const int l = obs_lm[o];
  const int base = lm_slot[l];
  int slot = -1;
  if (base >= 0) {
    slot = base + kSellWidth * (o - lm_ptr[l]);
    const int slot_e0 = base + kSellWidth * obs_row[o];
    const int c = obs_cam[o];
    const double2 uv = obs_uv[o];
    sell_cam[slot] = c;
    sell_uv[slot] = uv;
    sell_cam_e0[slot_e0] = c;
    sell_uv_e0[slot_e0] = uv;
    sell_row_e0[slot] = obs_row[o];
  }
  obs_slot[o] = slot;
}

// ---- the sliced-ELL order on the device (the rule of build_sell, engine.cu) -----------------------------------
// sell_key of engine.cu: centre of the first stretch of `span` cameras that holds most of the observations
__device__ __forceinline__ int sell_key_dev(const int* __restrict__ cams, int deg, int span) {
  int best_i = 0, best_j = 0;
  for (int i = 0, j = 0; i < deg; ++i) {
    if (j < i) j = i;
    while (j + 1 < deg && cams[j + 1] - cams[i] < span) ++j;
    if (j - i > best_j - best_i) {
      best_i = i;
      best_j = j;
    }
  }
  return (cams[best_i] + cams[best_j]) / 2;
}

// key of every landmark: its key camera, or num_cams (sorts last) for the landmarks outside the set
__global__ void __launch_bounds__(kBlock)
k_sell_keys(int L, int num_cams, int span, int max_deg, const int* __restrict__ lm_ptr, const int* __restrict__ obs_cam,
            int* __restrict__ keys, int* __restrict__ ids) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const int b = lm_ptr[l], deg = lm_ptr[l + 1] - b;
  keys[l] = (deg >= 1 && deg <= max_deg) ? sell_key_dev(obs_cam + b, deg, span) : num_cams;
  ids[l] = l;
}

// second key of the n landmarks of the set, in key order: (window, 32 - degree)
__global__ void __launch_bounds__(kBlock)
k_sell_window_keys(int n, int window, const int* __restrict__ ids, const int* __restrict__ lm_ptr,
                   int* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int l = ids[i];
  keys[i] = ((i / window) << 6) | (32 - (lm_ptr[l + 1] - lm_ptr[l]));
}

// one warp per slice: the landmarks of the slice (padding -1), its number of rows (= the degree of its first
// landmark: the largest), the cameras it meets
__global__ void __launch_bounds__(kBlock)
k_sell_slices(int num_slices, int n, const int* __restrict__ ids, const int* __restrict__ lm_ptr,
              const int* __restrict__ obs_cam, int* __restrict__ sell_lm, int* __restrict__ slice_len,
              int* __restrict__ slice_lo, int* __restrict__ slice_hi) {
  const int sl = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (sl >= num_slices) return;
  const int i = kSellWidth * sl + lane;
  int lm = -1, deg = 0, lo = 0x7fffffff, hi = -1;
  if (i < n) {
    lm = ids[i];
    const int b = lm_ptr[lm], e = lm_ptr[lm + 1];
    deg = e - b;
    lo = obs_cam[b];
    hi = obs_cam[e - 1];
  }
  sell_lm[i] = lm;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off));
  }
  deg = __shfl_sync(0xffffffffu, deg, 0);
  if (lane == 0) {
    slice_len[sl] = deg;
    slice_lo[sl] = lo;
    slice_hi[sl] = hi;
  }
}

}  // namespace

// out: C + 1 zeroed ints (k_validate_obs); lm_ptr has been checked on the host (monotone, inside the list)
cudaError_t validate_obs(int L, int C, int sms, const int* lm_ptr, const int* obs_cam, int* out, const LaunchCfg& lc) {
  if (L <= 0) return cudaSuccess;
  const size_t smem = sizeof(int) * static_cast<size_t>(C);
  const int blocks = std::max(1, std::min((L + kBlock - 1) / kBlock, 4 * sms));
  if (smem <= 200 * 1024) {
    if (smem > 48 * 1024) {
      const cudaError_t e = cudaFuncSetAttribute(k_validate_obs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(smem));
      if (e != cudaSuccess) return e;
    }
    k_validate_obs<true><<<blocks, kBlock, smem, lc.stream>>>(L, C, lm_ptr, obs_cam, out);
  } else {
    k_validate_obs<false><<<blocks, kBlock, 0, lc.stream>>>(L, C, lm_ptr, obs_cam, out);
  }
  if (lc.launch_counter) *lc.launch_counter += 1;
  return cudaGetLastError();
}

size_t index_sort_temp_bytes(int nnz, int num_cams) {
  size_t bytes = 0;
  int bits = 1;
  while ((1 << bits) < num_cams) ++bits;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, static_cast<const int*>(nullptr), static_cast<int*>(nullptr),
                                  static_cast<const int*>(nullptr), static_cast<int*>(nullptr), nnz, 0, bits);
  return bytes;
}

// scratch: iota [nnz] (reused for the row numbers once the sort is done), keys_out [nnz], perm [nnz], lm_slot [L],
// cub temp
cudaError_t build_device_index(const DeviceIndex& ix, int* iota, int* keys_out, int* perm, int* lm_slot,
                               void* sort_temp, size_t sort_temp_bytes, const LaunchCfg& lc) {
  const int nnz = ix.nnz, L = ix.L;
  cudaStream_t st = lc.stream;
  int launches = 0;
  if (L > 0) {
    k_obs_lm<<<(L + kBlock - 1) / kBlock, kBlock, 0, st>>>(L, ix.lm_ptr, ix.obs_lm);
    ++launches;
  }
  if (nnz > 0) {
    const int blocks = (nnz + kBlock - 1) / kBlock;
    k_iota<<<blocks, kBlock, 0, st>>>(nnz, iota);
    int bits = 1;
    while ((1 << bits) < ix.C) ++bits;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(sort_temp, sort_temp_bytes, ix.obs_cam, keys_out, iota,
                                                    perm, nnz, 0, bits, st);
    if (e != cudaSuccess) return e;
    k_csc_gather<<<blocks, kBlock, 0, st>>>(nnz, perm, ix.obs_lm, ix.obs_uv, ix.csc_lm, ix.csc_uv);
    e = cudaMemsetAsync(lm_slot, 0xFF, sizeof(int) * static_cast<size_t>(L), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(ix.sell_cam, 0xFF, sizeof(int) * static_cast<size_t>(ix.sell_slots), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(ix.sell_cam_e0, 0xFF, sizeof(int) * static_cast<size_t>(ix.sell_slots), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(ix.sell_row_e0, 0, static_cast<size_t>(ix.sell_slots), st);
    if (e != cudaSuccess) return e;
    const int groups = kSellWidth * ix.num_slices;
    if (groups > 0) {
      k_lm_slot<<<(groups + kBlock - 1) / kBlock, kBlock, 0, st>>>(groups, ix.slice_ptr, ix.sell_lm, lm_slot);
      ++launches;
    }
    unsigned char* obs_row = reinterpret_cast<unsigned char*>(iota);   // the sort has consumed iota
    const int quarters = 4 * ix.num_slices;
    if (quarters > 0) {
      k_sell_rows<<<(quarters + 127) / 128, 128, 0, st>>>(quarters, ix.slice_ptr, ix.sell_lm, ix.lm_ptr, ix.obs_cam,
                                                         obs_row);
      ++launches;
    }
    k_sell_fill<<<blocks, kBlock, 0, st>>>(nnz, ix.lm_ptr, ix.obs_lm, ix.obs_cam, ix.obs_uv, lm_slot, obs_row,
                                           ix.sell_cam, ix.sell_uv, ix.sell_cam_e0, ix.sell_uv_e0, ix.sell_row_e0,
                                           ix.obs_slot);
    launches += 5;   // iota, radix sort (counted once), gather, fill
  }
  if (lc.launch_counter) *lc.launch_counter += launches;
  return cudaGetLastError();
}

// The sliced-ELL order of the n landmarks with 1..32 observations, made on the device with the rule of
// build_sell (engine.cu): stable radix sort by key camera, then by (window, descending degree).  Out: sell_lm
// [32 * ceil(n / 32)], slice_len / slice_lo / slice_hi [ceil(n / 32)].  Scratch: keys_a, keys_b, ids_a, ids_b [L],
// cub temp of sell_sort_temp_bytes.
size_t sell_sort_temp_bytes(int L, int num_cams, int n, int window) {
  size_t a = 0, b = 0;
  int bits1 = 1;
  while ((1 << bits1) <= num_cams) ++bits1;
  int bits2 = 7;
  while ((1LL << (bits2 - 6)) <= (n + window - 1) / window) ++bits2;
  cub::DeviceRadixSort::SortPairs(nullptr, a, static_cast<const int*>(nullptr), static_cast<int*>(nullptr),
                                  static_cast<const int*>(nullptr), static_cast<int*>(nullptr), L, 0, bits1);
  cub::DeviceRadixSort::SortPairs(nullptr, b, static_cast<const int*>(nullptr), static_cast<int*>(nullptr),
                                  static_cast<const int*>(nullptr), static_cast<int*>(nullptr), n > 0 ? n : 1, 0, bits2);
  return a > b ? a : b;
}

cudaError_t build_device_sell(int L, int num_cams, int n, int window, int max_deg, const int* lm_ptr, const int* obs_cam,
                              int* keys_a, int* keys_b, int* ids_a, int* ids_b, void* sort_temp,
                              size_t sort_temp_bytes, int* sell_lm, int* slice_len, int* slice_lo, int* slice_hi,
                              const LaunchCfg& lc) {
  if (L <= 0 || n <= 0) return cudaSuccess;
  cudaStream_t st = lc.stream;
  int bits1 = 1;
  while ((1 << bits1) <= num_cams) ++bits1;
  int bits2 = 7;
  while ((1LL << (bits2 - 6)) <= (n + window - 1) / window) ++bits2;
  k_sell_keys<<<(L + kBlock - 1) / kBlock, kBlock, 0, st>>>(L, num_cams, kSellKeySpan, max_deg, lm_ptr, obs_cam, keys_a,
                                                            ids_a);
  cudaError_t e = cub::DeviceRadixSort::SortPairs(sort_temp, sort_temp_bytes, keys_a, keys_b, ids_a, ids_b, L, 0,
                                                  bits1, st);
  if (e != cudaSuccess) return e;
  // the first n of ids_b are the landmarks of the set in key order
  k_sell_window_keys<<<(n + kBlock - 1) / kBlock, kBlock, 0, st>>>(n, window, ids_b, lm_ptr, keys_a);
  e = cub::DeviceRadixSort::SortPairs(sort_temp, sort_temp_bytes, keys_a, keys_b, ids_b, ids_a, n, 0, bits2, st);
  if (e != cudaSuccess) return e;
  const int num_slices = (n + kSellWidth - 1) / kSellWidth;
  k_sell_slices<<<(num_slices * 32 + kBlock - 1) / kBlock, kBlock, 0, st>>>(num_slices, n, ids_a, lm_ptr, obs_cam,
                                                                          sell_lm, slice_len, slice_lo, slice_hi);
  if (lc.launch_counter) *lc.launch_counter += 5;
  return cudaGetLastError();
}

// ---- canonical order of an unordered observation list (povar_create_device) -----------------------------------
// The order of povar_canonical_order (host/bal_io.cpp): landmark, then camera ascending.  Every observation of the
// list gets the 64-bit key (landmark << cam_bits) | camera, one radix sort by key brings them into that order, and
// the shard [lm_begin, lm_end) is then one contiguous run of the sorted list.  The keys are those of the whole
// problem, not of the shard, so that every rank sees a duplicate pair or an index out of range anywhere in the list
// and fails its povar_create_device, as povar_canonical_order fails for every rank of the host route.
namespace {

// key of every entry (all ones for an entry with an index out of range: it sorts last), its position, and the
// counts: info[kOrderBefore] valid entries of landmarks below lm_begin, info[kOrderCount] of the shard,
// info[kOrderFlags] |= 1 for an index out of range.  Integer sums: the counts do not depend on the order of the
// atomics.
__global__ void __launch_bounds__(kBlock)
k_obs_keys(int n, int C, int num_lms, int lm_begin, int lm_end, int cam_bits, const int* __restrict__ obs_cam,
           const int* __restrict__ obs_lm, unsigned long long* __restrict__ keys, int* __restrict__ pos,
           int* __restrict__ info) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool before = false, in = false, bad = false;
  if (i < n) {
    const int c = obs_cam[i], l = obs_lm[i];
    bad = static_cast<unsigned>(c) >= static_cast<unsigned>(C) || static_cast<unsigned>(l) >= static_cast<unsigned>(num_lms);
    keys[i] = bad ? ~0ULL : (static_cast<unsigned long long>(l) << cam_bits) | static_cast<unsigned>(c);
    pos[i] = i;
    before = !bad && l < lm_begin;
    in = !bad && l >= lm_begin && l < lm_end;
  }
  const int nb = __syncthreads_count(before), ni = __syncthreads_count(in), nbad = __syncthreads_or(bad);
  if (threadIdx.x == 0) {
    if (nb) atomicAdd(&info[kOrderBefore], nb);
    if (ni) atomicAdd(&info[kOrderCount], ni);
    if (nbad) atomicOr(&info[kOrderFlags], 1);
  }
}

// One thread per sorted entry: equal neighbours are a duplicate pair (info[kOrderFlags] |= 2); an entry of the shard
// goes to its place in the landmark-major arrays, and the first entry of every landmark opens the ranges of the
// landmarks up to its own (those in between have no observations: empty ranges, as povar_canonical_order makes
// them); the last entry of the shard closes the ranges of the landmarks after it.
__global__ void __launch_bounds__(kBlock)
k_obs_place(int n, int cam_bits, int lm_begin, int L, const unsigned long long* __restrict__ keys,
            const int* __restrict__ pos, const double* __restrict__ uv_in, int* __restrict__ info,
            int* __restrict__ lm_ptr, int* __restrict__ obs_cam, int* __restrict__ obs_lm, double2* __restrict__ obs_uv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = keys[i];
  if (key == ~0ULL) return;   // an index out of range, already flagged
  if (i > 0 && keys[i - 1] == key) atomicOr(&info[kOrderFlags], 2);
  const int l = static_cast<int>(key >> cam_bits) - lm_begin;
  if (l < 0 || l >= L) return;
  const int lo = info[kOrderBefore], cnt = info[kOrderCount];
  const int p = i - lo;
  const int src = pos[i];
  obs_cam[p] = static_cast<int>(key & ((1ULL << cam_bits) - 1));
  obs_lm[p] = l;
  obs_uv[p] = make_double2(uv_in[2 * static_cast<size_t>(src)], uv_in[2 * static_cast<size_t>(src) + 1]);
  const int prev = p == 0 ? -1 : static_cast<int>(keys[i - 1] >> cam_bits) - lm_begin;
  for (int m = prev + 1; m <= l; ++m) lm_ptr[m] = p;
  if (p == cnt - 1) {
    for (int m = l + 1; m <= L; ++m) lm_ptr[m] = cnt;
  }
}

// The landmark table of Engine::upload on the device: info[kOrderSell] landmarks with 1..max_deg observations, and
// is_long[l] for the stable compaction of the long ones (max_deg = sell_max_degree of the shard's observation count).
__global__ void __launch_bounds__(kBlock)
k_lm_table(int L, int sms, const int* __restrict__ lm_ptr, int* __restrict__ info, unsigned char* __restrict__ is_long) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  const int max_deg = sell_max_degree(info[kOrderCount], sms);
  bool sell = false;
  if (l < L) {
    const int deg = lm_ptr[l + 1] - lm_ptr[l];
    is_long[l] = deg > max_deg ? 1 : 0;
    sell = deg > 0 && deg <= max_deg;
  }
  const int ns = __syncthreads_count(sell);
  if (threadIdx.x == 0 && ns) atomicAdd(&info[kOrderSell], ns);
}

int value_bits(long long n) {   // bits that hold every value below n
  int b = 1;
  while ((1LL << b) < n) ++b;
  return b;
}

}  // namespace

int order_cam_bits(int num_cams) { return value_bits(num_cams); }

// the key of an entry of landmark num_lms - 1 stays below the all-ones key of the rejected entries
int order_end_bit(int num_cams, int num_lms) { return order_cam_bits(num_cams) + value_bits(num_lms + 1LL); }

size_t device_order_temp_bytes(int n, int L, int end_bit) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, a, static_cast<const unsigned long long*>(nullptr),
                                  static_cast<unsigned long long*>(nullptr), static_cast<const int*>(nullptr),
                                  static_cast<int*>(nullptr), n > 0 ? n : 1, 0, end_bit);
  cub::DeviceSelect::Flagged(nullptr, b, cub::CountingInputIterator<int>(0), static_cast<const unsigned char*>(nullptr),
                             static_cast<int*>(nullptr), static_cast<int*>(nullptr), L > 0 ? L : 1);
  return a > b ? a : b;
}

cudaError_t device_order_keys(int n, int C, int num_lms, int lm_begin, int lm_end, const int* obs_cam, const int* obs_lm,
                              unsigned long long* keys, int* pos, int* info, const LaunchCfg& lc) {
  if (n <= 0) return cudaSuccess;
  k_obs_keys<<<(n + kBlock - 1) / kBlock, kBlock, 0, lc.stream>>>(n, C, num_lms, lm_begin, lm_end, order_cam_bits(C),
                                                                  obs_cam, obs_lm, keys, pos, info);
  if (lc.launch_counter) *lc.launch_counter += 1;
  return cudaGetLastError();
}

cudaError_t device_order_sort(int n, int end_bit, const unsigned long long* keys_in, unsigned long long* keys_out,
                              const int* pos_in, int* pos_out, void* temp, size_t temp_bytes, const LaunchCfg& lc) {
  if (n <= 0) return cudaSuccess;
  const cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, pos_in, pos_out, n, 0,
                                                        end_bit, lc.stream);
  if (lc.launch_counter) *lc.launch_counter += 1;   // counted once, like the other radix sorts
  return e;
}

cudaError_t device_order_place(int n, int C, int lm_begin, int sms, const unsigned long long* keys, const int* pos,
                               const double* obs_uv_in, int* info, const DeviceIndex& ix, unsigned char* is_long,
                               int* long_lms, void* temp, size_t temp_bytes, const LaunchCfg& lc) {
  cudaStream_t st = lc.stream;
  const int L = ix.L;
  int launches = 0;
  if (n > 0) {
    k_obs_place<<<(n + kBlock - 1) / kBlock, kBlock, 0, st>>>(n, order_cam_bits(C), lm_begin, L, keys, pos, obs_uv_in,
                                                              info, ix.lm_ptr, ix.obs_cam, ix.obs_lm, ix.obs_uv);
    ++launches;
  }
  if (L > 0) {
    k_lm_table<<<(L + kBlock - 1) / kBlock, kBlock, 0, st>>>(L, sms, ix.lm_ptr, info, is_long);
    const cudaError_t e = cub::DeviceSelect::Flagged(temp, temp_bytes, cub::CountingInputIterator<int>(0), is_long,
                                                     long_lms, info + kOrderLong, L, st);
    if (e != cudaSuccess) return e;
    launches += 2;
  }
  if (lc.launch_counter) *lc.launch_counter += launches;
  return cudaGetLastError();
}

namespace {
// one warp per landmark: bits (a, b) and (b, a) for every pair of its cameras, the diagonal included.  atomicOr is
// idempotent, so the bitmap does not depend on the order.
__global__ void __launch_bounds__(kBlock)
k_covisibility(int L, int words, const int* __restrict__ lm_ptr, const int* __restrict__ obs_cam,
               unsigned int* __restrict__ bits) {
  const int lane = threadIdx.x & 31;
  const int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (l >= L) return;
  const int ob = lm_ptr[l], deg = lm_ptr[l + 1] - ob;
  for (long long p = lane; p < static_cast<long long>(deg) * deg; p += 32) {
    const int a = obs_cam[ob + static_cast<int>(p / deg)], b = obs_cam[ob + static_cast<int>(p % deg)];
    atomicOr(bits + static_cast<size_t>(a) * words + (b >> 5), 1u << (b & 31));
  }
}
}  // namespace

cudaError_t build_covisibility(int L, int C, const int* lm_ptr, const int* obs_cam, unsigned int* bits,
                               const LaunchCfg& lc) {
  const int words = (C + 31) / 32;
  cudaError_t e = cudaMemsetAsync(bits, 0, sizeof(unsigned int) * static_cast<size_t>(C) * words, lc.stream);
  if (e != cudaSuccess || L <= 0) return e;
  const long long threads = 32LL * L;
  k_covisibility<<<static_cast<unsigned>((threads + kBlock - 1) / kBlock), kBlock, 0, lc.stream>>>(L, words, lm_ptr,
                                                                                                  obs_cam, bits);
  if (lc.launch_counter) *lc.launch_counter += 1;
  return cudaGetLastError();
}

}  // namespace povar
