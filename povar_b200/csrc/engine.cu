// Engine: device state of one landmark shard + kernel sequencing for the PoVar hot path.
//
// Mirrors, per call, what LinearizorPowerVarproj / LinearizorSC do
// (/root/reference/src/rootba_povar/solver/linearizor_power_varproj.cpp, linearizor_sc.cpp):
//   linearize  -> landmark pass (Jl^T Jl, Jl^T r, column scales) + camera pass (Jp^T Jp) + scales
//   solve      -> Hll^-1, B^-1, b, then the power series (or PCG / Cholesky)
//   apply      -> back-substitution + camera update, model cost change
// The Jacobian blocks are never stored: see device_math.cuh.
#include "engine.h"

#include <dlfcn.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>
#include <numeric>
#include <thread>

namespace povar {

// ---------------------------------------------------------------------------------------------
// NCCL through dlopen: libpovar_b200.so stays loadable on a box without NCCL; the entry points
// are only needed when world_size > 1.
// ---------------------------------------------------------------------------------------------
struct Id128 {   // ncclUniqueId: 128 opaque bytes, passed by value
  char bytes[128];
};
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Id128, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi* load_nccl(std::string* err) {
  static NcclApi api;
  if (api.lib) return &api;
  const char* names[] = {getenv("POVAR_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n) continue;
    api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) {
    if (err) *err = "cannot dlopen libnccl.so.2 (set POVAR_NCCL_LIB)";
    return nullptr;
  }
  api.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(api.lib, "ncclGetUniqueId"));
  api.CommInitRank =
      reinterpret_cast<int (*)(void**, int, Id128, int)>(dlsym(api.lib, "ncclCommInitRank"));
  api.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
      dlsym(api.lib, "ncclAllReduce"));
  api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(api.lib, "ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(api.lib, "ncclGetErrorString"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) {
    if (err) *err = "libnccl is missing expected symbols";
    dlclose(api.lib);
    api.lib = nullptr;
    return nullptr;
  }
  return &api;
}

static std::mutex& comm_cache_mutex() {
  static std::mutex m;
  return m;
}
static std::map<std::string, void*>& comm_cache() {
  static std::map<std::string, void*> cache;
  return cache;
}
// Stream, events and the page-locked scratch of a handle are kept for the next handle on the same device instead of
// being destroyed: cudaHostAlloc / cudaFreeHost are the erratic part of povar_create / povar_destroy (3 ms and 0.5 ms
// as a rule, 130 ms for one cudaFreeHost in a trace, and the likely cause of end-to-end steps of 420 to 580 ms on
// some hosts).  A kit goes back only after its stream was synchronised.
struct HostKit {
  int device = -1;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double* pinned = nullptr;   // 256 bytes
};
static std::mutex& kit_mutex() {
  static std::mutex m;
  return m;
}
static std::vector<HostKit>& kit_cache() {
  static std::vector<HostKit> cache;
  return cache;
}
static bool take_kit(int device, HostKit* out) {
  std::lock_guard<std::mutex> lock(kit_mutex());
  auto& cache = kit_cache();
  for (size_t i = 0; i < cache.size(); ++i) {
    if (cache[i].device == device) {
      *out = cache[i];
      cache.erase(cache.begin() + static_cast<long>(i));
      return true;
    }
  }
  return false;
}
static void give_kit(const HostKit& kit) {
  std::lock_guard<std::mutex> lock(kit_mutex());
  kit_cache().push_back(kit);
}

struct PeerShared {
  void* mem = nullptr;            // this rank's receive buffer + flags (cudaMalloc, IPC-exported)
  std::vector<void*> opened;      // the peers' buffers as mapped here
  PeerExchange px{};
  bool ok = false;
  void release() {
    ok = false;
    for (void* p : opened) cudaIpcCloseMemHandle(p);
    opened.clear();
    if (mem) cudaFree(mem);
    mem = nullptr;
    cudaGetLastError();
  }
};
static std::map<std::string, PeerShared*>& peer_cache() {
  static std::map<std::string, PeerShared*> cache;
  return cache;
}
static std::string comm_key(const povar_comm_desc& c) {
  std::string key(reinterpret_cast<const char*>(c.nccl_id), 128);
  key += ":" + std::to_string(c.rank) + ":" + std::to_string(c.world_size) + ":" + std::to_string(c.device);
  return key;
}

static void release_rendezvous();   // host rendezvous segments (below)

// destroys every cached communicator; handles made with them must have been destroyed before
int nccl_finalize() {
  std::lock_guard<std::mutex> lock(comm_cache_mutex());
  NcclApi* api = comm_cache().empty() ? nullptr : load_nccl(nullptr);
  for (auto& kv : peer_cache()) {
    kv.second->release();
    delete kv.second;
  }
  peer_cache().clear();
  release_rendezvous();
  for (auto& kv : comm_cache()) {
    if (api && kv.second) api->CommDestroy(kv.second);
  }
  comm_cache().clear();
  return POVAR_OK;
}

int nccl_unique_id(uint8_t id[128], std::string* err) {
  NcclApi* api = load_nccl(err);
  if (!api) return POVAR_ERR_NCCL;
  const int rc = api->GetUniqueId(id);
  if (rc != 0) {
    if (err) *err = std::string("ncclGetUniqueId: ") + (api->GetErrorString ? api->GetErrorString(rc) : "?");
    return POVAR_ERR_NCCL;
  }
  return POVAR_OK;
}

// ---------------------------------------------------------------------------------------------
// Host rendezvous: a POSIX shared-memory segment instead of an NCCL communicator for the ONE thing the
// communicator is needed for when the peer buffers carry every reduction -- swapping the CUDA IPC handles at
// set-up.  Selected by a communicator id that starts with kHostIdMagic (povar_comm_host_id).  It is what lets
// several ranks share one device (NCCL refuses two ranks on the same GPU): the sharded arithmetic, the IPC
// mapping and the tagged peer stores are then exactly those of a multi-GPU run, on a one-GPU box.
// ---------------------------------------------------------------------------------------------
static const char kHostIdMagic[] = "POVAR-SHM:";
constexpr int kRdvRounds = 64;       // rendezvous per id (one per distinct camera count)
constexpr int kRdvSlotWords = 160;   // >= kMaxPeers * 17 words
struct RdvRegion {
  std::atomic<unsigned int> arrived[kRdvRounds][2];
  unsigned int payload[kRdvRounds][2][kMaxPeers][kRdvSlotWords];
};
struct HostRendezvous {
  RdvRegion* region = nullptr;
  int next_round = 0;
  std::string name;
};
static std::map<std::string, HostRendezvous>& rdv_cache() {
  static std::map<std::string, HostRendezvous> cache;
  return cache;
}
static void release_rendezvous() {
  for (auto& kv : rdv_cache()) {
    if (kv.second.region) munmap(kv.second.region, sizeof(RdvRegion));
    shm_unlink(kv.first.c_str());
  }
  rdv_cache().clear();
}
static bool is_host_id(const uint8_t* id) { return std::memcmp(id, kHostIdMagic, sizeof(kHostIdMagic) - 1) == 0; }

int host_unique_id(uint8_t id[128]) {
  static std::atomic<unsigned int> counter{0};
  std::memset(id, 0, 128);
  const auto now = std::chrono::steady_clock::now().time_since_epoch().count();
  std::snprintf(reinterpret_cast<char*>(id), 128, "%s/povar_%d_%u_%llx", kHostIdMagic, static_cast<int>(getpid()),
                counter.fetch_add(1), static_cast<unsigned long long>(now));
  return POVAR_OK;
}

// comm_cache_mutex() held by the caller
static HostRendezvous* open_rendezvous(const uint8_t* id, std::string* err) {
  const std::string name(reinterpret_cast<const char*>(id) + sizeof(kHostIdMagic) - 1);
  auto& cache = rdv_cache();
  auto it = cache.find(name);
  if (it != cache.end()) return &it->second;
  const int fd = shm_open(name.c_str(), O_CREAT | O_RDWR, 0600);
  if (fd < 0 || ftruncate(fd, sizeof(RdvRegion)) != 0) {   // a new segment reads as zeros; same size on every rank
    if (fd >= 0) close(fd);
    if (err) *err = "host rendezvous: shm_open(" + name + ") failed";
    return nullptr;
  }
  void* p = mmap(nullptr, sizeof(RdvRegion), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (p == MAP_FAILED) {
    if (err) *err = "host rendezvous: mmap failed";
    return nullptr;
  }
  HostRendezvous& r = cache[name];
  r.region = static_cast<RdvRegion*>(p);
  r.name = name;
  return &r;
}

// element-wise sum over the ranks of `words` unsigned ints (what the set-up does with ncclAllReduce otherwise)
static bool rendezvous_sum(HostRendezvous* r, int round, int phase, int rank, int world, unsigned int* data,
                           int words) {
  if (round >= kRdvRounds || words > kRdvSlotWords) return false;
  RdvRegion* g = r->region;
  std::memcpy(g->payload[round][phase][rank], data, sizeof(unsigned int) * words);
  g->arrived[round][phase].fetch_add(1, std::memory_order_acq_rel);
  const auto t0 = std::chrono::steady_clock::now();
  while (g->arrived[round][phase].load(std::memory_order_acquire) < static_cast<unsigned int>(world)) {
    if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(120)) return false;   // a rank never came
    std::this_thread::sleep_for(std::chrono::microseconds(50));
  }
  for (int w = 0; w < words; ++w) data[w] = 0;
  for (int q = 0; q < world; ++q) {
    for (int w = 0; w < words; ++w) data[w] += g->payload[round][phase][q][w];
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
// host-side index construction
// ---------------------------------------------------------------------------------------------
// Static chunking over a few host threads: povar_create walks the observation list a handful of times
// (validation, per-camera counts, sliced-ELL order) and at 5e6 observations a single thread spends more
// on that than the GPU on ten LM iterations.  Results never depend on the thread count.
static int g_host_threads_override = 0;   // povar_debug_sell_layout: tests compare thread counts
void set_host_threads_override(int n) { g_host_threads_override = n; }
static int host_threads(long long work) {
  static const int forced = getenv("POVAR_HOST_THREADS") ? atoi(getenv("POVAR_HOST_THREADS")) : 0;
  if (g_host_threads_override > 0) return g_host_threads_override;
  if (forced > 0) return forced;
  if (work < (1 << 18)) return 1;
  const unsigned hw = std::thread::hardware_concurrency();
  return static_cast<int>(std::min<unsigned>(hw == 0 ? 1 : hw, 16));
}
template <typename F>
static void parallel_chunks(int chunks, F&& body) {   // body(chunk index)
  if (chunks <= 1) {
    body(0);
    return;
  }
  std::vector<std::thread> pool;
  pool.reserve(chunks - 1);
  for (int t = 1; t < chunks; ++t) pool.emplace_back([&body, t] { body(t); });
  body(0);
  for (auto& th : pool) th.join();
}

// Sliced ELL order of the landmarks with 1..32 observations (the landmark half of E0 gives a lane
// to each landmark and walks its observations serially, so the 32 landmarks of a slice should have the
// same degree).  Landmarks are first put in the order of their KEY camera (stable counting sort): the centre
// of the stretch of kSellKeySpan cameras that holds most of the landmark's observations (the first such
// stretch; for a landmark whose cameras span less than that, the middle between its first and its last
// camera).  Neighbouring slices then gather from one stretch of the camera table, as short as the tracks
// allow -- a block of the landmark half stages exactly that stretch in shared memory (kernels_series.cu); with
// the median camera as key the stretch was twice as long on banded scenes.  Inside windows of `window`
// landmarks of that order: stable sort by descending degree, kSellWidth landmarks per slice, slice length =
// largest degree in it.  The order of the observations INSIDE a landmark is untouched (camera ascending), so
// every H_l keeps its bits.
int sell_key(const int* cams, int deg, int span) {
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

int sell_window(int landmarks, int max_window) {
  int w = max_window;
  while (w > 512 && static_cast<long long>(w) * 128 > landmarks) w /= 2;
  return w;
}

void build_sell(const std::vector<int>& lm_ptr, const int* obs_cam, int num_cams, int max_window,
                SellLayout* out, int max_deg) {
  const int L = static_cast<int>(lm_ptr.size()) - 1;
  out->slice_ptr.assign(1, 0);
  out->sell_lm.clear();
  out->slice_lo.clear();
  out->slice_hi.clear();
  out->long_lms.clear();
  out->rows = 0;
  if (L <= 0) return;
  const int T = host_threads(L);
  auto chunk_begin = [&](int t) { return static_cast<int>(static_cast<long long>(L) * t / T); };
  // key camera of every landmark (-1: not in the set), made once
  std::vector<int> keys(static_cast<size_t>(L));
  // landmarks with 1..32 observations by key camera: stable counting sort, one histogram per chunk
  // (chunk t's landmarks of a camera go after those of the chunks before it)
  std::vector<std::vector<int>> hist(T, std::vector<int>(static_cast<size_t>(num_cams), 0));
  std::vector<std::vector<int>> longs(T);
  parallel_chunks(T, [&](int t) {
    std::vector<int>& h = hist[t];
    for (int l = chunk_begin(t); l < chunk_begin(t + 1); ++l) {
      const int deg = lm_ptr[l + 1] - lm_ptr[l];
      keys[l] = -1;
      if (deg > max_deg) {
        longs[t].push_back(l);
      } else if (deg > 0) {
        keys[l] = sell_key(obs_cam + lm_ptr[l], deg, kSellKeySpan);
        h[keys[l]]++;
      }
    }
  });
  for (int t = 0; t < T; ++t) out->long_lms.insert(out->long_lms.end(), longs[t].begin(), longs[t].end());
  int n = 0;
  for (int c = 0; c < num_cams; ++c) {
    for (int t = 0; t < T; ++t) {
      const int cnt = hist[t][c];
      hist[t][c] = n;   // first position of chunk t's landmarks with key camera c
      n += cnt;
    }
  }
  std::vector<int> by_cam(static_cast<size_t>(n));
  parallel_chunks(T, [&](int t) {
    std::vector<int>& h = hist[t];
    for (int l = chunk_begin(t); l < chunk_begin(t + 1); ++l) {
      if (keys[l] >= 0) by_cam[h[keys[l]]++] = l;
    }
  });
  // windows of `window` landmarks of that order, each sorted (stably) by descending degree and cut into
  // slices: the windows are independent, and where a window's slices go is known up front.  A long window
  // means little padding (2.6 % at 4,096 on venice-1778, 16 % at 512) but its slices mix the keys of the whole
  // window; a shard with few landmarks per camera takes a shorter one, so that the cameras a block of the
  // landmark half meets stay one stretch of the table: `max_window`, halved while there are fewer than 128
  // windows, not below 512.
  const int window = sell_window(n, max_window);
  const int num_windows = (n + window - 1) / window;
  const int W = kSellWidth;
  const int slices_per_full = (window + W - 1) / W;
  const int last_cnt = n - (num_windows - 1) * window;
  const int num_slices = num_windows == 0 ? 0 : (num_windows - 1) * slices_per_full + (last_cnt + W - 1) / W;
  out->sell_lm.assign(static_cast<size_t>(num_slices) * W, -1);
  out->slice_lo.assign(static_cast<size_t>(num_slices), 0);
  out->slice_hi.assign(static_cast<size_t>(num_slices), 0);
  std::vector<int> slice_len(static_cast<size_t>(num_slices), 0);
  parallel_chunks(T, [&](int t) {
    int head[34];
    std::vector<int> order(window);
    const int wb = static_cast<int>(static_cast<long long>(num_windows) * t / T);
    const int we = static_cast<int>(static_cast<long long>(num_windows) * (t + 1) / T);
    for (int w = wb; w < we; ++w) {
      const int w0 = w * window, w1 = std::min(n, w0 + window);
      for (int k = 0; k < 34; ++k) head[k] = 0;
      for (int i = w0; i < w1; ++i) head[32 - (lm_ptr[by_cam[i] + 1] - lm_ptr[by_cam[i]]) + 1]++;
      for (int k = 0; k < 33; ++k) head[k + 1] += head[k];
      for (int i = w0; i < w1; ++i) order[head[32 - (lm_ptr[by_cam[i] + 1] - lm_ptr[by_cam[i]])]++] = by_cam[i];
      const int cnt = w1 - w0;
      int sl = w * slices_per_full;
      for (int i = 0; i < cnt; i += W, ++sl) {
        slice_len[sl] = lm_ptr[order[i] + 1] - lm_ptr[order[i]];   // the largest degree of the slice
        int lo = num_cams, hi = -1;
        for (int g = 0; g < W && i + g < cnt; ++g) {
          const int l = order[i + g];
          out->sell_lm[static_cast<size_t>(sl) * W + g] = l;
          lo = std::min(lo, obs_cam[lm_ptr[l]]);            // cameras ascend inside a landmark
          hi = std::max(hi, obs_cam[lm_ptr[l + 1] - 1]);
        }
        out->slice_lo[sl] = lo;
        out->slice_hi[sl] = hi;
      }
    }
  });
  out->slice_ptr.resize(static_cast<size_t>(num_slices) + 1);
  int rows = 0;
  for (int sl = 0; sl < num_slices; ++sl) {
    rows += slice_len[sl];
    out->slice_ptr[sl + 1] = rows;
  }
  out->rows = rows;
}

// ---- plan of the landmark half (LmPlan, povar_internal.h) ----
// Shared memory of one block: [mbarriers][warps x stages x stage_bytes of stream ring][window].
size_t landmark_half_smem(int warps, int stages, int stage_bytes, int win_cams, int rec_bytes) {
  return lm_bar_bytes(warps, stages) + static_cast<size_t>(warps) * stages * stage_bytes +
         static_cast<size_t>(win_cams) * rec_bytes;
}

LmPlanHost plan_landmark_half(const SellLayout& sell, int num_cams, int num_long, int rec_bytes, int stage_bytes,
                              int sms, int max_warps_per_sm, int reserve_bytes) {
  const int S = static_cast<int>(sell.slice_ptr.size()) - 1;
  constexpr size_t kSmemPerSm = 228 * 1024;   // sm_100: 228 KB per SM, 1 KB of it reserved per resident block
  struct Cand {
    int warps, stages, bps;
  };
  // preference: small blocks while the table still fits beside the rings (short launches on small shards,
  // less tail), then one block per SM with the deepest ring, then fewer warps around a larger window
  // (operations with many registers per lane ask for at most 16 warps per SM: 128 registers per thread)
  const Cand cands[] = {{8, 3, 4}, {16, 3, 2}, {32, 3, 1}, {32, 2, 1}, {24, 2, 1},
                        {8, 3, 2}, {16, 3, 1}, {16, 2, 1}};
  LmPlanHost best;
  int best_win = -1;
  for (const Cand& cd : cands) {
    if (cd.warps * cd.bps > max_warps_per_sm) continue;
    LmPlanHost h;
    LmPlan& p = h.p;
    p.warps = cd.warps;
    p.stages = cd.stages;
    p.blocks_per_sm = cd.bps;
    const long long resident = static_cast<long long>(sms) * cd.bps * cd.warps;   // warps of one wave
    p.ranges = static_cast<int>(std::min<long long>(resident, S));
    // ranges of (nearly) equal cost -- rows plus kSliceCost per slice (opening and closing a slice: its landmarks
    // in, its results out, about two rows' worth; blocks of many short slices were 20 % behind those of few
    // long ones with rows alone): range w starts at the first slice at or after cost w * total / ranges
    h.range_slice.assign(static_cast<size_t>(p.ranges) + 1, S);
    {
      const long long total = S > 0 ? sell.slice_ptr[S] + static_cast<long long>(kSliceCost) * S : 0;
      int sl = 0;
      for (int w = 0; w < p.ranges; ++w) {
        const long long target = total * w / p.ranges;
        while (sl < S && sell.slice_ptr[sl] + static_cast<long long>(kSliceCost) * sl < target) ++sl;
        h.range_slice[w] = sl;
      }
    }
    const int slice_blocks = (p.ranges + cd.warps - 1) / cd.warps;
    const int long_blocks = static_cast<int>(std::min<long long>(static_cast<long long>(sms) * cd.bps,
                                                                 (num_long + cd.warps - 1) / cd.warps));
    p.blocks = std::max(slice_blocks, long_blocks);
    // cameras every block meets
    std::vector<int> lo(static_cast<size_t>(std::max(p.blocks, 1)), num_cams), hi(lo.size(), -1);
    int need = 1;
    for (int b = 0; b < slice_blocks; ++b) {
      const int s0 = h.range_slice[static_cast<size_t>(b) * cd.warps];
      const int s1 = h.range_slice[std::min<size_t>(static_cast<size_t>(b + 1) * cd.warps, p.ranges)];
      for (int sl = s0; sl < s1; ++sl) {
        lo[b] = std::min(lo[b], sell.slice_lo[sl]);
        hi[b] = std::max(hi[b], sell.slice_hi[sl]);
      }
      if (hi[b] >= lo[b]) need = std::max(need, hi[b] - lo[b] + 1);
    }
    const size_t budget = kSmemPerSm / cd.bps - 1024 - static_cast<size_t>(reserve_bytes);
    const size_t fixed = landmark_half_smem(cd.warps, cd.stages, stage_bytes, 0, rec_bytes);
    const int fit = budget > fixed ? static_cast<int>((budget - fixed) / rec_bytes) : 0;
    p.win_cams = std::min(num_cams, std::min(need, fit));
    p.covered = fit >= std::min(need, num_cams) ? 1 : 0;
    h.blk_lo.assign(static_cast<size_t>(std::max(p.blocks, 1)), 0);
    for (int b = 0; b < p.blocks; ++b) {
      int start = 0;
      if (hi[b] >= lo[b]) {
        const int span = hi[b] - lo[b] + 1;
        start = span <= p.win_cams ? lo[b] : lo[b] + (span - p.win_cams) / 2;   // not covered: the middle
      }
      h.blk_lo[b] = std::max(0, std::min(start, num_cams - p.win_cams));
    }
    h.smem_bytes = landmark_half_smem(cd.warps, cd.stages, stage_bytes, p.win_cams, rec_bytes);
    if (p.covered) return h;
    if (p.win_cams > best_win) {
      best_win = p.win_cams;
      best = std::move(h);
    }
  }
  return best;
}

int choose_item_len(long long nnz) {
  // enough items to fill every SM with 64 warps a couple of times, at most 256 entries per item (measured on the
  // venice-1778 shape: 128 -> camera half 67.8 us, 256 -> 58.7 us, 512 -> 61.8 us)
  long long len = nnz / (static_cast<long long>(sm_count()) * 64 * 2);
  len = (len + 31) / 32 * 32;
  if (len < 32) len = 32;
  if (len > 256) len = 256;
  return static_cast<int>(len);
}

void build_items(const std::vector<int>& cam_ptr, int item_len, std::vector<int>* item_ptr,
                 std::vector<int>* item_cam, std::vector<int>* cam_item_ptr) {
  const int C = static_cast<int>(cam_ptr.size()) - 1;
  item_ptr->clear();
  item_cam->clear();
  cam_item_ptr->assign(C + 1, 0);
  item_ptr->push_back(0);
  for (int c = 0; c < C; ++c) {
    (*cam_item_ptr)[c] = static_cast<int>(item_cam->size());
    for (int b = cam_ptr[c]; b < cam_ptr[c + 1]; b += item_len) {
      item_cam->push_back(c);
      item_ptr->push_back(std::min(b + item_len, cam_ptr[c + 1]));
    }
  }
  (*cam_item_ptr)[C] = static_cast<int>(item_cam->size());
}


// ---------------------------------------------------------------------------------------------
int Engine::fail(int code, const std::string& what) {
  err_ = what;
  return code;
}

int Engine::check(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return POVAR_OK;
  err_ = std::string(what) + ": " + cudaGetErrorString(e);
  return POVAR_ERR_CUDA;
}

#define PV_CUDA(call)                                   \
  do {                                                  \
    const int rc_ = check((call), #call);               \
    if (rc_ != POVAR_OK) return rc_;                    \
  } while (0)

double Engine::elapsed(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  return ms * 1e-3;
}

// Stream-ordered allocation from the device's default memory pool, which is told to keep what it is
// given back: creating a handle after another one was destroyed costs no cudaMalloc.
template <typename T>
static int dev_alloc(std::vector<void*>& allocs, cudaStream_t stream, T** p, size_t n) {
  void* q = nullptr;
  if (n == 0) n = 1;
  const cudaError_t e = cudaMallocAsync(&q, n * sizeof(T), stream);
  if (e != cudaSuccess) return POVAR_ERR_CUDA;
  cudaMemsetAsync(q, 0, n * sizeof(T), stream);
  allocs.push_back(q);
  *p = static_cast<T*>(q);
  return POVAR_OK;
}

#define PV_ALLOC(ptr, n)                                                        \
  do {                                                                          \
    if (dev_alloc(allocs_, stream_, &(ptr), static_cast<size_t>(n)) != POVAR_OK) \
      return fail(POVAR_ERR_CUDA, std::string("cudaMalloc failed for ") + #ptr); \
  } while (0)

int Engine::create(const povar_problem_desc* desc, const povar_options* opt,
                   const povar_comm_desc* comm, Engine** out, std::string* err) {
  *out = nullptr;
  if (!desc || !opt || desc->num_cams <= 0 || desc->num_lms < 0 || desc->num_obs < 0 ||
      !desc->lm_ptr || !desc->cam_P || (desc->num_obs > 0 && (!desc->obs_cam || !desc->obs_uv))) {
    if (err) *err = "povar_create: invalid problem description";
    return POVAR_ERR_INVALID;
  }
  if (desc->num_obs >= (1LL << 31)) {
    if (err) *err = "povar_create: more than 2^31 observations in one shard";
    return POVAR_ERR_UNSUPPORTED;
  }
  return create_with(opt, comm, out, err, [desc](Engine* e) { return e->upload(desc); });
}

int Engine::create_device(const povar_device_problem_desc* desc, const povar_options* opt,
                          const povar_comm_desc* comm, Engine** out, std::string* err) {
  *out = nullptr;
  const char* bad = nullptr;
  if (!desc || !opt || desc->num_cams <= 0 || desc->num_lms < 0 || desc->num_obs < 0 || !desc->cam_P ||
      (desc->num_obs > 0 && (!desc->obs_cam || !desc->obs_lm || !desc->obs_uv))) {
    bad = "povar_create_device: invalid problem description";
  } else if (desc->lm_begin < 0 || desc->lm_begin > desc->lm_end || desc->lm_end > desc->num_lms) {
    bad = "povar_create_device: landmark range [lm_begin, lm_end) is not inside [0, num_lms]";
  }
  if (bad) {
    if (err) *err = bad;
    return POVAR_ERR_INVALID;
  }
  if (desc->num_obs >= (1LL << 31)) {
    if (err) *err = "povar_create_device: 2^31 or more observations";
    return POVAR_ERR_UNSUPPORTED;
  }
  return create_with(opt, comm, out, err, [desc](Engine* e) { return e->upload_device(desc); });
}

int Engine::create_with(const povar_options* opt, const povar_comm_desc* comm, Engine** out, std::string* err,
                        const std::function<int(Engine*)>& upload) {
  const auto t_create = std::chrono::steady_clock::now();
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    if (err) *err = "povar_create: no CUDA device (this library has no CPU fallback)";
    return POVAR_ERR_NO_DEVICE;
  }
  Engine* e = new Engine();
  e->opt_ = *opt;
  e->rank_ = comm ? comm->rank : 0;
  e->world_ = comm ? comm->world_size : 1;
  e->device_ = comm ? comm->device : 0;
  if (e->device_ < 0 || e->device_ >= ndev) {
    if (err) *err = "povar_create: device ordinal out of range";
    delete e;
    return POVAR_ERR_INVALID;
  }
  int rc = e->check(cudaSetDevice(e->device_), "cudaSetDevice");
  if (rc == POVAR_OK) {
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, e->device_) == cudaSuccess) {
      unsigned long long keep = ~0ULL;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  HostKit kit;
  if (rc == POVAR_OK && take_kit(e->device_, &kit)) {
    e->stream_ = kit.stream;
    for (int i = 0; i < 8; ++i) e->ev_[i] = kit.ev[i];
    e->host_out_ = kit.pinned;
  } else {
    if (rc == POVAR_OK) rc = e->check(cudaStreamCreateWithFlags(&e->stream_, cudaStreamNonBlocking), "cudaStreamCreate");
    for (int i = 0; i < 8 && rc == POVAR_OK; ++i) rc = e->check(cudaEventCreate(&e->ev_[i]), "cudaEventCreate");
    if (rc == POVAR_OK) rc = e->check(cudaHostAlloc(reinterpret_cast<void**>(&e->host_out_), 256, cudaHostAllocDefault), "cudaHostAlloc");
  }
  if (rc == POVAR_OK && e->world_ > 1 && opt->solver_type_step_1 == POVAR_CHOLESKY) {
    // the direct solver's reduced camera system is not sharded (solver/linearizor_sc.cpp:121-128 is serial too)
    rc = e->fail(POVAR_ERR_UNSUPPORTED, "CHOLESKY is single-GPU: create the handle without a communicator");
  }
  if (rc == POVAR_OK && e->world_ > 1 && is_host_id(comm->nccl_id)) {
    // host rendezvous (povar_comm_host_id): no NCCL communicator at all, every reduction over the peer buffers
    e->comm_key_ = comm_key(*comm);
    std::lock_guard<std::mutex> lock(comm_cache_mutex());
    std::string herr;
    e->rdv_ = open_rendezvous(comm->nccl_id, &herr);
    if (!e->rdv_) rc = e->fail(POVAR_ERR_NCCL, herr);
  } else if (rc == POVAR_OK && e->world_ > 1) {
    std::string nerr;
    e->nccl_ = load_nccl(&nerr);
    if (!e->nccl_) {
      rc = e->fail(POVAR_ERR_NCCL, nerr);
    } else {
      // one communicator per (id, rank) and process: the step-1 and step-2 linearizors of a solve, and
      // every later handle made with the same descriptor, share it (ncclCommInitRank accepts an id once)
      const std::string key = comm_key(*comm);
      e->comm_key_ = key;
      std::lock_guard<std::mutex> lock(comm_cache_mutex());
      auto& cache = comm_cache();
      auto it = cache.find(key);
      if (it != cache.end()) {
        e->nccl_comm_ = it->second;
      } else {
        Id128 id;
        std::memcpy(id.bytes, comm->nccl_id, 128);
        const int nrc = e->nccl_->CommInitRank(&e->nccl_comm_, e->world_, id, e->rank_);
        if (nrc != 0) {
          e->nccl_comm_ = nullptr;
          rc = e->fail(POVAR_ERR_NCCL, "ncclCommInitRank failed");
        } else {
          cache[key] = e->nccl_comm_;
        }
      }
    }
  }
  if (getenv("POVAR_TRACE_CREATE") != nullptr) {
    std::fprintf(stderr, "povar_create: %-28s %8.3f ms\n", "device, stream, scratch",
                 std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_create).count());
  }
  if (rc == POVAR_OK) rc = upload(e);
  if (rc == POVAR_OK) rc = e->setup_peer_exchange();
  if (rc != POVAR_OK) {
    if (err) *err = e->err_;
    delete e;
    return rc;
  }
  *out = e;
  return POVAR_OK;
}

Engine::~Engine() {
  static const bool trace = getenv("POVAR_TRACE_CREATE") != nullptr;   // phase times of povar_destroy on stderr
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "povar_destroy: %-27s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  if (device_ >= 0) cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  lap("synchronize");
  // the communicator belongs to the process-wide cache (povar_comm_finalize releases it)
  for (void*& g : series_graph_) {
    if (g) cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(g));
    g = nullptr;
  }
  if (solve_graph_) cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(solve_graph_));
  solve_graph_ = nullptr;
  lap("graphs");
  if (peer_owned_ && peer_) {
    peer_->release();
    delete peer_;
  }
  for (void* p : allocs_) cudaFreeAsync(p, stream_);
  lap("free (enqueue)");
  bool clean = stream_ != nullptr && host_out_ != nullptr && cudaStreamSynchronize(stream_) == cudaSuccess;
  for (auto& ev : ev_) clean = clean && ev != nullptr;
  lap("free (synchronize)");
  if (join_ev_) cudaEventDestroy(join_ev_);
  if (clean) {
    // stream, events and scratch wait for the next handle on this device (HostKit)
    HostKit kit;
    kit.device = device_;
    kit.stream = stream_;
    for (int i = 0; i < 8; ++i) kit.ev[i] = ev_[i];
    kit.pinned = host_out_;
    give_kit(kit);
  } else {
    if (host_out_) cudaFreeHost(host_out_);
    for (auto& ev : ev_) {
      if (ev) cudaEventDestroy(ev);
    }
    if (stream_) cudaStreamDestroy(stream_);
  }
  lap("stream, events, scratch");
}

// phase times of povar_create on stderr (POVAR_TRACE_CREATE)
namespace {
struct CreateLap {
  bool on = getenv("POVAR_TRACE_CREATE") != nullptr;
  std::chrono::steady_clock::time_point prev = std::chrono::steady_clock::now();
  void operator()(const char* what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "povar_create: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - prev).count());
    prev = now;
  }
};
}  // namespace

// Front half of the host route: the landmark table (one pass over lm_ptr) and the uploads of lm_ptr and the camera
// indices; everything per observation -- the check of the camera indices and the per-camera counts included -- is
// made on the device (kernels_index.cu)
int Engine::upload(const povar_problem_desc* desc) {
  const int C = desc->num_cams, L = desc->num_lms;
  const int nnz = static_cast<int>(desc->num_obs);
  C_ = C;
  L_ = L;
  nnz_ = nnz;
  CreateLap lap;
  std::vector<int> lm_ptr(L + 1);
  std::vector<int> long_lms;   // landmarks with more than sell_max_deg observations
  int sell_n = 0;              // landmarks with 1..sell_max_deg observations
  const int sell_max_deg = sell_max_degree(nnz, sm_count());
  d_.ix.sell_max_deg = sell_max_deg;
  if (desc->lm_ptr[0] != 0 || desc->lm_ptr[L] != nnz) return fail(POVAR_ERR_INVALID, "lm_ptr does not span the observations");
  // (one thread: a million trivial iterations cost about a millisecond, less than starting threads does on a
  // virtualised host -- the threaded version of this pass took 6 to 11 ms on the bench boxes)
  for (int l = 0; l < L; ++l) {
    const int64_t b = desc->lm_ptr[l], e = desc->lm_ptr[l + 1];
    if (e < b || b < 0 || e > nnz) return fail(POVAR_ERR_INVALID, "lm_ptr is not monotone");
    lm_ptr[l] = static_cast<int>(b);
    if (e - b > sell_max_deg) long_lms.push_back(l);
    else if (e > b) ++sell_n;
  }
  lm_ptr[L] = nnz;
  lap("landmark table");
  // the observation list starts travelling now: camera indices first (the device checks and counts them while
  // the image coordinates follow, build_index), and the copies run while the host derives the work items
  DeviceIndex& ix = d_.ix;
  PV_ALLOC(ix.lm_ptr, L + 1);
  PV_ALLOC(ix.obs_cam, nnz);
  PV_ALLOC(ix.obs_lm, nnz);
  PV_ALLOC(ix.obs_uv, nnz);
  PV_CUDA(cudaMemcpyAsync(ix.lm_ptr, lm_ptr.data(), sizeof(int) * (L + 1), cudaMemcpyHostToDevice, stream_));
  if (nnz > 0) {
    PV_CUDA(cudaMemcpyAsync(ix.obs_cam, desc->obs_cam, sizeof(int) * static_cast<size_t>(nnz), cudaMemcpyHostToDevice,
                            stream_));
  }
  ix.num_long = static_cast<int>(long_lms.size());
  return build_index(sell_n, long_lms.data(), desc->obs_uv, desc->cam_P);
}

int Engine::check_device_ptr(const void* p, const char* what) {
  cudaPointerAttributes a{};
  const cudaError_t e = cudaPointerGetAttributes(&a, p);
  cudaGetLastError();   // not sticky: a failed query must not fail the next call
  if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != device_) {
    return fail(POVAR_ERR_INVALID, std::string(what) + " is not device memory of device " + std::to_string(device_));
  }
  return POVAR_OK;
}

int Engine::wait_for(cudaStream_t waiter, cudaStream_t producer) {
  if (!join_ev_) PV_CUDA(cudaEventCreateWithFlags(&join_ev_, cudaEventDisableTiming));
  const cudaError_t e = cudaEventRecord(join_ev_, producer);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(POVAR_ERR_INVALID, std::string("stream of the caller: ") + cudaGetErrorString(e));
  }
  PV_CUDA(cudaStreamWaitEvent(waiter, join_ev_, 0));
  return POVAR_OK;
}

// Front half of the device route: the canonical order of the caller's list on the device (kernels_index.cu), the
// shard's entries gathered straight into the landmark-major arrays, the landmark table made there too; the host
// reads the shard's observation count as soon as the keys are counted (the sort runs meanwhile) and the landmark
// table once it is made.
int Engine::upload_device(const povar_device_problem_desc* desc) {
  const int C = desc->num_cams, L = desc->lm_end - desc->lm_begin;
  const int n = static_cast<int>(desc->num_obs);
  PV_CUDA(cudaSetDevice(device_));
  for (const auto& pw : {std::make_pair(static_cast<const void*>(desc->cam_P), "cam_P"),
                         std::make_pair(static_cast<const void*>(desc->obs_cam), "obs_cam"),
                         std::make_pair(static_cast<const void*>(desc->obs_lm), "obs_lm"),
                         std::make_pair(static_cast<const void*>(desc->obs_uv), "obs_uv")}) {
    if (n == 0 && pw.first != desc->cam_P) continue;
    const int rc = check_device_ptr(pw.first, pw.second);
    if (rc != POVAR_OK) return rc;
  }
  {
    const int rc = wait_for(stream_, static_cast<cudaStream_t>(desc->stream));
    if (rc != POVAR_OK) return rc;
  }
  CreateLap lap;
  C_ = C;
  L_ = L;
  // scratch, returned to the pool when this function returns
  const size_t keep = allocs_.size();
  struct Scratch {
    Engine* e;
    std::vector<void*> mine;
    ~Scratch() {
      for (void* p : mine) {
        cudaFreeAsync(p, e->stream_);
        e->allocs_.erase(std::find(e->allocs_.begin(), e->allocs_.end(), p));
      }
    }
  } scratch{this, {}};
  unsigned long long *keys_a = nullptr, *keys_b = nullptr;
  int *pos_a = nullptr, *pos_b = nullptr, *info = nullptr, *long_tmp = nullptr;
  unsigned char* is_long = nullptr;
  char* temp = nullptr;
  const int end_bit = order_end_bit(C, desc->num_lms);
  const size_t temp_bytes = device_order_temp_bytes(n, L, end_bit);
  PV_ALLOC(keys_a, n);
  PV_ALLOC(keys_b, n);
  PV_ALLOC(pos_a, n);
  PV_ALLOC(pos_b, n);
  PV_ALLOC(info, kOrderInfo);
  PV_ALLOC(long_tmp, L);
  PV_ALLOC(is_long, L);
  PV_ALLOC(temp, temp_bytes);
  scratch.mine.assign(allocs_.begin() + keep, allocs_.end());
  int* counts = reinterpret_cast<int*>(host_out_);   // pinned: the read-backs below overlap the device work
  PV_CUDA(device_order_keys(n, C, desc->num_lms, desc->lm_begin, desc->lm_end, desc->obs_cam, desc->obs_lm, keys_a,
                            pos_a, info, lc()));
  PV_CUDA(cudaMemcpyAsync(counts, info, sizeof(int) * kOrderInfo, cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaEventRecord(join_ev_, stream_));
  PV_CUDA(device_order_sort(n, end_bit, keys_a, keys_b, pos_a, pos_b, temp, temp_bytes, lc()));
  PV_CUDA(cudaEventSynchronize(join_ev_));
  if (counts[kOrderFlags] & 1) return fail(POVAR_ERR_INVALID, "povar_create_device: camera or landmark index out of range");
  const int nnz = counts[kOrderCount];
  nnz_ = nnz;
  lap("order keys + counts (device)");
  DeviceIndex& ix = d_.ix;
  PV_ALLOC(ix.lm_ptr, L + 1);
  PV_ALLOC(ix.obs_cam, nnz);
  PV_ALLOC(ix.obs_lm, nnz);
  PV_ALLOC(ix.obs_uv, nnz);
  ix.L = L;
  PV_CUDA(device_order_place(n, C, desc->lm_begin, sm_count(), keys_b, pos_b, desc->obs_uv, info, ix, is_long, long_tmp,
                             temp, temp_bytes, lc()));
  PV_CUDA(cudaMemcpyAsync(counts, info, sizeof(int) * kOrderInfo, cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  if (counts[kOrderFlags] & 2) return fail(POVAR_ERR_INVALID, "povar_create_device: duplicate (camera, landmark) pair");
  ix.num_long = counts[kOrderLong];
  d_.ix.sell_max_deg = sell_max_degree(nnz, sm_count());
  lap("canonical order + landmark table (device)");
  return build_index(counts[kOrderSell], long_tmp, nullptr, desc->cam_P);
}

// Back half, shared by both routes: from the landmark-major list in ix (lm_ptr, obs_cam; obs_uv unless host_uv
// still has to be uploaded) and the landmark table (sell_n, ix.num_long long landmarks at long_lms) to the whole
// index and the state.  long_lms and cam_P may be host or device memory.
int Engine::build_index(int sell_n, const int* long_lms, const double* host_uv, const double* cam_P) {
  const int C = C_, L = L_;
  const int nnz = static_cast<int>(nnz_);
  const int sell_max_deg = d_.ix.sell_max_deg;
  CreateLap lap;
  std::vector<int> cam_ptr(C + 1, 0);
  SellLayout sell;    // sliced-ELL order: the slices from the device
#define PV_UP(dst, src, n) PV_CUDA(cudaMemcpyAsync((dst), (src), (n), cudaMemcpyHostToDevice, stream_))
  DeviceIndex& ix = d_.ix;
  {
    int* d_count = nullptr;
    const size_t keep = allocs_.size();
    PV_ALLOC(d_count, static_cast<size_t>(C) + 1);
    PV_CUDA(validate_obs(L, C, sm_count(), ix.lm_ptr, ix.obs_cam, d_count, lc()));
    std::vector<int> count(static_cast<size_t>(C) + 1);
    PV_CUDA(cudaMemcpyAsync(count.data(), d_count, sizeof(int) * count.size(), cudaMemcpyDeviceToHost, stream_));
    cudaEvent_t counted = nullptr;
    PV_CUDA(cudaEventCreateWithFlags(&counted, cudaEventDisableTiming));
    cudaEventRecord(counted, stream_);
    if (host_uv && nnz > 0) {
      const cudaError_t ce = cudaMemcpyAsync(ix.obs_uv, host_uv, sizeof(double) * 2 * static_cast<size_t>(nnz),
                                             cudaMemcpyHostToDevice, stream_);
      if (ce != cudaSuccess) {
        cudaEventDestroy(counted);
        return fail(POVAR_ERR_CUDA, cudaGetErrorString(ce));
      }
    }
    const cudaError_t we = cudaEventSynchronize(counted);
    cudaEventDestroy(counted);
    if (we != cudaSuccess) return fail(POVAR_ERR_CUDA, cudaGetErrorString(we));
    while (allocs_.size() > keep) {
      cudaFreeAsync(allocs_.back(), stream_);
      allocs_.pop_back();
    }
    if (count[C] & 1) return fail(POVAR_ERR_INVALID, "camera index out of range");
    if (count[C] & 2) return fail(POVAR_ERR_INVALID, "observations of a landmark must have strictly ascending camera indices");
    for (int c = 0; c < C; ++c) cam_ptr[c + 1] = cam_ptr[c] + count[c];
    if (cam_ptr[C] != nnz) return fail(POVAR_ERR_INVALID, "camera counts do not add up to the observations");
  }
  lap("camera check + counts (device)");
  // the sliced-ELL order of the landmarks (rule: build_sell above, which the CPU tests check) on the device, as soon
  // as the copies above have landed; the host derives the camera work items meanwhile
  const int sell_slices = (sell_n + kSellWidth - 1) / kSellWidth;
  const int window = sell_window(sell_n, kSellWindow);
  std::vector<int> slice_len(static_cast<size_t>(sell_slices)), slice_lo(slice_len.size()), slice_hi(slice_len.size());
  PV_ALLOC(ix.sell_lm, static_cast<size_t>(sell_slices) * kSellWidth);
  if (sell_n > 0) {
    int *keys_a = nullptr, *keys_b = nullptr, *ids_a = nullptr, *ids_b = nullptr, *d_len = nullptr, *d_lo = nullptr,
        *d_hi = nullptr;
    char* sort_temp = nullptr;
    const size_t temp_bytes = sell_sort_temp_bytes(L, C, sell_n, window);
    const size_t keep = allocs_.size();
    PV_ALLOC(keys_a, L);
    PV_ALLOC(keys_b, L);
    PV_ALLOC(ids_a, L);
    PV_ALLOC(ids_b, L);
    PV_ALLOC(d_len, sell_slices);
    PV_ALLOC(d_lo, sell_slices);
    PV_ALLOC(d_hi, sell_slices);
    PV_ALLOC(sort_temp, temp_bytes);
    PV_CUDA(build_device_sell(L, C, sell_n, window, sell_max_deg, ix.lm_ptr, ix.obs_cam, keys_a, keys_b, ids_a, ids_b,
                              sort_temp, temp_bytes, ix.sell_lm, d_len, d_lo, d_hi, lc()));
    PV_CUDA(cudaMemcpyAsync(slice_len.data(), d_len, sizeof(int) * slice_len.size(), cudaMemcpyDeviceToHost, stream_));
    PV_CUDA(cudaMemcpyAsync(slice_lo.data(), d_lo, sizeof(int) * slice_lo.size(), cudaMemcpyDeviceToHost, stream_));
    PV_CUDA(cudaMemcpyAsync(slice_hi.data(), d_hi, sizeof(int) * slice_hi.size(), cudaMemcpyDeviceToHost, stream_));
    while (allocs_.size() > keep) {
      cudaFreeAsync(allocs_.back(), stream_);
      allocs_.pop_back();
    }
  }
  std::vector<int> item_ptr, item_cam, cam_item_ptr;
  build_items(cam_ptr, choose_item_len(nnz), &item_ptr, &item_cam, &cam_item_ptr);
  lap("items (+ device: sliced-ELL order)");
  PV_CUDA(cudaStreamSynchronize(stream_));
  sell.slice_ptr.assign(static_cast<size_t>(sell_slices) + 1, 0);
  for (int sl = 0; sl < sell_slices; ++sl) sell.slice_ptr[sl + 1] = sell.slice_ptr[sl] + slice_len[sl];
  sell.rows = sell.slice_ptr[sell_slices];
  sell.slice_lo.swap(slice_lo);
  sell.slice_hi.swap(slice_hi);
  lap("wait for the order");
  if (static_cast<long long>(sell.rows) * kSellWidth >= (1LL << 31)) {
    return fail(POVAR_ERR_UNSUPPORTED, "sliced-ELL layout exceeds 2^31 slots in one shard");
  }

  ix.C = C;
  ix.L = L;
  ix.nnz = nnz;
  ix.num_items = static_cast<int>(item_cam.size());
  ix.num_slices = static_cast<int>(sell.slice_ptr.size()) - 1;
  ix.sell_slots = static_cast<long long>(kSellWidth) * sell.rows;
  const size_t slots = static_cast<size_t>(ix.sell_slots);
  PV_ALLOC(ix.cam_ptr, C + 1);
  PV_ALLOC(ix.csc_lm, nnz);
  PV_ALLOC(ix.csc_uv, nnz);
  PV_ALLOC(ix.item_cam, item_cam.size());
  PV_ALLOC(ix.item_ptr, item_ptr.size());
  PV_ALLOC(ix.cam_item_ptr, C + 1);
  PV_ALLOC(ix.slice_ptr, sell.slice_ptr.size());
  PV_ALLOC(ix.sell_cam, slots);
  PV_ALLOC(ix.sell_uv, slots);
  PV_ALLOC(ix.sell_cam_e0, slots);
  PV_ALLOC(ix.sell_uv_e0, slots);
  PV_ALLOC(ix.sell_row_e0, slots + 32);
  PV_ALLOC(ix.obs_slot, nnz);
  PV_ALLOC(ix.long_lm, ix.num_long);
  if (nnz > 0) PV_UP(ix.item_cam, item_cam.data(), sizeof(int) * item_cam.size());
  PV_UP(ix.slice_ptr, sell.slice_ptr.data(), sizeof(int) * sell.slice_ptr.size());
  // landmark half: ranges of slices per warp, windows of cameras per block (kernels_series.cu), per model
  LmPlanHost lm_plans[5];   // alive until the synchronisation at the end of this function
  for (int m = 0; m < 5; ++m) {
    // [0..2] landmark half of a term (pOSE, joint, pOSE + HUBER); [3], [4] once-per-trial walks: more registers
    // per lane (16 warps per SM), no long landmarks, 256 bytes of static shared memory for the block sums
    const int rec_bytes = 8 * (m == 1 ? kCamRecJoint : m == 3 ? kCamTab1 : m == 4 ? kCamTab2 : kCamRecPose);
    const int stage_bytes = (m == 1 || m == 2) ? kStageWide : (m == 3 ? kStageLin : kStagePose);
    lm_plans[m] = m < 3 ? plan_landmark_half(sell, C, ix.num_long, rec_bytes, stage_bytes, sm_count(), 32, 0)
                        : plan_landmark_half(sell, C, 0, rec_bytes, stage_bytes, sm_count(), 16, 256);
    const LmPlanHost& h = lm_plans[m];
    d_.plan[m] = h.p;
    PV_ALLOC(d_.plan[m].range_slice, h.range_slice.size());
    PV_ALLOC(d_.plan[m].blk_lo, h.blk_lo.size());
    PV_UP(d_.plan[m].range_slice, h.range_slice.data(), sizeof(int) * h.range_slice.size());
    PV_UP(d_.plan[m].blk_lo, h.blk_lo.data(), sizeof(int) * h.blk_lo.size());
  }
  if (ix.num_long > 0) {
    PV_CUDA(cudaMemcpyAsync(ix.long_lm, long_lms, sizeof(int) * static_cast<size_t>(ix.num_long), cudaMemcpyDefault,
                            stream_));
  }
  PV_UP(ix.cam_ptr, cam_ptr.data(), sizeof(int) * (C + 1));
  PV_UP(ix.item_ptr, item_ptr.data(), sizeof(int) * item_ptr.size());
  PV_UP(ix.cam_item_ptr, cam_item_ptr.data(), sizeof(int) * (C + 1));
  {
    // scratch of the device-side build, returned to the pool right after
    int *iota = nullptr, *keys_out = nullptr, *perm = nullptr, *lm_slot = nullptr;
    char* sort_temp = nullptr;
    const size_t temp_bytes = index_sort_temp_bytes(nnz, C);
    const size_t keep = allocs_.size();
    PV_ALLOC(iota, nnz);
    PV_ALLOC(keys_out, nnz);
    PV_ALLOC(perm, nnz);
    PV_ALLOC(lm_slot, L);
    PV_ALLOC(sort_temp, temp_bytes);
    PV_CUDA(build_device_index(ix, iota, keys_out, perm, lm_slot, sort_temp, temp_bytes, lc()));
    while (allocs_.size() > keep) {
      cudaFreeAsync(allocs_.back(), stream_);
      allocs_.pop_back();
    }
  }
  // ---- state and work arrays
  const size_t C12 = static_cast<size_t>(C) * 12, C144 = static_cast<size_t>(C) * 144;
  PV_ALLOC(d_.P, C12);
  PV_ALLOC(d_.P_bak, C12);
  PV_ALLOC(P_prev_, C12);
  PV_ALLOC(d_.X, static_cast<size_t>(L) * 4);
  PV_ALLOC(d_.X_bak, static_cast<size_t>(L) * 4);
  PV_ALLOC(d_.pose_scale, C12);
  PV_ALLOC(d_.lm_scale, static_cast<size_t>(L) * 4);
  PV_ALLOC(d_.lm_hraw, static_cast<size_t>(L) * 10);
  PV_ALLOC(d_.lm_graw, static_cast<size_t>(L) * 4);
  PV_ALLOC(d_.hll_inv, static_cast<size_t>(L) * 6);
  PV_ALLOC(d_.lm_rec, static_cast<size_t>(L) * kLmRec);
  PV_ALLOC(d_.lm_fold, static_cast<size_t>(L) * 10);
  PV_ALLOC(d_.cam_rec, static_cast<size_t>(C) * kCamRecStride);
  PV_ALLOC(d_.cam_tab, static_cast<size_t>(C) * kCamTab2);
  {
    const size_t plane = static_cast<size_t>(ix.num_slices) * kSellWidth;
    PV_ALLOC(d_.sell_hraw, plane * 10);
    PV_ALLOC(d_.sell_graw, plane * 4);
    PV_ALLOC(d_.sell_scale, plane * 4);
    PV_ALLOC(d_.sell_hinv, plane * 6);
    PV_ALLOC(d_.sell_step, plane * 4);
  }
  PV_ALLOC(d_.sell_x, static_cast<size_t>(ix.num_slices) * 4 * kSellWidth);
  PV_ALLOC(d_.sell_fold, static_cast<size_t>(ix.num_slices) * 10 * kSellWidth);
  PV_ALLOC(d_.kron, static_cast<size_t>(C) * kKron);
  PV_ALLOC(d_.kron2, static_cast<size_t>(C) * kKron);
  PV_ALLOC(d_.item_kron, static_cast<size_t>(ix.num_items) * kKron);
  PV_ALLOC(d_.item_part, static_cast<size_t>(ix.num_items) * 12);
  PV_ALLOC(d_.cam_raw, C12);
  PV_ALLOC(d_.Bmat, C144);
  PV_ALLOC(d_.Binv, C144);
  PV_ALLOC(d_.Mprec, C144);
  PV_ALLOC(d_.b, C12);
  PV_ALLOC(d_.vec_tmp, C12);
  PV_ALLOC(d_.vec_acc, C12);
  PV_ALLOC(d_.vec_y, C12);
  PV_ALLOC(d_.vec_x, C12);
  PV_ALLOC(d_.cg_r, C12);
  PV_ALLOC(d_.cg_p, C12);
  PV_ALLOC(d_.cg_z, C12);
  PV_ALLOC(d_.cg_q, C12);
  PV_ALLOC(d_.cg_x, C12);
  PV_ALLOC(d_.norm_part, static_cast<size_t>(C) * 4);
  PV_ALLOC(d_.cost_part, static_cast<size_t>(cost_blocks(d_)) * 8);
  PV_ALLOC(d_.cost_out, 1);
  PV_ALLOC(d_.scalar_part, static_cast<size_t>(scalar_blocks(d_)) + 8);
  PV_ALLOC(d_.trial_out, 16);
  PV_ALLOC(d_.flags, 4);
  PV_ALLOC(d_.ctl, 1);
  PV_ALLOC(d_.cg, 1);
  PV_CUDA(cudaMemcpyAsync(d_.P, cam_P, sizeof(double) * C12, cudaMemcpyDefault, stream_));
#undef PV_UP
  lap("allocate + enqueue uploads");
  // the host tables above live on this stack frame
  PV_CUDA(cudaStreamSynchronize(stream_));
  lap("device index build + sync");
  return POVAR_OK;
}

// Peer-memory exchange for the per-term camera sums: one cudaMalloc per rank (receive buffer + exchange
// counter), exported with CUDA IPC, handles swapped through the NCCL communicator (or the host rendezvous),
// mapped with peer access over NVLink.  Every rank takes the same decisions (the inputs of each decision are
// all-reduced), because a rank that fell back to NCCL alone would deadlock the others.  The mapping is made
// once per (communicator, camera count) and process -- like the communicator itself -- and shared by later
// handles: ranks create their handles in the same order, so cache hits are symmetric.
//
// The number of an exchange -- its tag and the parity of the slots it uses -- is a DEVICE-side counter that
// lives next to the receive buffer and is advanced by the kernel that performed the exchange (k_term16,
// k_peer_allreduce): terms that are enqueued but skipped after the series converged do not count, every rank
// performs the same sequence of exchanges, and the count survives the handle (the slots keep their tags).
static constexpr size_t kPeerCounterBytes = 256;
int Engine::sum_setup_words(unsigned int* host, int words, int phase, int round) {
  if (rdv_) {
    if (!rendezvous_sum(rdv_, round, phase, rank_, world_, host, words)) {
      return fail(POVAR_ERR_NCCL, "host rendezvous: a rank did not arrive (peer exchange setup)");
    }
    return POVAR_OK;
  }
  unsigned int* dev = nullptr;
  PV_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dev), sizeof(unsigned int) * words, stream_));
  PV_CUDA(cudaMemcpyAsync(dev, host, sizeof(unsigned int) * words, cudaMemcpyHostToDevice, stream_));
  if (nccl_->AllReduce(dev, dev, words, /*ncclUint32*/ 3, /*ncclSum*/ 0, nccl_comm_, stream_) != 0) {
    return fail(POVAR_ERR_NCCL, "ncclAllReduce failed (peer exchange setup)");
  }
  PV_CUDA(cudaMemcpyAsync(host, dev, sizeof(unsigned int) * words, cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  PV_CUDA(cudaFreeAsync(dev, stream_));
  return POVAR_OK;
}

int Engine::setup_peer_exchange() {
  const char* env = getenv("POVAR_PEER_EXCHANGE");
  const bool forbid = env != nullptr && std::strcmp(env, "0") == 0;
  if (forbid && rdv_) return fail(POVAR_ERR_NCCL, "the host rendezvous needs the peer exchange (POVAR_PEER_EXCHANGE=0 set)");
  if (forbid) return POVAR_OK;
  if (world_ > kMaxPeers || C_ <= 0) {
    if (rdv_) return fail(POVAR_ERR_UNSUPPORTED, "host rendezvous: more ranks than the peer exchange supports");
    return POVAR_OK;
  }
  if (world_ == 1) {
    // POVAR_PEER_EXCHANGE=self: a single GPU runs the exchange protocol against its own buffer (isolates the
    // protocol's cost from the NVLink hop)
    if (env == nullptr || std::strcmp(env, "self") != 0) return POVAR_OK;
    PeerShared* ps = new PeerShared();
    const size_t bytes = 16 * 2 * static_cast<size_t>(C_) * 12;
    if (cudaMalloc(&ps->mem, bytes + kPeerCounterBytes) != cudaSuccess ||
        cudaMemset(ps->mem, 0, bytes + kPeerCounterBytes) != cudaSuccess) {
      delete ps;
      return fail(POVAR_ERR_CUDA, "cudaMalloc failed for the self exchange buffer");
    }
    ps->px.recv[0] = static_cast<double*>(ps->mem);
    ps->px.rank = 0;
    ps->px.world = 1;
    ps->px.stride = static_cast<unsigned long long>(C_) * 12;
    ps->px.count = reinterpret_cast<unsigned int*>(static_cast<char*>(ps->mem) + bytes);
    ps->ok = true;
    peer_ = ps;
    peer_owned_ = true;
    peer_ok_ = true;
    return POVAR_OK;
  }
  if (env != nullptr && std::strcmp(env, "self") == 0) env = nullptr;
  const bool must = env != nullptr || rdv_ != nullptr;   // asked for explicitly, or no NCCL to fall back to
  const std::string key = comm_key_ + ":" + std::to_string(C_);
  std::lock_guard<std::mutex> lock(comm_cache_mutex());
  auto& cache = peer_cache();
  auto it = cache.find(key);
  if (it != cache.end()) {
    peer_ = it->second;
    peer_ok_ = peer_->ok;
    if (!peer_ok_ && must) {
      return fail(POVAR_ERR_NCCL, "peer exchange requested but CUDA IPC / peer access is unavailable");
    }
    return POVAR_OK;
  }
  PeerShared* ps = new PeerShared();
  cache[key] = ps;
  peer_ = ps;
  const int round = rdv_ ? rdv_->next_round++ : 0;
  // 16-byte tagged slots, [2 parities][world][60*C]; zero = "exchange 0", never waited for
  const size_t stride = static_cast<size_t>(C_) * kKron;
  const size_t recv_pad = 16 * 2 * static_cast<size_t>(world_) * stride;
  unsigned int ok = 1;
  cudaIpcMemHandle_t mine{};
  if (cudaMalloc(&ps->mem, recv_pad + kPeerCounterBytes) != cudaSuccess) {
    ps->mem = nullptr;
    ok = 0;
  }
  if (ok && cudaMemsetAsync(ps->mem, 0, recv_pad + kPeerCounterBytes, stream_) != cudaSuccess) ok = 0;
  if (ok && cudaStreamSynchronize(stream_) != cudaSuccess) ok = 0;   // zeroed before any peer can store into it
  if (ok && cudaIpcGetMemHandle(&mine, ps->mem) != cudaSuccess) ok = 0;
  cudaGetLastError();
  // swap: [world][16 words of handle] + [world] ok flags, summed as uint32 (everything else is zero)
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  const int words = world_ * 17;
  std::vector<unsigned int> host(words, 0u);
  if (ok) std::memcpy(host.data() + 16 * rank_, &mine, 64);
  host[16 * world_ + rank_] = ok;
  {
    const int rc = sum_setup_words(host.data(), words, 0, round);
    if (rc != POVAR_OK) return rc;
  }
  unsigned int all_ok = 1;
  for (int r = 0; r < world_; ++r) all_ok &= host[16 * world_ + r];
  std::vector<void*> base(world_, nullptr);
  if (all_ok) {
    for (int r = 0; r < world_; ++r) {
      if (r == rank_) {
        base[r] = ps->mem;
        continue;
      }
      cudaIpcMemHandle_t h;
      std::memcpy(&h, host.data() + 16 * r, 64);
      void* ptr = nullptr;
      if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        all_ok = 0;
        break;
      }
      ps->opened.push_back(ptr);
      base[r] = ptr;
    }
  }
  // second round: did everybody map everybody?
  unsigned int mapped = all_ok;
  {
    const int rc = sum_setup_words(&mapped, 1, 1, round);
    if (rc != POVAR_OK) return rc;
  }
  if (mapped != static_cast<unsigned int>(world_)) {
    ps->release();   // the entry stays, marked unavailable: later handles do not try again
    if (must) {   // asked for explicitly: do not hide it
      return fail(POVAR_ERR_NCCL, "peer exchange requested but CUDA IPC / peer access is unavailable");
    }
    return POVAR_OK;   // ncclAllReduce per term instead
  }
  for (int r = 0; r < world_; ++r) {
    ps->px.recv[r] = static_cast<double*>(base[r]);
  }
  ps->px.rank = rank_;
  ps->px.world = world_;
  ps->px.stride = stride;
  ps->px.count = reinterpret_cast<unsigned int*>(static_cast<char*>(ps->mem) + recv_pad);
  ps->ok = true;
  peer_ok_ = true;
  return POVAR_OK;
}

const PeerExchange* Engine::exchange() const { return peer_ok_ ? &peer_->px : nullptr; }

int Engine::allreduce(double* buf, size_t n, bool skip_when_done) {
  if (world_ <= 1) return POVAR_OK;
  if (peer_ok_ && n <= peer_->px.stride && peer_small_) {
    launch_peer_allreduce(d_, buf, n, peer_->px, lc(), skip_when_done);
    return POVAR_OK;
  }
  if (!nccl_comm_) return fail(POVAR_ERR_NCCL, "reduction needs an NCCL communicator (host rendezvous handle)");
  // ncclDouble = 8, ncclSum = 0
  const int rc = nccl_->AllReduce(buf, buf, n, 8, 0, nccl_comm_, stream_);
  if (rc != 0) return fail(POVAR_ERR_NCCL, "ncclAllReduce failed");
  return POVAR_OK;
}

void Engine::set_model(double alpha) {
  mp_.c1 = std::sqrt(1.0 - alpha);
  mp_.c2 = std::sqrt(alpha);
  mp_.robust_norm = opt_.robust_norm;
  mp_.huber = opt_.huber_parameter;
  mp_.jacobi_eps = opt_.jacobi_scaling_epsilon > 0 ? opt_.jacobi_scaling_epsilon : kEpsSqrtHost;
}

// ---------------------------------------------------------------------------------------------
int Engine::init_varproj(double alpha) {
  PV_CUDA(cudaSetDevice(device_));
  set_model(alpha);
  launch_init_varproj(d_, mp_, lc());
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

// cost kernels + (sharded) the in-place sum over the ranks: the result is trial_out[0..7] on the device
int Engine::enqueue_cost(bool joint, double alpha, bool reduce) {
  set_model(joint ? opt_.alpha : alpha);
  launch_cost(d_, mp_, joint, lc());
  return reduce ? allreduce(d_.trial_out, 8) : POVAR_OK;
}

void Engine::decode_cost(const double* v, povar_residual_info* out) {
  out->error_all = v[0];
  out->residual_sum_all = v[1];
  out->error_valid = v[2];
  out->residual_sum_valid = v[3];
  out->num_obs_all = static_cast<long long>(v[4] + 0.5);
  out->num_obs_valid = static_cast<long long>(v[5] + 0.5);
  out->is_numerically_valid = v[6] > 0 ? 0 : 1;
}

int Engine::cost(bool joint, double alpha, povar_residual_info* out) {
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaEventRecord(ev_[0], stream_));
  {
    const int rc = enqueue_cost(joint, alpha);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(cudaGetLastError());
  double* v = host_out_ + 8;
  PV_CUDA(cudaMemcpyAsync(v, d_.trial_out, 8 * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaEventRecord(ev_[1], stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  times_.residual += elapsed(ev_[0], ev_[1]);
  decode_cost(v, out);
  return POVAR_OK;
}

// per-observation coefficients the term kernels stream (kernels_series.cu): step 2's coefficients, step 1's HUBER
// weights
int Engine::alloc_lin_buffers(bool joint) {
  if (joint && !d_.obs_d) {
    PV_ALLOC(d_.obs_d, static_cast<size_t>(nnz_) * 3);
    PV_ALLOC(d_.csc_d, static_cast<size_t>(nnz_) * 3);
    PV_ALLOC(d_.sell_d, static_cast<size_t>(d_.ix.sell_slots) * 3);
  }
  if (!joint && opt_.robust_norm == POVAR_NORM_HUBER && !d_.obs_w) {
    PV_ALLOC(d_.obs_w, static_cast<size_t>(nnz_));
    PV_ALLOC(d_.csc_w, static_cast<size_t>(nnz_));
    PV_ALLOC(d_.sell_w, static_cast<size_t>(d_.ix.sell_slots));
  }
  return POVAR_OK;
}

int Engine::linearize(bool joint, double alpha, bool defer_check) {
  PV_CUDA(cudaSetDevice(device_));
  set_model(joint ? opt_.alpha : alpha);
  joint_lin_ = joint ? 1 : 0;
  have_solve_ = false;
  dim_ = joint ? 11 : 12;
  {
    const int rc = alloc_lin_buffers(joint);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(mark(6));
  PV_CUDA(cudaMemsetAsync(d_.flags, 0, 4 * sizeof(int), stream_));
  // landmark side: Jl^T Jl, Jl^T r, column scales (LinearizorSC step 1 does not scale Jl:
  // solver/linearizor_sc.cpp:174-203; step 2 scales it for every solver)
  launch_lin_landmark(d_, mp_, joint, joint || lm_power_step(opt_, false), lc());
  // camera side: Jp^T Jp as Kronecker sums, then the pose scales
  launch_kron(d_, mp_, joint, KRON_HPP, lc());
  launch_reduce_items(d_, d_.item_kron, kKron, d_.kron, false, lc());
  {
    const int rc = allreduce(d_.kron, static_cast<size_t>(C_) * kKron);
    if (rc != POVAR_OK) return rc;
  }
  launch_cam_scale(d_, mp_, lc());
  launch_cam_rec_static(d_, joint, lc());
  // numerical-failure flag of this shard as a double, summed over the ranks in place
  launch_flag_to_double(d_, lc());
  {
    const int rc = allreduce(d_.trial_out + 9, 1);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(mark(7));
  PV_CUDA(cudaGetLastError());
  if (capturing_) return POVAR_OK;   // the decision kernel of the trial reads the flag
  if (defer_check) {
    // the caller goes on to a trial(): the flag comes back with that trial's results (one synchronisation)
    lin_check_pending_ = true;
    return POVAR_OK;
  }
  double* v = host_out_ + 8;
  PV_CUDA(cudaMemcpyAsync(v + 9, d_.trial_out + 9, sizeof(double), cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  times_.linearize += elapsed(ev_[6], ev_[7]);
  if (v[9] > 0) return fail(POVAR_NUM_LINEARIZATION, "did not expect numerical failure during linearization");
  return POVAR_OK;
}

// raw_c = sum over the observations of camera c of the camera half of E0 (or of b), all ranks.
// skip_when_done: the launches return at once when ctl->done is set (inside a power series or a CG solve).
// fused_reduce: the caller's term kernel adds the item partials (and exchanges them) itself.
int Engine::e0_product(bool joint, bool skip_when_done, bool fused_reduce) {
  // the passes gather y from the camera records (cam_rec), written by whoever made y
  launch_e0_landmark_v2(d_, mp_, joint, skip_when_done, lc());
  launch_passB_e0_v2(d_, mp_, joint, skip_when_done, lc());
  if (fused_reduce) return POVAR_OK;
  launch_reduce_items(d_, d_.item_part, 12, d_.cam_raw, skip_when_done, lc());
  return allreduce(d_.cam_raw, static_cast<size_t>(C_) * 12, skip_when_done);
}

int Engine::solve_power(bool joint, double lambda) {
  const bool poba = !joint && opt_.solver_type_step_1 == POVAR_POWER_SCHUR_COMPLEMENT;
  const double lambda_lm = joint ? lambda : (poba ? lambda : 0.0);
  PV_CUDA(mark(0));
  // prepare_Hb_*: Hll^-1 and Hll^-1 Jl^T r per landmark; B^-1 per camera; b
  launch_prep_landmark(d_, joint, lambda_lm, false, lc(), (joint || poba) ? lambda_dev_ : nullptr);
  launch_cam_binv(d_, joint, lambda, lc(), lambda_dev_);
  launch_passB(d_, mp_, joint, lc());
  launch_reduce_items(d_, d_.item_part, 12, d_.cam_raw, false, lc());
  {
    const int rc = allreduce(d_.cam_raw, static_cast<size_t>(C_) * 12);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(mark(1));
  // solve_*: accum = B^-1(-b); tmp = B^-1 E0 tmp; accum += tmp; early exit on zeta < eta
  {
    const int rc = enqueue_series(joint);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(mark(2));
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

// One power series is b -> x0, series start, then per term landmark half, camera half, term kernel -- the same
// arguments in every solve of a model (the damping enters before, the stopping rule is applied on the device, the
// number of a peer exchange and of a term are device-side counters).  capture_series builds it once per model as a
// CUDA graph with a conditional WHILE node whose body is one term: k_series_start and the last block of k_term16 set
// the condition (cudaGraphSetConditional), so a solve is ONE launch that runs exactly the terms the reference's
// stopping rule asks for.  (Until this round the graph held all m terms and the converged ones returned at once:
// 430 skipped launches of 2-4 us per venice-1778 solve.)  The first solve of a model runs eagerly -- it sets
// function attributes -- and so does a series whose exchange is ncclAllReduce (no peer memory).  Inside the solve
// graph the same prefix and WHILE node go into the graph being captured.
int Engine::enqueue_series(bool joint) {
  if (capturing_) return capture_series(joint);
  const int m = opt_.power_sc_iterations;
  const int which = joint ? 1 : 0;
  const bool graphable = term_mode() != kTermRaw;
  if (!graphable || series_calls_[which]++ == 0) {
    launch_finish_b(d_, joint, lc());
    launch_series_start(d_, opt_.r_tolerance, m, lc());
    for (int i = 1; i <= m; ++i) {
      const int rc = e0_product(joint, true, term_mode() != kTermRaw);
      if (rc != POVAR_OK) return rc;
      launch_series_term(d_, joint, i, opt_.eta, opt_.r_tolerance, term_mode(), exchange(), lc());
    }
    series_terms_counted_ = true;   // the launches above are in launches_ (skipped ones included)
    return POVAR_OK;
  }
  // the graph holds the model parameters of its capture (alpha, robust norm): other ones need a new graph
  const ModelParams& was = series_mp_[which];
  if (series_graph_[which] && (was.c1 != mp_.c1 || was.c2 != mp_.c2 || was.robust_norm != mp_.robust_norm ||
                               was.huber != mp_.huber || was.jacobi_eps != mp_.jacobi_eps)) {
    PV_CUDA(cudaStreamSynchronize(stream_));   // its last launch may still run
    cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(series_graph_[which]));
    series_graph_[which] = nullptr;
  }
  if (!series_graph_[which]) {
    const int rc = capture_graph(&series_graph_[which], [&]() { return capture_series(joint); });
    if (rc != POVAR_OK) return rc;
    series_mp_[which] = mp_;
  }
  PV_CUDA(cudaGraphLaunch(static_cast<cudaGraphExec_t>(series_graph_[which]), stream_));
  launches_ += 2;                  // b -> x0 and the series start; the terms are counted when the solve reports them
  series_terms_counted_ = false;
  return POVAR_OK;
}

int Engine::finish_solve(bool joint, double* inc, int32_t* iterations) {
  SeriesCtl h{};
  PV_CUDA(cudaMemcpyAsync(&h, d_.ctl, sizeof(h), cudaMemcpyDeviceToHost, stream_));
  if (inc) {
    PV_CUDA(cudaMemcpyAsync(inc, d_.vec_acc, sizeof(double) * static_cast<size_t>(C_) * (joint ? 11 : 12),
                            cudaMemcpyDeviceToHost, stream_));
  }
  PV_CUDA(cudaStreamSynchronize(stream_));
  times_.prepare += elapsed(ev_[0], ev_[1]);
  times_.reduced_solve += elapsed(ev_[1], ev_[2]);
  if (iterations) *iterations = h.iterations;
  count_series_terms(h.term);
  if (h.peer_timeout) return fail(POVAR_ERR_NCCL, "peer exchange of the camera sums timed out (a rank is gone?)");
  if (h.nonfinite) return POVAR_NUM_NONFINITE_INC;
  return POVAR_OK;
}

// kernels the loop of the series graph ran: three per term (the host learns the count with the solve's results)
void Engine::count_series_terms(int terms) {
  if (series_terms_counted_) return;
  series_terms_counted_ = true;
  launches_ += 3LL * terms;
}

int Engine::enqueue_solve(bool joint, double lambda) {
  if (static_cast<int>(joint) != joint_lin_) return fail(POVAR_ERR_INVALID, "solve called without a matching linearize");
  have_solve_ = true;
  if (joint) return opt_.solver_type_step_2 == POVAR_RIPOBA ? solve_power(true, lambda) : solve_pcg(true, lambda);
  switch (opt_.solver_type_step_1) {
    case POVAR_POWER_VARPROJ:
    case POVAR_POWER_SCHUR_COMPLEMENT:
      return solve_power(false, lambda);
    case POVAR_PCG:
      return solve_pcg(false, lambda);
    case POVAR_CHOLESKY:
      return solve_cholesky(lambda);
    default:
      return fail(POVAR_ERR_INVALID, "unknown solver_type_step_1");
  }
}

int Engine::solve(bool joint, double lambda, double* inc, int32_t* iterations) {
  PV_CUDA(cudaSetDevice(device_));
  const int rc = enqueue_solve(joint, lambda);
  if (rc != POVAR_OK) return rc;
  return finish_solve(joint, inc, iterations);
}

// b (and B, B^-1) exactly as the power solvers build them; shared by PCG / RIPCG / CHOLESKY
int Engine::prepare_reduced_system(bool joint, double lambda, double lambda_lm) {
  launch_prep_landmark(d_, joint, lambda_lm, true, lc(), joint ? lambda_dev_ : nullptr);
  launch_cam_binv(d_, joint, lambda, lc(), lambda_dev_);
  launch_passB(d_, mp_, joint, lc());
  launch_reduce_items(d_, d_.item_part, 12, d_.cam_raw, false, lc());
  const int rc = allreduce(d_.cam_raw, static_cast<size_t>(C_) * 12);
  if (rc != POVAR_OK) return rc;
  launch_finish_b(d_, joint, lc());
  return POVAR_OK;
}

// out = S p = B p - E0 p   (the reduced camera system applied implicitly)
int Engine::schur_product(bool joint, const double* p, double* out, bool skip_when_done) {
  const int n = C_ * (joint ? 11 : 12);
  launch_make_y(d_, joint, p, d_.vec_y, lc());
  const int rc = e0_product(joint, skip_when_done, false);
  if (rc != POVAR_OK) return rc;
  launch_e0_finish(d_, joint, d_.vec_x, lc());
  launch_block_matvec(d_, joint ? 11 : 12, d_.Bmat, p, out, lc());
  launch_axpby(d_, n, 1.0, out, -1.0, d_.vec_x, out, lc());
  return POVAR_OK;
}

// ConjugateGradientsSolver::solve / solve_joint (cg/conjugate_gradient.hpp:114-489) with the block-Jacobi
// preconditioner (cg/preconditioner.hpp:70-144), x0 = 0, r_tolerance = -1, then x = -x
// (solver/linearizor_base.cpp:102-147).  The scalars (rho, beta, alpha, Q) and every termination test of the
// reference's loop -- its NaN behaviour included -- live on the device (k_cg_scalar): the host enqueues
// iterations a few at a time and reads the control block once per batch; after termination the remaining
// launches of a batch return at once.
int Engine::solve_pcg(bool joint, double lambda) {
  const int D = joint ? 11 : 12;
  const int n = C_ * D;
  const size_t bytes = sizeof(double) * static_cast<size_t>(n);
  PV_CUDA(mark(0));
  // LinearizorSC step 1 has no landmark damping (landmark_block.hpp:360-374); step 2 has (:414-431)
  int rc = prepare_reduced_system(joint, lambda, joint ? lambda : 0.0);
  if (rc != POVAR_OK) return rc;
  launch_kron(d_, mp_, joint, KRON_SDIAG, lc());
  launch_reduce_items(d_, d_.item_kron, kKron, d_.kron2, false, lc());
  rc = allreduce(d_.kron2, static_cast<size_t>(C_) * kKron);
  if (rc != POVAR_OK) return rc;
  launch_cam_precond(d_, joint, d_.kron2, lc());
  PV_CUDA(mark(1));

  const double* b = d_.b;
  double *x = d_.cg_x, *r = d_.cg_r, *p = d_.cg_p, *z = d_.cg_z, *q = d_.cg_q, *tmp = d_.vec_tmp;
  const int min_it = opt_.min_linear_solver_iterations, max_it = opt_.max_linear_solver_iterations;
  PV_CUDA(cudaMemsetAsync(x, 0, bytes, stream_));
  PV_CUDA(cudaMemsetAsync(p, 0, bytes, stream_));
  PV_CUDA(cudaMemcpyAsync(r, b, bytes, cudaMemcpyDeviceToDevice, stream_));   // r = b - S*0
  launch_dot_partials(d_, n, b, b, lc());
  launch_cg_scalar(d_, CG_BEGIN, 0, opt_.eta, min_it, max_it, lc());          // |b| = 0: done at once
  // iteration it (+ *base on the device)
  auto iteration = [&](int it, const int* base) -> int {
    launch_block_matvec(d_, D, d_.Mprec, r, z, lc());                         // z = M^-1 r
    launch_dot_partials(d_, n, r, z, lc());
    launch_cg_scalar(d_, CG_RHO, it, opt_.eta, min_it, max_it, lc(), base);
    launch_cg_update(d_, CG_UPDATE_P, n, it, z, p, lc(), base);               // p = z + beta p
    int rc2 = schur_product(joint, p, q, true);                               // q = S p
    if (rc2 != POVAR_OK) return rc2;
    launch_dot_partials(d_, n, p, q, lc());
    launch_cg_scalar(d_, CG_PQ, it, opt_.eta, min_it, max_it, lc(), base);
    launch_cg_update(d_, CG_UPDATE_X, n, it, p, x, lc(), base);               // x += alpha p
    if (it % 10 == 0) {                                                       // residual_reset_period
      rc2 = schur_product(joint, x, tmp, true);
      if (rc2 != POVAR_OK) return rc2;
      launch_axpby(d_, n, 1.0, b, -1.0, tmp, r, lc());                        // r = b - S x
    } else {
      launch_cg_update(d_, CG_UPDATE_R, n, it, q, r, lc(), base);             // r -= alpha q
    }
    launch_axpby(d_, n, 1.0, b, 1.0, r, tmp, lc());
    launch_dot_partials(d_, n, x, tmp, lc());
    launch_cg_scalar(d_, CG_ZETA, it, opt_.eta, min_it, max_it, lc(), base);  // Q, zeta < eta, max iterations
    return POVAR_OK;
  };
  if (capturing_) {
    // a WHILE node around ten iterations, numbered from a device counter, so that the residual reset falls on
    // the same iterations; the node ends when the device's termination tests set ctl->done
    int* base = &lm_->cg_base;
    unsigned long long h = 0;
    rc = new_cond(&h);
    if (rc != POVAR_OK) return rc;
    launch_cg_loop(d_.ctl, base, max_it, false, h, lc());
    rc = capture_cond(cudaGraphCondTypeWhile, h, [&]() -> int {
      for (int k = 1; k <= 10; ++k) {
        const int rc2 = iteration(k, base);
        if (rc2 != POVAR_OK) return rc2;
      }
      launch_cg_loop(d_.ctl, base, max_it, true, h, lc());
      return POVAR_OK;
    });
    if (rc != POVAR_OK) return rc;
  } else {
    SeriesCtl* hctl = reinterpret_cast<SeriesCtl*>(host_out_);
    constexpr int kBatch = 4;
    for (int it = 1; it <= max_it;) {
      for (int k = 0; k < kBatch && it <= max_it; ++k, ++it) {
        rc = iteration(it, nullptr);
        if (rc != POVAR_OK) return rc;
      }
      PV_CUDA(cudaMemcpyAsync(hctl, d_.ctl, sizeof(SeriesCtl), cudaMemcpyDeviceToHost, stream_));
      PV_CUDA(cudaStreamSynchronize(stream_));
      if (hctl->done) break;
    }
  }
  launch_axpby(d_, n, -1.0, x, 0.0, nullptr, d_.vec_acc, lc());   // "negate the pose increment"
  launch_finite_check(d_, n, d_.vec_acc, lc());
  PV_CUDA(mark(2));
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

// CHOLESKY, step 1 (solver/linearizor_sc.cpp:121-128, sc/linearization_sc.hpp:236-245): the reference
// factorises the sparse reduced camera system with Eigen::SimplicialLLT; here S is assembled without atomics and
// factorised by the hand-written blocked LL^T of kernels_chol.cu (FP64 tensor-core tile updates).  S is dense while
// that fits under kCholDenseCap, tile-sparse beyond (only the tiles of the factor that can be non-zero, in reverse
// Cuthill-McKee camera order).  The solution of S x = -b is unique, so ordering / blocking do not change the result
// beyond rounding.
constexpr long long kCholDenseCap = 96LL << 30;

// the tile pattern of the factor: co-visibility bitmap on the device, ordering and symbolic factorisation on the
// host, the pattern and the tiles in device memory.  Fails with POVAR_ERR_UNSUPPORTED when the factor would not fit.
int Engine::setup_cholesky_tiles() {
  const size_t words = (static_cast<size_t>(C_) + 31) / 32;
  std::vector<unsigned int> bits(static_cast<size_t>(C_) * words);
  {   // the bitmap (C^2 / 8 bytes) lives only until the host has it
    void* dbits = nullptr;
    PV_CUDA(cudaMallocAsync(&dbits, sizeof(unsigned int) * bits.size(), stream_));
    cudaError_t e = build_covisibility(L_, C_, d_.ix.lm_ptr, d_.ix.obs_cam, static_cast<unsigned int*>(dbits), lc());
    if (e == cudaSuccess) {
      e = cudaMemcpyAsync(bits.data(), dbits, sizeof(unsigned int) * bits.size(), cudaMemcpyDeviceToHost, stream_);
    }
    cudaFreeAsync(dbits, stream_);
    PV_CUDA(e);
    PV_CUDA(cudaStreamSynchronize(stream_));
  }
  CholPattern& p = chol_pat_;
  chol_symbolic(C_, 12, bits, 0, &p);
  const size_t T = static_cast<size_t>(p.T), tiles = static_cast<size_t>(p.tiles());
  const size_t need = sizeof(double) * (tiles * 4096 + (chol_linv_ ? 0 : T * 4096 + static_cast<size_t>(p.n_pad))) +
                      sizeof(int) * (T * T + 2 * (T + 1) + 2 * tiles + static_cast<size_t>(C_));
  size_t free_b = 0, total_b = 0;
  PV_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (need > free_b) {
    return fail(POVAR_ERR_UNSUPPORTED, "CHOLESKY: tile-sparse factor needs " + std::to_string(need) + " bytes, " +
                                           std::to_string(free_b) + " bytes free on the device");
  }
  int *slot = nullptr, *col_ptr = nullptr, *col_row = nullptr, *row_ptr = nullptr, *row_col = nullptr, *perm = nullptr;
  PV_ALLOC(chol_dev_.tiles, tiles * 4096);
  PV_ALLOC(slot, T * T);
  PV_ALLOC(col_ptr, T + 1);
  PV_ALLOC(row_ptr, T + 1);
  PV_ALLOC(col_row, tiles);
  PV_ALLOC(row_col, tiles);
  PV_ALLOC(perm, C_);
  auto up = [&](int* dst, const std::vector<int>& src) {
    return cudaMemcpyAsync(dst, src.data(), sizeof(int) * src.size(), cudaMemcpyHostToDevice, stream_);
  };
  PV_CUDA(up(slot, p.slot));
  PV_CUDA(up(col_ptr, p.col_ptr));
  PV_CUDA(up(col_row, p.col_row));
  PV_CUDA(up(row_ptr, p.row_ptr));
  PV_CUDA(up(row_col, p.row_col));
  PV_CUDA(up(perm, p.perm));
  PV_CUDA(cudaStreamSynchronize(stream_));   // the host vectors are pageable
  chol_dev_.T = p.T;
  chol_dev_.slot = slot;
  chol_dev_.col_ptr = col_ptr;
  chol_dev_.col_row = col_row;
  chol_dev_.row_ptr = row_ptr;
  chol_dev_.row_col = row_col;
  chol_dev_.perm = perm;
  chol_tiled_ready_ = true;
  return POVAR_OK;
}

// S dense or tile-sparse; the first solve with either builds the tile pattern or allocates the dense matrix, then the
// factor's diagonal inverses and the right-hand side (the same sizes on both paths: a handle switched between the two
// shares them)
int Engine::alloc_cholesky(bool* tiled) {
  const int n_pad = chol_padded(12 * C_);
  *tiled = chol_storage_ == 1 || static_cast<long long>(n_pad) * n_pad * 8 > kCholDenseCap;
  if (*tiled && !chol_tiled_ready_) {
    const int rc = setup_cholesky_tiles();
    if (rc != POVAR_OK) return rc;
  }
  if (!*tiled && !d_.dense_S) PV_ALLOC(d_.dense_S, static_cast<size_t>(n_pad) * n_pad);
  if (!chol_linv_) {
    PV_ALLOC(chol_linv_, static_cast<size_t>(n_pad) * 64);
    PV_ALLOC(chol_rhs_, static_cast<size_t>(n_pad));
  }
  return POVAR_OK;
}

int Engine::solve_cholesky(double lambda) {
  const int n = 12 * C_;
  const int n_pad = chol_padded(n);
  PV_CUDA(mark(0));
  int rc = prepare_reduced_system(false, lambda, 0.0);
  if (rc != POVAR_OK) return rc;
  bool tiled = false;
  rc = alloc_cholesky(&tiled);   // on first use inside this trial's prepare time
  chol_tiled_active_ = tiled;
  if (rc != POVAR_OK) return rc;
  if (tiled) {
    PV_CUDA(cudaMemsetAsync(chol_dev_.tiles, 0, sizeof(double) * 4096 * static_cast<size_t>(chol_pat_.tiles()), stream_));
    launch_schur_tiles(d_, mp_, chol_dev_, n_pad, lc());
  } else {
    PV_CUDA(cudaMemsetAsync(d_.dense_S, 0, sizeof(double) * static_cast<size_t>(n_pad) * n_pad, stream_));
    launch_schur_lower(d_, mp_, d_.dense_S, n_pad, lc());
  }
  PV_CUDA(mark(1));
  PV_CUDA(cudaMemsetAsync(chol_rhs_, 0, sizeof(double) * static_cast<size_t>(n_pad), stream_));
  int* info = d_.flags + 2;
  if (tiled) {
    launch_perm_gather_neg(C_, chol_dev_.perm, d_.b, chol_rhs_, lc());
    launch_cholesky_factor_tiles(chol_pat_, chol_dev_, chol_linv_, info, lc());
    launch_cholesky_solve_tiles(chol_pat_, chol_dev_, chol_linv_, chol_rhs_, info, lc());
    launch_perm_scatter(C_, chol_dev_.perm, chol_rhs_, d_.vec_acc, lc());
  } else {
    launch_axpby(d_, n, -1.0, d_.b, 0.0, nullptr, chol_rhs_, lc());
    launch_cholesky_factor(d_.dense_S, n_pad, chol_linv_, info, lc());
    launch_cholesky_solve(d_.dense_S, n_pad, chol_linv_, chol_rhs_, info, lc());
    PV_CUDA(cudaMemcpyAsync(d_.vec_acc, chol_rhs_, sizeof(double) * static_cast<size_t>(n), cudaMemcpyDeviceToDevice, stream_));
  }
  if (capturing_) {   // the read-back below as a kernel: info != 0 makes the step invalid
    launch_chol_status(info, d_.ctl, lc());
    launch_finite_check(d_, n, d_.vec_acc, lc());
    PV_CUDA(mark(2));
    PV_CUDA(cudaGetLastError());
    return POVAR_OK;
  }
  int hinfo = 0;
  PV_CUDA(cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, stream_));
  SeriesCtl h{};
  h.done = 1;
  h.iterations = 0;   // the reference reports 0 linear solver iterations for the direct solve
  PV_CUDA(cudaMemcpyAsync(d_.ctl, &h, sizeof(h), cudaMemcpyHostToDevice, stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  if (hinfo != 0) {
    // not positive definite: SimplicialLLT would report NumericalIssue; surface it as an invalid step
    h.nonfinite = 1;
    PV_CUDA(cudaMemcpyAsync(d_.ctl, &h, sizeof(h), cudaMemcpyHostToDevice, stream_));
    PV_CUDA(cudaStreamSynchronize(stream_));
  } else {
    launch_finite_check(d_, n, d_.vec_acc, lc());
  }
  PV_CUDA(mark(2));
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

// the factorisation and substitution kernels on a caller-supplied symmetric matrix (tests)
int debug_cholesky(int n, const double* A, const double* b, double* x, int* info_out) {
  if (n <= 0 || !A || !b || !x) return POVAR_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return POVAR_ERR_NO_DEVICE;
  const int n_pad = chol_padded(n);
  double *S = nullptr, *linv = nullptr, *r = nullptr;
  int* info = nullptr;
  int rc = POVAR_OK;
  auto ok = [&](cudaError_t e) {
    if (e != cudaSuccess) rc = POVAR_ERR_CUDA;
    return e == cudaSuccess;
  };
  if (ok(cudaSetDevice(0)) && ok(cudaMalloc(&S, sizeof(double) * static_cast<size_t>(n_pad) * n_pad)) &&
      ok(cudaMalloc(&linv, sizeof(double) * static_cast<size_t>(n_pad) * 64)) &&
      ok(cudaMalloc(&r, sizeof(double) * static_cast<size_t>(n_pad))) && ok(cudaMalloc(&info, sizeof(int))) &&
      ok(cudaMemset(S, 0, sizeof(double) * static_cast<size_t>(n_pad) * n_pad)) &&
      ok(cudaMemset(r, 0, sizeof(double) * static_cast<size_t>(n_pad))) &&
      ok(cudaMemcpy2D(S, sizeof(double) * n_pad, A, sizeof(double) * n, sizeof(double) * n, n, cudaMemcpyHostToDevice)) &&
      ok(cudaMemcpy(r, b, sizeof(double) * n, cudaMemcpyHostToDevice))) {
    std::vector<double> ones(static_cast<size_t>(n_pad - n), 1.0);
    if (n_pad > n) {
      ok(cudaMemcpy2D(S + static_cast<size_t>(n) * n_pad + n, sizeof(double) * (n_pad + 1), ones.data(), sizeof(double),
                      sizeof(double), n_pad - n, cudaMemcpyHostToDevice));
    }
    LaunchCfg lc{};
    launch_cholesky_factor(S, n_pad, linv, info, lc);
    launch_cholesky_solve(S, n_pad, linv, r, info, lc);
    int hinfo = 0;
    ok(cudaMemcpy(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost));
    ok(cudaMemcpy(x, r, sizeof(double) * n, cudaMemcpyDeviceToHost));
    ok(cudaGetLastError());
    if (info_out) *info_out = hinfo;
  }
  cudaFree(S);
  cudaFree(linv);
  cudaFree(r);
  cudaFree(info);
  return rc;
}

// the tile-sparse factorisation and substitution on a caller-supplied symmetric matrix (tests): the pattern is that of
// the non-zero block x block blocks of A's lower triangle, ordered and factorised symbolically as a handle's S is
int debug_sparse_cholesky(int n, int block, const double* A, const double* b, double* x, int* info_out,
                          long long* stored_tiles) {
  if (n <= 0 || block <= 0 || !A || !b || !x) return POVAR_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return POVAR_ERR_NO_DEVICE;
  const int nb = (n + block - 1) / block;
  const size_t words = (static_cast<size_t>(nb) + 31) / 32;
  std::vector<unsigned int> bits(static_cast<size_t>(nb) * words, 0u);
  for (int a = 0; a < nb; ++a) {
    for (int c = 0; c <= a; ++c) {
      bool nz = a == c;
      for (int i = a * block; i < std::min(n, a * block + block) && !nz; ++i) {
        for (int j = c * block; j < std::min(i + 1, c * block + block); ++j) nz = nz || A[static_cast<size_t>(i) * n + j] != 0.0;
      }
      if (!nz) continue;
      bits[static_cast<size_t>(a) * words + (c >> 5)] |= 1u << (c & 31);
      bits[static_cast<size_t>(c) * words + (a >> 5)] |= 1u << (a & 31);
    }
  }
  CholPattern p;
  chol_symbolic(nb, block, bits, 0, &p);
  // original row of every row of the factor order, -1 on padding (identity)
  std::vector<int> at(nb), orig(p.n_pad, -1);
  for (int c = 0; c < nb; ++c) at[p.perm[c]] = c;
  for (int R = 0; R < p.n_pad; ++R) {
    const int pos = R / block;
    if (pos < nb && block * at[pos] + R % block < n) orig[R] = block * at[pos] + R % block;
  }
  const size_t tiles = static_cast<size_t>(p.tiles()), T = static_cast<size_t>(p.T);
  std::vector<double> H(tiles * 4096, 0.0), r(p.n_pad, 0.0);
  for (int J = 0; J < p.T; ++J) {
    for (int q = p.col_ptr[J]; q < p.col_ptr[J + 1]; ++q) {
      const int I = p.col_row[q];
      for (int rr = 0; rr < 64; ++rr) {
        for (int cc = 0; cc < 64; ++cc) {
          const int R = I * 64 + rr, Cc = J * 64 + cc;
          if (R < Cc) continue;
          const int oi = orig[R], oj = orig[Cc];
          H[static_cast<size_t>(q) * 4096 + rr * 64 + cc] =
              (oi < 0 || oj < 0) ? (R == Cc ? 1.0 : 0.0)
                                 : A[static_cast<size_t>(std::max(oi, oj)) * n + std::min(oi, oj)];
        }
      }
    }
  }
  for (int R = 0; R < p.n_pad; ++R) r[R] = orig[R] >= 0 ? b[orig[R]] : 0.0;
  double *dt = nullptr, *linv = nullptr, *dr = nullptr;
  int *slot = nullptr, *col_ptr = nullptr, *col_row = nullptr, *row_ptr = nullptr, *row_col = nullptr, *info = nullptr;
  int rc = POVAR_OK;
  auto ok = [&](cudaError_t e) {
    if (e != cudaSuccess) rc = POVAR_ERR_CUDA;
    return e == cudaSuccess;
  };
  auto up = [&](int** dst, const std::vector<int>& src) {
    return ok(cudaMalloc(dst, sizeof(int) * std::max<size_t>(src.size(), 1))) &&
           ok(cudaMemcpy(*dst, src.data(), sizeof(int) * src.size(), cudaMemcpyHostToDevice));
  };
  if (ok(cudaSetDevice(0)) && ok(cudaMalloc(&dt, sizeof(double) * H.size())) &&
      ok(cudaMalloc(&linv, sizeof(double) * T * 4096)) && ok(cudaMalloc(&dr, sizeof(double) * r.size())) &&
      ok(cudaMalloc(&info, sizeof(int))) &&
      ok(cudaMemcpy(dt, H.data(), sizeof(double) * H.size(), cudaMemcpyHostToDevice)) &&
      ok(cudaMemcpy(dr, r.data(), sizeof(double) * r.size(), cudaMemcpyHostToDevice)) && up(&slot, p.slot) &&
      up(&col_ptr, p.col_ptr) && up(&col_row, p.col_row) && up(&row_ptr, p.row_ptr) && up(&row_col, p.row_col)) {
    CholTilesDev s;
    s.T = p.T;
    s.tiles = dt;
    s.slot = slot;
    s.col_ptr = col_ptr;
    s.col_row = col_row;
    s.row_ptr = row_ptr;
    s.row_col = row_col;
    LaunchCfg lc{};
    launch_cholesky_factor_tiles(p, s, linv, info, lc);
    launch_cholesky_solve_tiles(p, s, linv, dr, info, lc);
    int hinfo = 0;
    ok(cudaMemcpy(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost));
    ok(cudaMemcpy(r.data(), dr, sizeof(double) * r.size(), cudaMemcpyDeviceToHost));
    ok(cudaGetLastError());
    for (int R = 0; R < p.n_pad; ++R) {
      if (orig[R] >= 0) x[orig[R]] = r[R];
    }
    if (info_out) *info_out = hinfo;
    if (stored_tiles) *stored_tiles = p.tiles();
  }
  for (void* q : {static_cast<void*>(dt), static_cast<void*>(linv), static_cast<void*>(dr), static_cast<void*>(slot),
                  static_cast<void*>(col_ptr), static_cast<void*>(col_row), static_cast<void*>(row_ptr),
                  static_cast<void*>(row_col), static_cast<void*>(info)}) {
    cudaFree(q);
  }
  return rc;
}

// back-substitution and camera update + (sharded) the sum of l_diff over the ranks: trial_out[8] on the device
int Engine::enqueue_apply(bool joint, double alpha, bool reduce) {
  if (static_cast<int>(joint) != joint_lin_ || !have_solve_) {
    return fail(POVAR_ERR_INVALID, "apply called without a matching linearize + solve");
  }
  set_model(joint ? opt_.alpha : alpha);
  const size_t C12 = static_cast<size_t>(C_) * 12;
  if (joint) {
    // apply_joint (linearizor_power_varproj.cpp:276-308): landmarks first, then P += s o (Pi inc)
    launch_make_y(d_, true, d_.vec_acc, d_.vec_y, lc());
    launch_backsub_joint(d_, mp_, d_.vec_y, lc());
    launch_cam_update_joint(d_, d_.vec_y, lc());
  } else if (opt_.solver_type_step_1 == POVAR_POWER_SCHUR_COMPLEMENT) {
    // linearizor_power_varproj.cpp:260-270
    launch_make_y(d_, false, d_.vec_acc, d_.vec_y, lc());
    launch_backsub_poba(d_, mp_, d_.vec_y, lc());
    launch_cam_update_pose(d_, d_.vec_acc, lc());
  } else {
    // VarPro flavours (linearizor_power_varproj.cpp:250-259, linearizor_sc.cpp:69-89):
    // cameras first, then the closed-form landmark re-solve
    PV_CUDA(cudaMemcpyAsync(P_prev_, d_.P, sizeof(double) * C12, cudaMemcpyDeviceToDevice, stream_));
    launch_cam_update_pose(d_, d_.vec_acc, lc());
    DeviceState tmp = d_;
    tmp.P_bak = P_prev_;
    launch_backsub_varpro(tmp, mp_, d_.vec_acc, lc());
  }
  return reduce ? allreduce(d_.trial_out + 8, 1) : POVAR_OK;
}

int Engine::apply(bool joint, double alpha, double* l_diff) {
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaEventRecord(ev_[0], stream_));
  {
    const int rc = enqueue_apply(joint, alpha);
    if (rc != POVAR_OK) return rc;
  }
  PV_CUDA(cudaGetLastError());
  double* v = host_out_ + 8;
  PV_CUDA(cudaMemcpyAsync(v + 8, d_.trial_out + 8, sizeof(double), cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaEventRecord(ev_[1], stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  times_.back_substitution += elapsed(ev_[0], ev_[1]);
  if (l_diff) *l_diff = v[8];
  return POVAR_OK;
}

// marks 0 (start), 1 (prepared), 2 (solved), 3 (applied)
int Engine::enqueue_trial(bool joint, double alpha, double lambda) {
  int rc = enqueue_solve(joint, lambda);
  if (rc != POVAR_OK) return rc;
  rc = backup(joint ? POVAR_STATE_JOINT : POVAR_STATE_POSE);
  if (rc != POVAR_OK) return rc;
  // sharded: the model decrease and the cost scalars of the trial travel together (trial_out[0..9), one exchange)
  rc = enqueue_apply(joint, alpha, /*reduce=*/false);
  if (rc != POVAR_OK) return rc;
  if (joint) {   // solver/bal_bundle_adjustment.cpp:700-705
    launch_normalize_cams(d_, lc());
    launch_normalize_joint(d_, lc());
  }
  PV_CUDA(mark(3));
  rc = enqueue_cost(joint, alpha, /*reduce=*/false);
  if (rc != POVAR_OK) return rc;
  return allreduce(d_.trial_out, 9);
}

int Engine::trial(bool joint, double alpha, double lambda, int32_t* iterations, double* l_diff,
                  povar_residual_info* ri) {
  PV_CUDA(cudaSetDevice(device_));
  const int rc = enqueue_trial(joint, alpha, lambda);
  if (rc != POVAR_OK) return rc;
  PV_CUDA(cudaGetLastError());
  static_assert(sizeof(SeriesCtl) <= 64, "SeriesCtl shares the pinned read-back buffer");
  SeriesCtl* hctl = reinterpret_cast<SeriesCtl*>(host_out_);
  double* v = host_out_ + 8;
  PV_CUDA(cudaMemcpyAsync(hctl, d_.ctl, sizeof(SeriesCtl), cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaMemcpyAsync(v, d_.trial_out, 16 * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaEventRecord(ev_[4], stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  times_.prepare += elapsed(ev_[0], ev_[1]);
  times_.reduced_solve += elapsed(ev_[1], ev_[2]);
  times_.back_substitution += elapsed(ev_[2], ev_[3]);
  times_.residual += elapsed(ev_[3], ev_[4]);
  if (lin_check_pending_) {
    lin_check_pending_ = false;
    times_.linearize += elapsed(ev_[6], ev_[7]);
    if (v[9] > 0) return fail(POVAR_NUM_LINEARIZATION, "did not expect numerical failure during linearization");
  }
  if (iterations) *iterations = hctl->iterations;
  count_series_terms(hctl->term);
  if (l_diff) *l_diff = v[8];
  if (ri) decode_cost(v, ri);
  if (hctl->peer_timeout) return fail(POVAR_ERR_NCCL, "peer exchange of the camera sums timed out (a rank is gone?)");
  if (hctl->nonfinite) return POVAR_NUM_NONFINITE_INC;
  return POVAR_OK;
}

int Engine::backup(int which) {
  (void)which;
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaMemcpyAsync(d_.P_bak, d_.P, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyDeviceToDevice, stream_));
  PV_CUDA(cudaMemcpyAsync(d_.X_bak, d_.X, sizeof(double) * static_cast<size_t>(L_) * 4, cudaMemcpyDeviceToDevice, stream_));
  return POVAR_OK;
}

int Engine::restore(int which) {
  (void)which;
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaMemcpyAsync(d_.P, d_.P_bak, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyDeviceToDevice, stream_));
  PV_CUDA(cudaMemcpyAsync(d_.X, d_.X_bak, sizeof(double) * static_cast<size_t>(L_) * 4, cudaMemcpyDeviceToDevice, stream_));
  return POVAR_OK;
}

int Engine::to_homogeneous() {
  PV_CUDA(cudaSetDevice(device_));
  launch_to_homogeneous(d_, lc());
  launch_normalize_cams(d_, lc());
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

int Engine::normalize_joint() {
  PV_CUDA(cudaSetDevice(device_));
  launch_normalize_cams(d_, lc());
  launch_normalize_joint(d_, lc());
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

int Engine::get_state(int which, double* cam_P, double* lms) {
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  if (cam_P) PV_CUDA(cudaMemcpy(cam_P, d_.P, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyDeviceToHost));
  if (lms && L_ > 0) {
    // straight into the caller's buffer (no staging vector: its page faults cost more than the copy);
    // step-1 landmarks are [x y z 1] on the device and [x y z] for the caller: a pitched copy drops w
    if (which == POVAR_STATE_JOINT) {
      PV_CUDA(cudaMemcpy(lms, d_.X, sizeof(double) * 4 * static_cast<size_t>(L_), cudaMemcpyDeviceToHost));
    } else {
      PV_CUDA(cudaMemcpy2D(lms, 3 * sizeof(double), d_.X, 4 * sizeof(double), 3 * sizeof(double),
                           static_cast<size_t>(L_), cudaMemcpyDeviceToHost));
    }
  }
  return POVAR_OK;
}

int Engine::set_state(int which, const double* cam_P, const double* lms) {
  PV_CUDA(cudaSetDevice(device_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  if (cam_P) PV_CUDA(cudaMemcpy(d_.P, cam_P, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyHostToDevice));
  if (lms) {
    std::vector<double> h(static_cast<size_t>(L_) * 4);
    for (int l = 0; l < L_; ++l) {
      if (which == POVAR_STATE_JOINT) {
        for (int k = 0; k < 4; ++k) h[4 * static_cast<size_t>(l) + k] = lms[4 * static_cast<size_t>(l) + k];
      } else {
        for (int k = 0; k < 3; ++k) h[4 * static_cast<size_t>(l) + k] = lms[3 * static_cast<size_t>(l) + k];
        h[4 * static_cast<size_t>(l) + 3] = 1.0;
      }
    }
    PV_CUDA(cudaMemcpy(d_.X, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice));
  }
  return POVAR_OK;
}

// get_state / set_state in device memory, ordered between the caller's stream and the handle's: the copies wait for
// the caller's work so far, the caller's stream waits for the copies
int Engine::get_state_device(int which, double* cam_P, double* lms, cudaStream_t caller) {
  PV_CUDA(cudaSetDevice(device_));
  if (cam_P && check_device_ptr(cam_P, "cam_P") != POVAR_OK) return POVAR_ERR_INVALID;
  if (lms && L_ > 0 && check_device_ptr(lms, "lms") != POVAR_OK) return POVAR_ERR_INVALID;
  int rc = wait_for(stream_, caller);
  if (rc != POVAR_OK) return rc;
  if (cam_P) {
    PV_CUDA(cudaMemcpyAsync(cam_P, d_.P, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyDeviceToDevice, stream_));
  }
  if (lms && L_ > 0) {
    if (which == POVAR_STATE_JOINT) {
      PV_CUDA(cudaMemcpyAsync(lms, d_.X, sizeof(double) * 4 * static_cast<size_t>(L_), cudaMemcpyDeviceToDevice, stream_));
    } else {
      PV_CUDA(cudaMemcpy2DAsync(lms, 3 * sizeof(double), d_.X, 4 * sizeof(double), 3 * sizeof(double),
                                static_cast<size_t>(L_), cudaMemcpyDeviceToDevice, stream_));
    }
  }
  return wait_for(caller, stream_);
}

int Engine::set_state_device(int which, const double* cam_P, const double* lms, cudaStream_t caller) {
  PV_CUDA(cudaSetDevice(device_));
  if (cam_P && check_device_ptr(cam_P, "cam_P") != POVAR_OK) return POVAR_ERR_INVALID;
  if (lms && L_ > 0 && check_device_ptr(lms, "lms") != POVAR_OK) return POVAR_ERR_INVALID;
  int rc = wait_for(stream_, caller);
  if (rc != POVAR_OK) return rc;
  if (cam_P) {
    PV_CUDA(cudaMemcpyAsync(d_.P, cam_P, sizeof(double) * static_cast<size_t>(C_) * 12, cudaMemcpyDeviceToDevice, stream_));
  }
  if (lms && L_ > 0) {
    if (which == POVAR_STATE_JOINT) {
      PV_CUDA(cudaMemcpyAsync(d_.X, lms, sizeof(double) * 4 * static_cast<size_t>(L_), cudaMemcpyDeviceToDevice, stream_));
    } else {
      PV_CUDA(cudaMemcpy2DAsync(d_.X, 4 * sizeof(double), lms, 3 * sizeof(double), 3 * sizeof(double),
                                static_cast<size_t>(L_), cudaMemcpyDeviceToDevice, stream_));
      launch_to_homogeneous(d_, lc());   // w = 1, as set_state writes it
      PV_CUDA(cudaGetLastError());
    }
  }
  return wait_for(caller, stream_);
}

int64_t Engine::debug_read(const char* name, double* out, int64_t capacity) {
  if (cudaSetDevice(device_) != cudaSuccess) return POVAR_ERR_CUDA;
  cudaStreamSynchronize(stream_);
  const std::string n(name ? name : "");
  const double* dsrc = nullptr;
  const int* isrc = nullptr;
  int64_t count = 0;
  const int D = dim_;
  if (n == "P") dsrc = d_.P, count = 12LL * C_;
  else if (n == "X") dsrc = d_.X, count = 4LL * L_;
  else if (n == "pose_scale") dsrc = d_.pose_scale, count = 12LL * C_;
  else if (n == "lm_scale") dsrc = d_.lm_scale, count = 4LL * L_;
  else if (n == "lm_hraw" || n == "lm_graw" || n == "hll_inv") {
    // by landmark for the caller: the landmarks of the sliced-ELL set keep these as lane-major planes
    // [slice][component][32], the others (more than 32 observations) by landmark
    const int K = n == "lm_hraw" ? 10 : (n == "lm_graw" ? 4 : 6);
    count = static_cast<int64_t>(K) * L_;
    if (!out) return count;
    if (capacity < count) {
      fail(POVAR_ERR_INVALID, "debug_read: buffer too small");
      return POVAR_ERR_INVALID;
    }
    const double* by_lm = K == 10 ? d_.lm_hraw : (K == 4 ? d_.lm_graw : d_.hll_inv);
    const double* planes = K == 10 ? d_.sell_hraw : (K == 4 ? d_.sell_graw : d_.sell_hinv);
    const size_t slots = static_cast<size_t>(kSellWidth) * d_.ix.num_slices;
    std::vector<double> hp(slots * K);
    std::vector<int> hlm(slots);
    if (cudaMemcpy(out, by_lm, sizeof(double) * count, cudaMemcpyDeviceToHost) != cudaSuccess) return POVAR_ERR_CUDA;
    if (slots > 0) {
      if (cudaMemcpy(hp.data(), planes, sizeof(double) * hp.size(), cudaMemcpyDeviceToHost) != cudaSuccess ||
          cudaMemcpy(hlm.data(), d_.ix.sell_lm, sizeof(int) * slots, cudaMemcpyDeviceToHost) != cudaSuccess) {
        return POVAR_ERR_CUDA;
      }
    }
    for (size_t i = 0; i < slots; ++i) {
      if (hlm[i] < 0) continue;
      const size_t sl = i / kSellWidth, lane = i % kSellWidth;
      for (int k = 0; k < K; ++k) out[static_cast<size_t>(hlm[i]) * K + k] = hp[(sl * K + k) * kSellWidth + lane];
    }
    return count;
  }
  else if (n == "lm_rec") dsrc = d_.lm_rec, count = static_cast<int64_t>(kLmRec) * L_;
  else if (n == "kron") dsrc = d_.kron, count = static_cast<int64_t>(kKron) * C_;
  else if (n == "b_mat") dsrc = d_.Bmat, count = 144LL * C_;
  else if (n == "b_inv") dsrc = d_.Binv, count = 144LL * C_;
  else if (n == "b") dsrc = d_.b, count = static_cast<int64_t>(D) * C_;
  else if (n == "inc") dsrc = d_.vec_acc, count = static_cast<int64_t>(D) * C_;
  else if (n == "cam_raw") dsrc = d_.cam_raw, count = 12LL * C_;
  else if (n == "vec_y") dsrc = d_.vec_y, count = 12LL * C_;
  else if (n == "lm_ptr") isrc = d_.ix.lm_ptr, count = L_ + 1;
  else if (n == "obs_cam") isrc = d_.ix.obs_cam, count = nnz_;
  else if (n == "obs_lm") isrc = d_.ix.obs_lm, count = nnz_;
  else if (n == "cam_ptr") isrc = d_.ix.cam_ptr, count = C_ + 1;
  else if (n == "csc_lm") isrc = d_.ix.csc_lm, count = nnz_;
  else if (n == "item_ptr") isrc = d_.ix.item_ptr, count = d_.ix.num_items + 1;
  else if (n == "item_cam") isrc = d_.ix.item_cam, count = d_.ix.num_items;
  else if (n == "slice_ptr") isrc = d_.ix.slice_ptr, count = d_.ix.num_slices + 1;
  else if (n == "sell_lm") isrc = d_.ix.sell_lm, count = static_cast<int64_t>(kSellWidth) * d_.ix.num_slices;
  else if (n == "sell_cam") isrc = d_.ix.sell_cam, count = d_.ix.sell_slots;
  else if (n == "sell_cam_e0") isrc = d_.ix.sell_cam_e0, count = d_.ix.sell_slots;
  else if (n == "sell_max_deg") {
    if (out && capacity >= 1) out[0] = d_.ix.sell_max_deg;
    return 1;
  }
  else if (n == "obs_slot") isrc = d_.ix.obs_slot, count = nnz_;
  else if (n == "chol_perm" || n == "chol_tiles") {   // tile-sparse CHOLESKY: 0 elements on the dense path
    count = !chol_tiled_active_ ? 0 : (n == "chol_tiles" ? 1 : C_);
    if (!out || count == 0) return count;
    if (capacity < count) {
      fail(POVAR_ERR_INVALID, "debug_read: buffer too small");
      return POVAR_ERR_INVALID;
    }
    if (n == "chol_tiles") out[0] = static_cast<double>(chol_pat_.tiles());
    else for (int c = 0; c < C_; ++c) out[c] = chol_pat_.perm[c];
    return count;
  }
  else {
    fail(POVAR_ERR_INVALID, "debug_read: unknown array '" + n + "'");
    return POVAR_ERR_INVALID;
  }
  if (!out) return count;
  if (capacity < count) {
    fail(POVAR_ERR_INVALID, "debug_read: buffer too small");
    return POVAR_ERR_INVALID;
  }
  if (dsrc) {
    if (cudaMemcpy(out, dsrc, sizeof(double) * count, cudaMemcpyDeviceToHost) != cudaSuccess) return POVAR_ERR_CUDA;
  } else {
    std::vector<int> h(count);
    if (cudaMemcpy(h.data(), isrc, sizeof(int) * count, cudaMemcpyDeviceToHost) != cudaSuccess) return POVAR_ERR_CUDA;
    for (int64_t i = 0; i < count; ++i) out[i] = h[i];
  }
  return count;
}

// E0 x with the current linearisation and the Hll^-1 of the last solve
int Engine::right_mul_e0(bool joint, const double* x, double* out) {
  PV_CUDA(cudaSetDevice(device_));
  if (static_cast<int>(joint) != joint_lin_ || !have_solve_) {
    return fail(POVAR_ERR_INVALID, "right_mul_e0: needs a matching linearize + solve");
  }
  const size_t n = static_cast<size_t>(C_) * (joint ? 11 : 12);
  PV_CUDA(cudaMemcpyAsync(d_.vec_x, x, sizeof(double) * n, cudaMemcpyHostToDevice, stream_));
  launch_make_y(d_, joint, d_.vec_x, d_.vec_y, lc());
  {
    const int rc = e0_product(joint, false, false);
    if (rc != POVAR_OK) return rc;
  }
  launch_e0_finish(d_, joint, d_.vec_x, lc());
  PV_CUDA(cudaGetLastError());
  PV_CUDA(cudaMemcpyAsync(out, d_.vec_x, sizeof(double) * n, cudaMemcpyDeviceToHost, stream_));
  PV_CUDA(cudaStreamSynchronize(stream_));
  return POVAR_OK;
}

// `terms` full power-series terms (landmark pass, camera pass, item reduction, allreduce, B^-1
// and norms) on the current linearisation, no early exit: the SpMV measurement of bench.py.
int Engine::bench_power_terms(bool joint, int terms, double* seconds_per_term) {
  PV_CUDA(cudaSetDevice(device_));
  if (static_cast<int>(joint) != joint_lin_ || !have_solve_) {
    return fail(POVAR_ERR_INVALID, "bench_power_terms: needs a matching linearize + solve");
  }
  if (terms <= 0) return fail(POVAR_ERR_INVALID, "bench_power_terms: terms must be positive");
  launch_finish_b(d_, joint, lc());
  launch_series_start(d_, -1.0, terms, lc());
  PV_CUDA(cudaEventRecord(ev_[0], stream_));
  for (int i = 1; i <= terms; ++i) {
    const int rc = e0_product(joint, true, term_mode() != kTermRaw);
    if (rc != POVAR_OK) return rc;
    launch_series_term(d_, joint, i, /*eta=*/-1.0, /*r_tolerance=*/-1.0, term_mode(), exchange(), lc());
  }
  PV_CUDA(cudaEventRecord(ev_[1], stream_));
  PV_CUDA(cudaGetLastError());
  PV_CUDA(cudaStreamSynchronize(stream_));
  if (seconds_per_term) *seconds_per_term = elapsed(ev_[0], ev_[1]) / terms;
  return POVAR_OK;
}

// average device time of each kernel of a power-series term, launched `reps` times back to back:
// [0] landmark half, [1] camera half, [2] item reduction, [3] B^-1 / accumulate / norms / test
int Engine::bench_power_kernels(bool joint, int reps, double* seconds) {
  PV_CUDA(cudaSetDevice(device_));
  if (static_cast<int>(joint) != joint_lin_ || !have_solve_) {
    return fail(POVAR_ERR_INVALID, "bench_power_kernels: needs a matching linearize + solve");
  }
  if (reps <= 0 || !seconds) return fail(POVAR_ERR_INVALID, "bench_power_kernels: bad arguments");
  launch_finish_b(d_, joint, lc());
  launch_series_start(d_, -1.0, reps, lc());
  for (int k = 0; k < 4; ++k) {
    PV_CUDA(cudaEventRecord(ev_[0], stream_));
    for (int i = 0; i < reps; ++i) {
      switch (k) {
        case 0:
          launch_e0_landmark_v2(d_, mp_, joint, true, lc());
          break;
        case 1:
          launch_passB_e0_v2(d_, mp_, joint, true, lc());
          break;
        case 2: launch_reduce_items(d_, d_.item_part, 12, d_.cam_raw, true, lc()); break;
        default: launch_series_term(d_, joint, i + 1, -1.0, -1.0, term_mode(), exchange(), lc()); break;
      }
    }
    PV_CUDA(cudaEventRecord(ev_[1], stream_));
    PV_CUDA(cudaGetLastError());
    PV_CUDA(cudaStreamSynchronize(stream_));
    seconds[k] = elapsed(ev_[0], ev_[1]) / reps;
  }
  return POVAR_OK;
}


// ---------------------------------------------------------------------------------------------
// povar_bundle_adjust_async: the two LM loops of host/lm_driver.cpp as ONE CUDA graph on the handle's stream.
//
//   step 1:  init_varproj -> cost -> k_lm_begin
//            WHILE(run): k_lm_top; IF(lin) { linearize }; solve -> backup -> apply -> cost -> k_lm_decide;
//                        IF(restore) { restore }
//            k_lm_end_step
//   IF(step 1 ok): to_homogeneous -> cost -> k_lm_begin -> the same WHILE for step 2 -> k_lm_end_step
//   k_lm_finish
//
// The bodies are stream captures of the host route's own enqueue functions (capturing_ set): the damping comes from
// the control block (lambda_dev_), the CG iterations from a device counter, the events become %globaltimer stamps
// (mark), the power series and the CG loop become nested WHILE nodes, CHOLESKY's read-back a kernel.  Nothing in a
// capture allocates or synchronises: build_solve_graph makes every allocation the host route makes lazily first.

cudaError_t Engine::mark(int k) {
  if (capturing_) {
    launch_lm_stamp(&lm_->stamp[k], lc());
    return cudaGetLastError();
  }
  return cudaEventRecord(ev_[k], stream_);
}

// what `body` enqueues on stream_, captured into a new graph (cap_graph_ while it runs) and instantiated into *exec.
// Nothing runs: launches_ is left as it was.
int Engine::capture_graph(void** exec, const std::function<int()>& body) {
  const long long before = launches_;
  cudaGraph_t graph = nullptr;
  PV_CUDA(cudaGraphCreate(&graph, 0));
  cap_graph_ = graph;
  int rc = check(cudaStreamBeginCaptureToGraph(stream_, graph, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed),
                 "cudaStreamBeginCaptureToGraph");
  if (rc == POVAR_OK) rc = body();
  cudaGraph_t same = nullptr;
  if (rc == POVAR_OK) rc = check(cudaStreamEndCapture(stream_, &same), "cudaStreamEndCapture");
  cudaGraphExec_t e = nullptr;
  if (rc == POVAR_OK) rc = check(cudaGraphInstantiate(&e, graph, 0), "cudaGraphInstantiate");
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (rc != POVAR_OK && cudaStreamIsCapturing(stream_, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone) {
    cudaStreamEndCapture(stream_, &same);
  }
  cudaGraphDestroy(graph);
  cap_graph_ = nullptr;
  launches_ = before;
  if (rc != POVAR_OK) {
    cudaGetLastError();
    return rc;
  }
  *exec = e;
  return POVAR_OK;
}

int Engine::new_cond(unsigned long long* h) {
  cudaGraphConditionalHandle c = 0;
  PV_CUDA(cudaGraphConditionalHandleCreate(&c, static_cast<cudaGraph_t>(cap_graph_), 0, 0));
  *h = static_cast<unsigned long long>(c);
  return POVAR_OK;
}

// a conditional node at the capture position of stream_ whose body `body` captures; the capture of the enclosing graph
// continues behind the node
int Engine::capture_cond(int type, unsigned long long h, const std::function<int()>& body) {
  cudaGraph_t g = static_cast<cudaGraph_t>(cap_graph_);
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  const cudaGraphNode_t* deps = nullptr;
  size_t num_deps = 0;
  PV_CUDA(cudaStreamGetCaptureInfo(stream_, &st, nullptr, nullptr, &deps, &num_deps));
  if (st != cudaStreamCaptureStatusActive) return fail(POVAR_ERR_CUDA, "stream capture is not active");
  cudaGraphNodeParams params{};
  params.type = cudaGraphNodeTypeConditional;
  params.conditional.handle = static_cast<cudaGraphConditionalHandle>(h);
  params.conditional.type = static_cast<cudaGraphConditionalNodeType>(type);
  params.conditional.size = 1;
  cudaGraphNode_t node = nullptr;
  PV_CUDA(cudaGraphAddNode(&node, g, deps, num_deps, &params));
  cudaGraph_t same = nullptr;
  PV_CUDA(cudaStreamEndCapture(stream_, &same));
  cap_graph_ = params.conditional.phGraph_out[0];
  PV_CUDA(cudaStreamBeginCaptureToGraph(stream_, params.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                        cudaStreamCaptureModeRelaxed));
  const int rc = body();
  const cudaError_t e = cudaStreamEndCapture(stream_, &same);
  cap_graph_ = g;
  if (rc != POVAR_OK) return rc;
  PV_CUDA(e);
  PV_CUDA(cudaStreamBeginCaptureToGraph(stream_, g, &node, nullptr, 1, cudaStreamCaptureModeRelaxed));
  return POVAR_OK;
}

// the power series as prefix + WHILE(term), into the graph being captured: the series graph of enqueue_series, or a
// node of the solve graph
int Engine::capture_series(bool joint) {
  const int m = opt_.power_sc_iterations;
  unsigned long long h = 0;
  const int rc = new_cond(&h);
  if (rc != POVAR_OK) return rc;
  SeriesLoop loop;
  loop.handle = h;
  loop.active = 1;
  loop.max_terms = m;
  launch_finish_b(d_, joint, lc());
  launch_series_start(d_, opt_.r_tolerance, m, lc(), loop);
  return capture_cond(cudaGraphCondTypeWhile, h, [&]() -> int {
    const int rc2 = e0_product(joint, true, true);
    launch_series_term(d_, joint, 0, opt_.eta, opt_.r_tolerance, term_mode(), exchange(), lc(), loop);
    return rc2;
  });
}

// one LM loop (run_step): iteration 0, then WHILE(run) over the trials; `ok`: the IF node of step 2 (step 1 only)
int Engine::capture_lm_step(const povar_options& opt, bool joint, unsigned long long ok) {
  const int step = joint ? 2 : 1;
  const int max_iter = joint ? opt.max_num_iterations_step_2 : opt.max_num_iterations_step_1;
  PV_CUDA(mark(0));
  int rc = enqueue_cost(joint, opt.alpha);
  if (rc != POVAR_OK) return rc;
  PV_CUDA(mark(1));
  LmConds h;
  rc = new_cond(&h.run);
  if (rc != POVAR_OK) return rc;
  launch_lm_begin(lm_, d_.trial_out, opt, step, lm_log_, lm_cap_, h, lc());
  rc = capture_cond(cudaGraphCondTypeWhile, h.run, [&]() -> int {
    LmConds b = h;
    int rc2 = new_cond(&b.lin);
    if (rc2 == POVAR_OK) rc2 = new_cond(&b.restore);
    if (rc2 != POVAR_OK) return rc2;
    launch_lm_top(lm_, b, lc());
    rc2 = capture_cond(cudaGraphCondTypeIf, b.lin, [&]() { return linearize(joint, opt.alpha, true); });
    if (rc2 != POVAR_OK) return rc2;
    rc2 = enqueue_trial(joint, opt.alpha, 0.0);   // the damping comes from lm_->loop.lambda
    if (rc2 != POVAR_OK) return rc2;
    PV_CUDA(mark(4));
    launch_lm_decide(lm_, d_.trial_out, d_.ctl, opt, step, lm_power_step(opt, joint), lm_log_, lm_cap_, b, lc());
    return capture_cond(cudaGraphCondTypeIf, b.restore, [&]() { return restore(0); });
  });
  if (rc != POVAR_OK) return rc;
  launch_lm_end_step(lm_, step, max_iter, ok, lc());
  PV_CUDA(cudaGetLastError());
  return POVAR_OK;
}

int Engine::build_solve_graph(const povar_options& opt) {
  // every allocation the host route makes on first use (linearize, solve_cholesky), and the control block and log
  for (const bool joint : {true, false}) {
    const int rc = alloc_lin_buffers(joint);
    if (rc != POVAR_OK) return rc;
  }
  if (opt_.solver_type_step_1 == POVAR_CHOLESKY) {
    bool tiled = false;
    const int rc = alloc_cholesky(&tiled);
    if (rc != POVAR_OK) return rc;
  }
  if (!lm_) {
    PV_ALLOC(lm_, 1);
    PV_ALLOC(lm_sum_, 1);
    PV_ALLOC(lm_status_, 1);
  }
  const long long cap = 2LL + std::max(0, opt.max_num_iterations_step_1) + std::max(0, opt.max_num_iterations_step_2);
  if (cap > std::numeric_limits<int>::max()) return fail(POVAR_ERR_INVALID, "too many iterations");
  if (cap > lm_cap_) {
    PV_ALLOC(lm_log_, static_cast<size_t>(cap));
    lm_cap_ = static_cast<int>(cap);
  }
  capturing_ = true;
  lambda_dev_ = &lm_->loop.lambda;
  const int rc = capture_graph(&solve_graph_, [&]() -> int {
    launch_lm_stamp(&lm_->t_start, lc());
    launch_lm_stamp(&lm_->t_it, lc());
    int rc2 = init_varproj(opt.alpha);   // :302-304
    unsigned long long ok = kNoCond;
    if (rc2 == POVAR_OK) rc2 = new_cond(&ok);
    if (rc2 == POVAR_OK) rc2 = capture_lm_step(opt, false, ok);
    if (rc2 == POVAR_OK) {
      rc2 = capture_cond(cudaGraphCondTypeIf, ok, [&]() -> int {
        const int rc3 = to_homogeneous();   // create_homogeneous_landmark, :544-553
        if (rc3 != POVAR_OK) return rc3;
        launch_lm_stamp(&lm_->t_it, lc());
        return capture_lm_step(opt, true, kNoCond);
      });
    }
    if (rc2 != POVAR_OK) return rc2;
    launch_lm_finish(lm_, lm_cap_, lm_sum_, lm_status_, lc());
    return POVAR_OK;
  });
  capturing_ = false;
  lambda_dev_ = nullptr;
  if (rc != POVAR_OK) return rc;
  solve_opt_ = opt;
  solve_window_ = d_.debug_window_cams;
  solve_storage_ = chol_storage_;
  return POVAR_OK;
}

int Engine::bundle_adjust_async(const povar_options& opt, povar_iteration* iterations, int max_iterations,
                                povar_solve_summary* summary, int* status, cudaStream_t caller) {
  PV_CUDA(cudaSetDevice(device_));
  if (max_iterations > 0 && check_device_ptr(iterations, "iterations") != POVAR_OK) return POVAR_ERR_INVALID;
  if (check_device_ptr(summary, "summary") != POVAR_OK) return POVAR_ERR_INVALID;
  if (check_device_ptr(status, "status") != POVAR_OK) return POVAR_ERR_INVALID;
  if (world_ > 1 && !peer_ok_) {
    return fail(POVAR_ERR_UNSUPPORTED, "povar_bundle_adjust_async: the reductions of this handle go through "
                                       "ncclAllReduce, which is not captured into graphs");
  }
  const bool same = solve_graph_ && std::memcmp(&solve_opt_, &opt, sizeof(opt)) == 0 &&
                    solve_window_ == d_.debug_window_cams && solve_storage_ == chol_storage_;
  if (!same) {
    if (solve_graph_) {
      PV_CUDA(cudaStreamSynchronize(stream_));   // a launch of the old graph may still be in flight
      cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(solve_graph_));
      solve_graph_ = nullptr;
    }
    const int rc = build_solve_graph(opt);
    if (rc != POVAR_OK) return rc;
  }
  int rc = wait_for(stream_, caller);
  if (rc != POVAR_OK) return rc;
  PV_CUDA(cudaGraphLaunch(static_cast<cudaGraphExec_t>(solve_graph_), stream_));
  launch_lm_clip(lm_sum_, max_iterations, LaunchCfg{stream_, nullptr});
  const int n = std::min(max_iterations, lm_cap_);
  if (n > 0) {
    PV_CUDA(cudaMemcpyAsync(iterations, lm_log_, sizeof(povar_iteration) * static_cast<size_t>(n),
                            cudaMemcpyDeviceToDevice, stream_));
  }
  PV_CUDA(cudaMemcpyAsync(summary, lm_sum_, sizeof(povar_solve_summary), cudaMemcpyDeviceToDevice, stream_));
  PV_CUDA(cudaMemcpyAsync(status, lm_status_, sizeof(int), cudaMemcpyDeviceToDevice, stream_));
  PV_CUDA(cudaGetLastError());
  return wait_for(caller, stream_);
}

}  // namespace povar
