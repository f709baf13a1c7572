// CHOLESKY on tile-sparse storage: the camera order and the symbolic factorisation at the level of 64x64 tiles.
//
//   order      reverse Cuthill-McKee on the co-visibility graph of the blocks (cameras): every connected component
//              from a pseudo-peripheral node (George-Liu), neighbours visited by ascending degree, ties by index;
//              the concatenated Cuthill-McKee sequence is reversed.  Block c sits at position perm[c] and owns rows
//              block * perm[c] ... block * perm[c] + block - 1 (a range that may straddle two tiles).
//   pattern    tile (I, J), I >= J, of S is stored when two coupled blocks (or a block with itself) own rows of
//              tiles I and J.
//   symbolic   right-looking and exact for any pattern: the stored rows below tile k of column k are OR-ed into
//              every column J among them (the tiles the update C(I, J) -= A(I, k) A(J, k)^T writes).  A loop closure
//              costs memory, never correctness.
// Host threads split the adjacency and the pattern of S by rows; every row is written by one thread, so the result
// does not depend on their number.
#include <algorithm>
#include <cstdint>
#include <thread>
#include <vector>

#include "../povar_internal.h"

namespace povar {

namespace {

constexpr int kTile = 64;

template <typename F>
void parallel_rows(int rows, int threads, F&& body) {   // body(begin, end)
  if (threads <= 1 || rows < 2) {
    body(0, rows);
    return;
  }
  std::vector<std::thread> pool;
  for (int t = 1; t < threads; ++t) {
    pool.emplace_back([&body, t, threads, rows] {
      body(static_cast<int>(static_cast<long long>(rows) * t / threads),
           static_cast<int>(static_cast<long long>(rows) * (t + 1) / threads));
    });
  }
  body(0, static_cast<int>(rows / threads));
  for (auto& th : pool) th.join();
}

// breadth-first level structure from r inside the nodes not yet ordered; returns the eccentricity and the last level
int bfs_levels(int r, const std::vector<std::vector<int>>& adj, const std::vector<char>& ordered, std::vector<int>& stamp,
               int tag, std::vector<int>* last) {
  std::vector<int> cur{r}, next;
  stamp[r] = tag;
  int ecc = 0;
  for (;;) {
    next.clear();
    for (int v : cur) {
      for (int w : adj[v]) {
        if (!ordered[w] && stamp[w] != tag) {
          stamp[w] = tag;
          next.push_back(w);
        }
      }
    }
    if (next.empty()) break;
    ++ecc;
    cur.swap(next);
  }
  *last = cur;
  return ecc;
}

}  // namespace

void chol_symbolic(int nb, int block, const std::vector<unsigned int>& bits, int threads, CholPattern* out) {
  CholPattern& P = *out;
  P = CholPattern();
  P.nb = nb;
  P.block = block;
  P.n_pad = (block * nb + kTile - 1) / kTile * kTile;
  P.T = P.n_pad / kTile;
  const int T = P.T;
  const size_t words = (static_cast<size_t>(nb) + 31) / 32;
  if (threads <= 0) {
    const unsigned hw = std::thread::hardware_concurrency();
    threads = static_cast<long long>(nb) * nb < (1LL << 22) ? 1 : static_cast<int>(std::min<unsigned>(hw ? hw : 1, 16));
  }

  // ---- adjacency (neighbours ascending, self excluded)
  std::vector<std::vector<int>> adj(nb);
  parallel_rows(nb, threads, [&](int b0, int b1) {
    for (int a = b0; a < b1; ++a) {
      const unsigned int* row = bits.data() + static_cast<size_t>(a) * words;
      for (size_t w = 0; w < words; ++w) {
        for (unsigned int m = row[w]; m != 0; m &= m - 1) {
          const int b = static_cast<int>(w * 32) + __builtin_ctz(m);
          if (b != a) adj[a].push_back(b);
        }
      }
    }
  });

  // ---- reverse Cuthill-McKee
  std::vector<char> ordered(nb, 0);
  std::vector<int> stamp(nb, -1), order;
  order.reserve(nb);
  int tag = 0;
  auto fewer = [&](int x, int y) {
    return adj[x].size() != adj[y].size() ? adj[x].size() < adj[y].size() : x < y;
  };
  for (int s = 0; s < nb; ++s) {
    if (ordered[s]) continue;
    // George-Liu: from the component's first node, move to a node of least degree in the last level while that
    // lengthens the level structure
    int r = s;
    std::vector<int> last;
    int ecc = bfs_levels(r, adj, ordered, stamp, tag++, &last);
    for (;;) {
      const int x = *std::min_element(last.begin(), last.end(), fewer);
      std::vector<int> last_x;
      const int ecc_x = bfs_levels(x, adj, ordered, stamp, tag++, &last_x);
      if (ecc_x <= ecc) break;
      r = x;
      ecc = ecc_x;
      last.swap(last_x);
    }
    size_t head = order.size();
    order.push_back(r);
    ordered[r] = 1;
    std::vector<int> nbr;
    while (head < order.size()) {
      const int v = order[head++];
      nbr.clear();
      for (int w : adj[v]) {
        if (!ordered[w]) {
          ordered[w] = 1;
          nbr.push_back(w);
        }
      }
      std::sort(nbr.begin(), nbr.end(), fewer);
      order.insert(order.end(), nbr.begin(), nbr.end());
    }
  }
  P.perm.assign(nb, 0);
  for (int i = 0; i < nb; ++i) P.perm[order[i]] = nb - 1 - i;
  std::vector<int> at(nb);   // block at position p
  for (int c = 0; c < nb; ++c) at[P.perm[c]] = c;

  // ---- tile pattern of S, by tile row (bit J of row I: tile (I, J), J <= I)
  const size_t tw = (static_cast<size_t>(T) + 63) / 64;
  std::vector<uint64_t> rowbits(static_cast<size_t>(T) * tw, 0);
  parallel_rows(T, threads, [&](int i0, int i1) {
    for (int I = i0; I < i1; ++I) {
      uint64_t* rb = rowbits.data() + static_cast<size_t>(I) * tw;
      rb[I >> 6] |= 1ull << (I & 63);   // every diagonal tile (the padding rows get the identity)
      const int p0 = I * kTile / block, p1 = std::min(nb - 1, ((I + 1) * kTile - 1) / block);
      for (int p = p0; p <= p1; ++p) {
        const int a = at[p];
        auto add = [&](int pb) {
          const int j0 = pb * block / kTile, j1 = (pb * block + block - 1) / kTile;
          for (int J = j0; J <= std::min(j1, I); ++J) rb[J >> 6] |= 1ull << (J & 63);
        };
        add(p);
        for (int b : adj[a]) {
          if (P.perm[b] < p) add(P.perm[b]);
        }
      }
    }
  });

  // ---- symbolic factorisation on column bitsets (bit I of column J: tile (I, J), I >= J)
  std::vector<uint64_t> colbits(static_cast<size_t>(T) * tw, 0);
  for (int I = 0; I < T; ++I) {
    const uint64_t* rb = rowbits.data() + static_cast<size_t>(I) * tw;
    for (size_t w = 0; w < tw; ++w) {
      for (uint64_t m = rb[w]; m != 0; m &= m - 1) {
        const int J = static_cast<int>(w * 64) + __builtin_ctzll(m);
        colbits[static_cast<size_t>(J) * tw + (I >> 6)] |= 1ull << (I & 63);
      }
    }
  }
  for (int k = 0; k < T; ++k) {
    const uint64_t* ck = colbits.data() + static_cast<size_t>(k) * tw;
    for (size_t w = static_cast<size_t>(k) >> 6; w < tw; ++w) {
      uint64_t m = ck[w];
      if (w == (static_cast<size_t>(k) >> 6)) m &= ~((2ull << (k & 63)) - 1);   // rows below k
      for (; m != 0; m &= m - 1) {
        const int J = static_cast<int>(w * 64) + __builtin_ctzll(m);
        uint64_t* cj = colbits.data() + static_cast<size_t>(J) * tw;
        const size_t w0 = static_cast<size_t>(J) >> 6;
        cj[w0] |= ck[w0] & ~((1ull << (J & 63)) - 1);   // rows >= J
        for (size_t v = w0 + 1; v < tw; ++v) cj[v] |= ck[v];
      }
    }
  }

  // ---- stored tiles: slots in column order, the column lists, the row lists and the slot map
  P.col_ptr.assign(T + 1, 0);
  P.slot.assign(static_cast<size_t>(T) * T, -1);
  std::vector<int> row_cnt(T, 0);
  for (int J = 0; J < T; ++J) {
    const uint64_t* cj = colbits.data() + static_cast<size_t>(J) * tw;
    for (size_t w = 0; w < tw; ++w) {
      for (uint64_t m = cj[w]; m != 0; m &= m - 1) {
        const int I = static_cast<int>(w * 64) + __builtin_ctzll(m);
        P.slot[static_cast<size_t>(I) * T + J] = static_cast<int>(P.col_row.size());
        P.col_row.push_back(I);
        ++row_cnt[I];
      }
    }
    P.col_ptr[J + 1] = static_cast<int>(P.col_row.size());
  }
  P.row_ptr.assign(T + 1, 0);
  for (int I = 0; I < T; ++I) P.row_ptr[I + 1] = P.row_ptr[I] + row_cnt[I];
  P.row_col.assign(P.col_row.size(), 0);
  std::vector<int> fill(P.row_ptr.begin(), P.row_ptr.end() - 1);
  for (int J = 0; J < T; ++J) {   // columns ascending: every row list comes out sorted, its diagonal last
    for (int q = P.col_ptr[J]; q < P.col_ptr[J + 1]; ++q) P.row_col[fill[P.col_row[q]]++] = J;
  }
}

void covisibility_host(int num_cams, int num_lms, const int64_t* lm_ptr, const int32_t* obs_cam,
                       std::vector<unsigned int>* bits) {
  const size_t words = (static_cast<size_t>(num_cams) + 31) / 32;
  bits->assign(static_cast<size_t>(num_cams) * words, 0u);
  for (int l = 0; l < num_lms; ++l) {
    for (int64_t i = lm_ptr[l]; i < lm_ptr[l + 1]; ++i) {
      for (int64_t j = lm_ptr[l]; j < lm_ptr[l + 1]; ++j) {
        const int a = obs_cam[i], b = obs_cam[j];
        (*bits)[static_cast<size_t>(a) * words + (b >> 5)] |= 1u << (b & 31);
      }
    }
  }
}

}  // namespace povar
