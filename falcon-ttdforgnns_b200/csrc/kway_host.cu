// kway_host.cu -- multilevel k-way graph partitioner on the HOST (SURVEY 8f-3).
//
// replaces: dgl.reorder_graph(graph, 'metis', permute_config={'k': k}) / dgl.metis_partition as called at
//           graphloader.py:370 (three METIS reorders in a row), :377, :440 (DGL 2.1 -> libmetis 5.1,
//           un-vendored: neither is part of the reference tree or of this image).
//
// METIS is host code in the reference too (offline preprocessing before the first epoch), so this stays
// on the host: no kernel, every pointer of ttg_partition_kway is HOST memory.  It follows the published
// multilevel k-way scheme (Karypis & Kumar, "Multilevel k-way partitioning scheme for irregular graphs",
// JPDC 1998), not METIS' sources:
//
//   symmetrise   the in-neighbour CSR becomes an undirected weighted graph (weight = number of
//                directed edges between the pair, self loops dropped) -- what DGL does before it
//                calls METIS (to_bidirected);
//   coarsen      heavy-edge matching in a seeded random vertex order (a vertex joins its unmatched
//                neighbour over the heaviest edge, bounded vertex weight), then a two-hop pass that
//                pairs unmatched low-degree vertices hanging off the same neighbour (power-law
//                graphs: the leaves of a hub); contraction merges the adjacency lists through a
//                marker array; stops at max(30 k, 256) vertices or when a level shrinks by < 5 %;
//   initial      k parts grown one after the other on the coarsest graph: the next vertex is the
//                frontier vertex with the heaviest connection to the growing part (lazy max-heap),
//                until the part holds its share of the remaining weight; eight seeded trials, each
//                refined on the coarsest graph, the smallest cut goes on;
//   uncoarsen    the partition is projected level by level and improved by greedy k-way refinement
//                (a vertex moves to the adjacent part with the largest cut gain that has room, ties
//                towards the lighter part; only vertices next to a move are revisited), preceded
//                by a balancing sweep when a part is outside its bounds; the bounds are 1.3 x wider on
//                every level but the finest, which lets split communities flow together.
//
// The result is a k-way partition with every part at most ubfactor * ceil(n / k) and at least
// floor(n / k) / ubfactor vertices (the bounds METIS' ufactor sets) and a cut in METIS' league -- NOT METIS' partition: parity with DGL's
// order is unpinned (no METIS here to compare with), tests/test_partition_cpu.py checks the
// invariants, determinism and the cut on graphs with a known optimum.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <exception>
#include <new>
#include <numeric>
#include <queue>
#include <thread>
#include <utility>
#include <vector>

#include "common.cuh"
#include "../../include/ttg_b200.h"

namespace ttg {
namespace {

// TTG_KWAY_VERBOSE=1: seconds per phase on stderr
struct PhaseClock {
  bool on = getenv("TTG_KWAY_VERBOSE") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  void lap(const char* what, long long n, long long m) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "kway: %-22s %9lld vertices %11lld edges %7.2f s\n", what, n, m,
            std::chrono::duration<double>(now - t).count());
    t = now;
  }
};

// Host threads for the data-parallel phase (symmetrise: 7.7 -> 4.1 s at 60 M edges on eight threads); the
// matching, the contraction, the grown parts and the refinement run on one.  The partition does not depend on
// the number of threads (the symmetrised lists are sorted).  TTG_KWAY_THREADS overrides min(16, hardware threads).
int host_threads() {
  if (const char* e = getenv("TTG_KWAY_THREADS")) return std::max(1, atoi(e));
  const unsigned hw = std::thread::hardware_concurrency();
  return (int)std::min(16u, std::max(1u, hw));
}

// fn(thread, chunk, begin, end) over [0, n) in chunks handed out dynamically
template <class F>
void parallel_chunks(int64_t n, int64_t chunk, F fn) {
  const int64_t nchunks = (n + chunk - 1) / chunk;
  const int nt = (int)std::min<int64_t>(host_threads(), nchunks);
  if (nt <= 1) {
    for (int64_t c = 0; c < nchunks; ++c) fn(0, c, c * chunk, std::min(n, (c + 1) * chunk));
    return;
  }
  std::atomic<int64_t> next{0};
  std::atomic<bool> failed{false};
  std::vector<std::thread> pool;
  for (int t = 0; t < nt; ++t)
    pool.emplace_back([&, t]() {
      try {
        for (int64_t c; (c = next.fetch_add(1)) < nchunks;) fn(t, c, c * chunk, std::min(n, (c + 1) * chunk));
      } catch (...) {
        failed = true;
      }
    });
  for (auto& th : pool) th.join();
  if (failed) throw std::bad_alloc();
}

struct WGraph {
  int32_t n = 0;
  std::vector<int64_t> xadj;   // n + 1
  std::vector<int32_t> adj;    // neighbours
  std::vector<int32_t> adjw;   // edge weights
  std::vector<int32_t> vw;     // vertex weights
};

struct Rng {   // splitmix64: the partition depends on the seed only
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed + 0x9e3779b97f4a7c15ull) {}
  uint64_t next() {
    uint64_t z = (s += 0x9e3779b97f4a7c15ull);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
  }
  uint32_t below(uint32_t n) { return (uint32_t)((next() >> 32) * (uint64_t)n >> 32); }
};

void random_order(int32_t n, Rng& rng, std::vector<int32_t>& order) {
  order.resize(n);
  std::iota(order.begin(), order.end(), 0);
  for (int32_t i = n - 1; i > 0; --i) std::swap(order[i], order[rng.below((uint32_t)i + 1)]);
}

// in-neighbour CSR (possibly directed, with duplicates and self loops) -> undirected weighted graph
void symmetrise(int64_t n, const int64_t* indptr, const int32_t* indices, WGraph& g) {
  g.n = (int32_t)n;
  g.xadj.assign(n + 1, 0);
  // degrees and the fill of both directions with relaxed atomic counters: the order inside a vertex's segment
  // depends on the threads, the sort below removes that again
  int64_t* deg = g.xadj.data() + 1;
  parallel_chunks(n, 16384, [&](int, int64_t, int64_t v0, int64_t v1) {
    for (int64_t v = v0; v < v1; ++v) {
      int64_t own = 0;
      for (int64_t e = indptr[v]; e < indptr[v + 1]; ++e) {
        const int32_t u = indices[e];
        if (u == v) continue;
        ++own;
        __atomic_fetch_add(deg + u, (int64_t)1, __ATOMIC_RELAXED);
      }
      __atomic_fetch_add(deg + v, own, __ATOMIC_RELAXED);
    }
  });
  for (int64_t v = 0; v < n; ++v) g.xadj[v + 1] += g.xadj[v];
  std::vector<int32_t> raw(g.xadj[n]);
  std::vector<int64_t> pos(g.xadj.begin(), g.xadj.end() - 1);
  parallel_chunks(n, 16384, [&](int, int64_t, int64_t v0, int64_t v1) {
    for (int64_t v = v0; v < v1; ++v)
      for (int64_t e = indptr[v]; e < indptr[v + 1]; ++e) {
        const int32_t u = indices[e];
        if (u == v) continue;
        raw[__atomic_fetch_add(&pos[v], (int64_t)1, __ATOMIC_RELAXED)] = u;
        raw[__atomic_fetch_add(&pos[u], (int64_t)1, __ATOMIC_RELAXED)] = (int32_t)v;
      }
  });
  // per vertex: sort, merge equal neighbours into one weighted edge (two passes: count, then write in place)
  std::vector<int64_t> nx(n + 1, 0);
  parallel_chunks(n, 16384, [&](int, int64_t, int64_t v0, int64_t v1) {
    for (int64_t v = v0; v < v1; ++v) {
      const int64_t b = g.xadj[v], e = g.xadj[v + 1];
      std::sort(raw.begin() + b, raw.begin() + e);
      int64_t uniq = 0;
      for (int64_t i = b; i < e; ++i) uniq += (i == b || raw[i] != raw[i - 1]);
      nx[v + 1] = uniq;
    }
  });
  for (int64_t v = 0; v < n; ++v) nx[v + 1] += nx[v];
  const int64_t out = nx[n];
  g.adj.resize(out);
  g.adjw.resize(out);
  parallel_chunks(n, 16384, [&](int, int64_t, int64_t v0, int64_t v1) {
    for (int64_t v = v0; v < v1; ++v) {
      const int64_t b = g.xadj[v], e = g.xadj[v + 1];
      int64_t o = nx[v];
      for (int64_t i = b; i < e;) {
        int64_t j = i + 1;
        while (j < e && raw[j] == raw[i]) ++j;
        g.adj[o] = raw[i];
        g.adjw[o] = (int32_t)(j - i);
        ++o;
        i = j;
      }
    }
  });
  g.xadj.swap(nx);
  g.vw.assign(n, 1);
}

// heavy-edge matching + two-hop pass; returns the number of coarse vertices and fills cmap
int32_t match_and_map(const WGraph& g, Rng& rng, int32_t maxvw, std::vector<int32_t>& cmap) {
  const int32_t n = g.n;
  std::vector<int32_t> match(n, -1), order;
  random_order(n, rng, order);
  for (int32_t v : order) {
    if (match[v] >= 0) continue;
    int32_t best = -1, bestw = 0;
    for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e) {
      const int32_t u = g.adj[e];
      if (match[u] < 0 && g.adjw[e] > bestw && g.vw[v] + g.vw[u] <= maxvw) {
        best = u;
        bestw = g.adjw[e];
      }
    }
    if (best >= 0) {
      match[v] = best;
      match[best] = v;
    }
  }
  // two-hop: unmatched vertices of small degree that share a neighbour are paired with each other
  constexpr int64_t kSmallDegree = 8;
  for (int32_t u : order) {
    int32_t pending = -1;
    for (int64_t e = g.xadj[u]; e < g.xadj[u + 1]; ++e) {
      const int32_t v = g.adj[e];
      if (match[v] >= 0 || g.xadj[v + 1] - g.xadj[v] > kSmallDegree) continue;
      if (pending < 0) {
        pending = v;
      } else if (g.vw[pending] + g.vw[v] <= maxvw) {
        match[pending] = v;
        match[v] = pending;
        pending = -1;
      }
    }
  }
  cmap.assign(n, -1);
  int32_t cn = 0;
  for (int32_t v = 0; v < n; ++v) {
    if (cmap[v] >= 0) continue;
    cmap[v] = cn;
    if (match[v] >= 0) cmap[match[v]] = cn;
    ++cn;
  }
  return cn;
}

void contract(const WGraph& g, const std::vector<int32_t>& cmap, int32_t cn, WGraph& c) {
  c.n = cn;
  c.vw.assign(cn, 0);
  // members of every coarse vertex (one or two)
  std::vector<int32_t> first(cn, -1), second(cn, -1);
  for (int32_t v = 0; v < g.n; ++v) {
    const int32_t cv = cmap[v];
    c.vw[cv] += g.vw[v];
    if (first[cv] < 0) first[cv] = v; else second[cv] = v;
  }
  // sequential: the merge is bound by random reads of cmap and of the marker array; eight host threads over
  // chunks of coarse vertices (per-thread markers, buffers copied behind each other) measured 2.2 s against 3.3 s
  // on the first level and no gain below it -- not worth the second copy of the coarse graph
  c.xadj.assign((size_t)cn + 1, 0);
  c.adj.clear();
  c.adjw.clear();
  c.adj.reserve(g.adj.size());
  c.adjw.reserve(g.adj.size());
  std::vector<int64_t> where(cn, -1);   // position of coarse neighbour x in the list being built
  for (int32_t cv = 0; cv < cn; ++cv) {
    const int64_t begin = (int64_t)c.adj.size();
    for (int m = 0; m < 2; ++m) {
      const int32_t v = m == 0 ? first[cv] : second[cv];
      if (v < 0) continue;
      for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e) {
        const int32_t cu = cmap[g.adj[e]];
        if (cu == cv) continue;
        if (where[cu] >= begin) {
          c.adjw[where[cu]] += g.adjw[e];
        } else {
          where[cu] = (int64_t)c.adj.size();
          c.adj.push_back(cu);
          c.adjw.push_back(g.adjw[e]);
        }
      }
    }
    c.xadj[cv + 1] = (int64_t)c.adj.size();
  }
  c.adj.shrink_to_fit();
  c.adjw.shrink_to_fit();
}

// k parts grown one after the other; part p takes total_left / parts_left of the weight
void initial_partition(const WGraph& g, int32_t k, Rng& rng, std::vector<int32_t>& part) {
  const int32_t n = g.n;
  part.assign(n, -1);
  int64_t left = 0;
  for (int32_t v = 0; v < n; ++v) left += g.vw[v];
  std::vector<int32_t> order;
  random_order(n, rng, order);
  size_t cursor = 0;                 // next candidate seed in the random order
  std::vector<int32_t> conn(n, 0);   // connection weight of an unassigned vertex to the growing part
  std::vector<int32_t> frontier_of_previous;
  for (int32_t p = 0; p < k; ++p) {
    const int64_t target = (left + (k - p) - 1) / (k - p);
    if (p == k - 1) {
      for (int32_t v = 0; v < n; ++v)
        if (part[v] < 0) part[v] = p;
      break;
    }
    int64_t w = 0;
    std::priority_queue<std::pair<int32_t, int32_t>> heap;   // (connection, vertex), lazily updated
    std::vector<int32_t> touched;
    auto take = [&](int32_t v) {
      part[v] = p;
      w += g.vw[v];
      for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e) {
        const int32_t u = g.adj[e];
        if (part[u] >= 0) continue;
        if (conn[u] == 0) touched.push_back(u);
        conn[u] += g.adjw[e];
        heap.emplace(conn[u], u);
      }
    };
    while (w < target) {
      int32_t v = -1;
      while (!heap.empty()) {
        const auto top = heap.top();
        heap.pop();
        if (part[top.second] < 0 && conn[top.second] == top.first) {
          v = top.second;
          break;
        }
      }
      if (v < 0) {   // a new seed: next to the parts made so far if possible, else the random order
        while (!frontier_of_previous.empty() && v < 0) {
          const int32_t c = frontier_of_previous.back();
          frontier_of_previous.pop_back();
          if (part[c] < 0) v = c;
        }
        while (v < 0 && cursor < order.size()) {
          const int32_t c = order[cursor++];
          if (part[c] < 0) v = c;
        }
        if (v < 0) break;   // nothing left
      }
      // the vertex that would overshoot the share by more than it is short now stays for a later part
      if (w > 0 && w + g.vw[v] - target > target - w) break;
      take(v);
    }
    left -= w;
    frontier_of_previous.clear();
    for (int32_t t : touched) {
      if (part[t] < 0) frontier_of_previous.push_back(t);
      conn[t] = 0;
    }
  }
}

struct Refiner {
  const WGraph& g;
  int32_t k;
  int64_t maxpw, minpw;
  std::vector<int32_t>& part;
  std::vector<int64_t> pw;
  std::vector<int32_t> conn;        // connection of the current vertex to every part (sparse use)
  std::vector<int32_t> seen_parts;

  Refiner(const WGraph& g_, int32_t k_, int64_t maxpw_, int64_t minpw_, std::vector<int32_t>& part_)
      : g(g_), k(k_), maxpw(maxpw_), minpw(minpw_), part(part_), pw(k_, 0), conn(k_, 0) {
    for (int32_t v = 0; v < g.n; ++v) pw[part[v]] += g.vw[v];
  }

  void gather(int32_t v) {
    seen_parts.clear();
    for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e) {
      const int32_t p = part[g.adj[e]];
      if (conn[p] == 0) seen_parts.push_back(p);
      conn[p] += g.adjw[e];
    }
  }
  void clear() {
    for (int32_t p : seen_parts) conn[p] = 0;
  }

  // parts above the upper bound hand vertices to adjacent parts with room (the best connected one),
  // else to the lightest part; parts below the lower bound take adjacent vertices from parts that
  // can spare them; a part that stays below it (nothing adjacent: an empty part) is filled from the
  // heaviest parts
  void balance(Rng& rng) {
    for (int sweep = 0; sweep < 8; ++sweep) {
      bool off = false;
      for (int32_t p = 0; p < k; ++p) off = off || pw[p] > maxpw || pw[p] < minpw;
      if (!off) return;
      std::vector<int32_t> order;
      random_order(g.n, rng, order);
      for (int32_t v : order) {
        const int32_t from = part[v];
        int32_t best = -1;
        gather(v);
        if (pw[from] > maxpw) {
          for (int32_t p : seen_parts)
            if (p != from && pw[p] + g.vw[v] <= maxpw && (best < 0 || conn[p] > conn[best])) best = p;
          if (best < 0) {
            const int32_t lightest = (int32_t)(std::min_element(pw.begin(), pw.end()) - pw.begin());
            if (lightest != from && pw[lightest] + g.vw[v] <= maxpw) best = lightest;
          }
        } else if (pw[from] - g.vw[v] >= minpw) {
          for (int32_t p : seen_parts)
            if (p != from && pw[p] < minpw && (best < 0 || conn[p] > conn[best])) best = p;
        }
        clear();
        if (best >= 0) {
          pw[from] -= g.vw[v];
          pw[best] += g.vw[v];
          part[v] = best;
        }
      }
    }
    for (int32_t p = 0; p < k; ++p) {
      if (pw[p] >= minpw) continue;
      for (int32_t v = 0; v < g.n && pw[p] < minpw; ++v) {
        const int32_t from = part[v];
        if (from == p || pw[from] - g.vw[v] < minpw || pw[from] <= pw[p] + g.vw[v]) continue;
        if (pw[from] * (int64_t)k < (int64_t)std::accumulate(pw.begin(), pw.end(), (int64_t)0)) continue;  // below average
        pw[from] -= g.vw[v];
        pw[p] += g.vw[v];
        part[v] = p;
      }
    }
  }

  void refine(int passes, Rng& rng) {
    std::vector<uint8_t> active(g.n, 1), next_active(g.n, 0);
    std::vector<int32_t> order;
    random_order(g.n, rng, order);
    for (int pass = 0; pass < passes; ++pass) {
      int64_t moved = 0;
      for (int32_t v : order) {
        if (!active[v]) continue;
        active[v] = 0;
        const int32_t from = part[v];
        gather(v);
        if (seen_parts.size() > 1 || (seen_parts.size() == 1 && seen_parts[0] != from)) {
          const int32_t internal = conn[from];
          int32_t best = -1;
          for (int32_t p : seen_parts) {
            if (p == from || pw[p] + g.vw[v] > maxpw) continue;
            if (best < 0 || conn[p] > conn[best] || (conn[p] == conn[best] && pw[p] < pw[best])) best = p;
          }
          if (best >= 0 && pw[from] - g.vw[v] >= minpw) {
            const int32_t gain = conn[best] - internal;
            if (gain > 0 || (gain == 0 && pw[best] + g.vw[v] < pw[from])) {
              pw[from] -= g.vw[v];
              pw[best] += g.vw[v];
              part[v] = best;
              ++moved;
              for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e) next_active[g.adj[e]] = 1;
            }
          }
        }
        clear();
      }
      if (moved == 0) break;
      active.swap(next_active);
      std::fill(next_active.begin(), next_active.end(), 0);
    }
  }
};

int64_t weighted_cut(const WGraph& g, const std::vector<int32_t>& part) {
  int64_t cut = 0;
  for (int32_t v = 0; v < g.n; ++v)
    for (int64_t e = g.xadj[v]; e < g.xadj[v + 1]; ++e)
      if (part[g.adj[e]] != part[v]) cut += g.adjw[e];
  return cut / 2;
}

constexpr int kInitialTrials = 8;
constexpr double kCoarseSlack = 1.3;

// a few grown partitions of the coarsest graph, each refined there with the coarse bounds; the one with the
// smallest cut goes on (the host partitioner below and the device partitioner's host step, csrc/kway.cu)
void initial_parts(const WGraph& cg, int32_t k, int64_t maxpw_coarse, int64_t minpw_coarse, int32_t refine_passes,
                   Rng& rng, std::vector<int32_t>& part) {
  int64_t best_cut = -1;
  for (int trial = 0; trial < kInitialTrials; ++trial) {
    std::vector<int32_t> cand;
    initial_partition(cg, k, rng, cand);
    Refiner r(cg, k, maxpw_coarse, minpw_coarse, cand);
    r.balance(rng);
    r.refine(refine_passes, rng);
    r.balance(rng);
    const int64_t cut = weighted_cut(cg, cand);
    if (best_cut < 0 || cut < best_cut) {
      best_cut = cut;
      part.swap(cand);
    }
  }
}

}  // namespace

void kway_bounds(int64_t num_nodes, int32_t k, float ubfactor, KwayBounds* b) {
  const int64_t ideal = (num_nodes + k - 1) / k;
  b->maxpw = std::max<int64_t>(ideal, (int64_t)((double)ubfactor * (double)ideal));
  b->minpw = (int64_t)((double)(num_nodes / k) / (double)ubfactor);   // METIS keeps parts above 1/ufactor too
  // On every level but the finest the parts may be kCoarseSlack times heavier / lighter than the bound: with the
  // strict bound a community that the grown parts split in halves stays split (each half is balanced against the
  // other, the part it should join is full); with slack the halves flow together and the parts that lose them
  // take their own strays back, so the bound is met again by the time the finest level enforces it.
  b->maxpw_coarse = (int64_t)(b->maxpw * kCoarseSlack);
  b->minpw_coarse = (int64_t)(b->minpw / kCoarseSlack);
}

}  // namespace ttg

extern "C" int ttg_partition_kway(int64_t num_nodes, const int64_t* indptr, const int32_t* indices,
                                  int32_t k, float ubfactor, uint64_t seed, int32_t refine_passes,
                                  int32_t* part_out, int64_t* edge_cut_out) {
  using namespace ttg;
  TTG_CHECK_ARG(num_nodes >= 0 && num_nodes < (int64_t)INT32_MAX, "partition_kway: %lld nodes out of range",
                (long long)num_nodes);
  TTG_CHECK_ARG(num_nodes == 0 || (indptr != nullptr && part_out != nullptr), "partition_kway: null pointer");
  TTG_CHECK_ARG(k >= 1 && (num_nodes == 0 || k <= num_nodes), "partition_kway: k=%d for %lld nodes", k,
                (long long)num_nodes);
  TTG_CHECK_ARG(ubfactor >= 1.0f, "partition_kway: ubfactor %g below 1", (double)ubfactor);
  if (edge_cut_out) *edge_cut_out = 0;
  if (num_nodes == 0) return TTG_OK;
  TTG_CHECK_ARG(indptr[0] == 0, "partition_kway: indptr[0] = %lld", (long long)indptr[0]);
  for (int64_t v = 0; v < num_nodes; ++v)
    TTG_CHECK_ARG(indptr[v + 1] >= indptr[v], "partition_kway: indptr decreases at node %lld", (long long)v);
  const int64_t num_edges = indptr[num_nodes];
  TTG_CHECK_ARG(num_edges == 0 || indices != nullptr, "partition_kway: null indices");
  for (int64_t e = 0; e < num_edges; ++e)
    TTG_CHECK_ARG(indices[e] >= 0 && indices[e] < num_nodes, "partition_kway: neighbour id %d out of range",
                  indices[e]);
  if (k == 1) {
    std::memset(part_out, 0, sizeof(int32_t) * (size_t)num_nodes);
    return TTG_OK;
  }
  if (refine_passes <= 0) refine_passes = 10;
  try {
  Rng rng(seed);
  std::vector<WGraph> levels(1);
  PhaseClock clk;
  symmetrise(num_nodes, indptr, indices, levels[0]);
  clk.lap("symmetrise", levels[0].n, (long long)levels[0].adj.size());
  std::vector<std::vector<int32_t>> cmaps;
  const int32_t coarsen_to = std::max<int64_t>(30ll * k, 256);
  while (levels.back().n > coarsen_to && levels.size() < 48) {
    const WGraph& g = levels.back();
    // a coarse vertex stays below 1.5 x the average weight it would have at the target size
    const int32_t maxvw = (int32_t)std::max<int64_t>(1, 3 * num_nodes / (2 * (int64_t)coarsen_to));
    std::vector<int32_t> cmap;
    const int32_t cn = match_and_map(g, rng, maxvw, cmap);
    clk.lap("match", g.n, (long long)g.adj.size());
    if (cn > g.n - g.n / 20) break;   // the matching stalls (< 5 % fewer vertices)
    WGraph c;
    contract(g, cmap, cn, c);
    clk.lap("contract", c.n, (long long)c.adj.size());
    cmaps.push_back(std::move(cmap));
    levels.push_back(std::move(c));
  }
  KwayBounds b;
  kway_bounds(num_nodes, k, ubfactor, &b);
  const int64_t maxpw = b.maxpw, minpw = b.minpw, maxpw_coarse = b.maxpw_coarse, minpw_coarse = b.minpw_coarse;
  std::vector<int32_t> part;
  initial_parts(levels.back(), k, maxpw_coarse, minpw_coarse, refine_passes, rng, part);
  for (size_t lv = levels.size(); lv-- > 0;) {
    Refiner r(levels[lv], k, lv > 0 ? maxpw_coarse : maxpw, lv > 0 ? minpw_coarse : minpw, part);
    r.balance(rng);
    r.refine(refine_passes, rng);
    r.balance(rng);
    clk.lap("refine", levels[lv].n, (long long)levels[lv].adj.size());
    if (lv > 0) {   // project onto the next finer graph
      const std::vector<int32_t>& cmap = cmaps[lv - 1];
      std::vector<int32_t> fine(levels[lv - 1].n);
      for (int32_t v = 0; v < levels[lv - 1].n; ++v) fine[v] = part[cmap[v]];
      part.swap(fine);
      levels[lv] = WGraph();   // free the coarse level
    }
  }
  std::memcpy(part_out, part.data(), sizeof(int32_t) * (size_t)num_nodes);
  if (edge_cut_out) {
    int64_t cut = 0;
    for (int64_t v = 0; v < num_nodes; ++v)
      for (int64_t e = indptr[v]; e < indptr[v + 1]; ++e) cut += part[indices[e]] != part[v];
    *edge_cut_out = cut;
  }
  } catch (const std::exception& ex) {   // host memory (the graph is held about three times) or a worker thread
    set_error("partition_kway: %s", ex.what());
    return TTG_ENOMEM;
  }
  return TTG_OK;
}

extern "C" int ttg_partition_kway_initial(int64_t num_nodes, const int64_t* xadj, const int32_t* adj,
                                          const int32_t* adjw, const int32_t* vw, int64_t total_nodes, int32_t k,
                                          float ubfactor, uint64_t seed, int32_t refine_passes, int32_t* part_out) {
  using namespace ttg;
  TTG_CHECK_ARG(num_nodes > 0 && num_nodes <= total_nodes && total_nodes < (int64_t)INT32_MAX,
                "partition_kway_initial: %lld of %lld nodes out of range", (long long)num_nodes,
                (long long)total_nodes);
  TTG_CHECK_ARG(xadj != nullptr && vw != nullptr && part_out != nullptr, "partition_kway_initial: null pointer");
  TTG_CHECK_ARG(k >= 1 && k <= total_nodes, "partition_kway_initial: k=%d for %lld nodes", k, (long long)total_nodes);
  TTG_CHECK_ARG(ubfactor >= 1.0f, "partition_kway_initial: ubfactor %g below 1", (double)ubfactor);
  TTG_CHECK_ARG(xadj[0] == 0, "partition_kway_initial: xadj[0] = %lld", (long long)xadj[0]);
  for (int64_t v = 0; v < num_nodes; ++v)
    TTG_CHECK_ARG(xadj[v + 1] >= xadj[v] && vw[v] >= 1, "partition_kway_initial: bad row or weight at vertex %lld",
                  (long long)v);
  const int64_t m = xadj[num_nodes];
  TTG_CHECK_ARG(m == 0 || (adj != nullptr && adjw != nullptr), "partition_kway_initial: null adjacency");
  for (int64_t e = 0; e < m; ++e)
    TTG_CHECK_ARG(adj[e] >= 0 && adj[e] < num_nodes && adjw[e] >= 1,
                  "partition_kway_initial: neighbour id %d out of range", adj[e]);
  if (refine_passes <= 0) refine_passes = 10;
  try {
    WGraph g;
    g.n = (int32_t)num_nodes;
    g.xadj.assign(xadj, xadj + num_nodes + 1);
    g.adj.assign(adj, adj + m);
    g.adjw.assign(adjw, adjw + m);
    g.vw.assign(vw, vw + num_nodes);
    KwayBounds b;
    kway_bounds(total_nodes, k, ubfactor, &b);
    Rng rng(seed);
    std::vector<int32_t> part;
    initial_parts(g, k, b.maxpw_coarse, b.minpw_coarse, refine_passes, rng, part);
    std::memcpy(part_out, part.data(), sizeof(int32_t) * (size_t)num_nodes);
  } catch (const std::exception& ex) {
    set_error("partition_kway_initial: %s", ex.what());
    return TTG_ENOMEM;
  }
  return TTG_OK;
}
