// Host-side index builder: produces the reference's hnsw_slim `.graph` file for a corpus.
//
// Not on the GPU hot path — it exists so that benchmarks and deployments can create the
// engine's input without the reference binary: (1) a multi-threaded HNSW construction
// (Malkov & Yashunin, the algorithm the reference inherits from hnswlib: hnsw.h:1248-1376
// addPoint, :326-479 searchBaseLayer, :481-523 getNeighborsByHeuristic2, :525-660
// mutuallyConnectNewElement), then (2) HNSW-Slim's pruning into the CHAL layout
// (slim.h:867-1108 convertFromHNSW) and (3) the file format of saveIndex (slim.h:717-751).
// Written from the algorithm descriptions; the output is loadable by the reference's own
// HierarchicalNSWSlim::loadIndex (tests/test_host.py::test_builder_writes_the_reference_format checks that with oracle/_ref).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <queue>
#include <thread>
#include <vector>

#include "hs_internal.h"

namespace hs {
namespace {

using Pair = std::pair<float, uint32_t>;

__attribute__((target_clones("avx512f", "avx2", "default")))
float l2sqr(const float *a, const float *b, size_t dim) {
  float acc[16] = {0};
  size_t i = 0;
  for (; i + 16 <= dim; i += 16)
    for (int j = 0; j < 16; ++j) {
      const float d = a[i + j] - b[i + j];
      acc[j] += d * d;
    }
  float s = 0;
  for (int j = 0; j < 16; ++j) s += acc[j];
  for (; i < dim; ++i) {
    const float d = a[i] - b[i];
    s += d * d;
  }
  return s;
}

__attribute__((target_clones("avx512f", "avx2", "default")))
float ipdist(const float *a, const float *b, size_t dim) {
  float acc[16] = {0};
  size_t i = 0;
  for (; i + 16 <= dim; i += 16)
    for (int j = 0; j < 16; ++j) acc[j] += a[i + j] * b[i + j];
  float s = 0;
  for (int j = 0; j < 16; ++j) s += acc[j];
  for (; i < dim; ++i) s += a[i] * b[i];
  return 1.0f - s;
}

struct SpinLock {
  std::atomic_flag f = ATOMIC_FLAG_INIT;
  void lock() {
    while (f.test_and_set(std::memory_order_acquire)) {
    }
  }
  void unlock() { f.clear(std::memory_order_release); }
};

// splitmix64: per-node reproducible randomness (levels do not depend on thread timing)
inline uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

struct Hnsw {
  const float *data;
  size_t n, dim;
  int metric;
  size_t M, maxM, maxM0, efc;
  std::vector<int8_t> level;
  std::vector<uint32_t> links0;            // n * maxM0
  std::vector<uint16_t> cnt0;              // n
  std::vector<std::vector<uint32_t>> up;   // node -> level * (maxM + 1): [count, ids...]
  std::unique_ptr<SpinLock[]> locks;
  std::mutex global;
  std::atomic<int> maxlevel{-1};
  std::atomic<uint32_t> enter{kInvalid};

  float dist(const float *a, const float *b) const { return metric == HS_METRIC_IP ? ipdist(a, b, dim) : l2sqr(a, b, dim); }
  const float *vec(uint32_t i) const { return data + (size_t)i * dim; }

  uint32_t *list(uint32_t node, int lvl, uint32_t **cnt16or32, bool *is0) {
    (void)cnt16or32;
    (void)is0;
    return lvl == 0 ? &links0[(size_t)node * maxM0] : &up[node][(size_t)(lvl - 1) * (maxM + 1) + 1];
  }
  uint32_t count(uint32_t node, int lvl) const {
    return lvl == 0 ? cnt0[node] : up[node][(size_t)(lvl - 1) * (maxM + 1)];
  }
  void set_count(uint32_t node, int lvl, uint32_t c) {
    if (lvl == 0) cnt0[node] = (uint16_t)c; else up[node][(size_t)(lvl - 1) * (maxM + 1)] = c;
  }
  const uint32_t *clist(uint32_t node, int lvl) const {
    return lvl == 0 ? &links0[(size_t)node * maxM0] : &up[node][(size_t)(lvl - 1) * (maxM + 1) + 1];
  }
};

struct Visited {
  std::vector<uint16_t> tag;
  uint16_t cur = 0;
  explicit Visited(size_t n) : tag(n, 0) {}
  void next() {
    if (++cur == 0) {
      std::fill(tag.begin(), tag.end(), 0);
      cur = 1;
    }
  }
};

// ef-bounded best-first search on one layer; returns candidates sorted ascending by distance.
void search_layer(Hnsw &h, const float *q, uint32_t ep, float ep_dist, int lvl, size_t ef, Visited &vis,
                  std::vector<Pair> &out) {
  vis.next();
  std::priority_queue<Pair> top;                                        // farthest on top
  std::priority_queue<Pair, std::vector<Pair>, std::greater<Pair>> cand;  // closest on top
  top.emplace(ep_dist, ep);
  cand.emplace(ep_dist, ep);
  vis.tag[ep] = vis.cur;
  float bound = ep_dist;
  std::vector<uint32_t> nb;
  while (!cand.empty()) {
    const Pair c = cand.top();
    if (c.first > bound && top.size() >= ef) break;
    cand.pop();
    {
      SpinLock &l = h.locks[c.second];
      l.lock();
      const uint32_t cnt = h.count(c.second, lvl);
      const uint32_t *ids = h.clist(c.second, lvl);
      nb.assign(ids, ids + cnt);
      l.unlock();
    }
    for (uint32_t id : nb) {
      if (vis.tag[id] == vis.cur) continue;
      vis.tag[id] = vis.cur;
      const float d = h.dist(q, h.vec(id));
      if (top.size() < ef || d < bound) {
        cand.emplace(d, id);
        top.emplace(d, id);
        if (top.size() > ef) top.pop();
        bound = top.top().first;
      }
    }
  }
  out.resize(top.size());
  for (size_t i = top.size(); i-- > 0;) {
    out[i] = top.top();
    top.pop();
  }
}

// relative-neighbourhood heuristic: scan closest first, keep a candidate only if it is not
// closer to an already kept one than to the base point (hnsw.h:481-523, slim.h:837-865)
void select_heuristic(const Hnsw &h, const std::vector<Pair> &sorted, size_t M, std::vector<uint32_t> &kept) {
  kept.clear();
  for (const Pair &c : sorted) {
    if (kept.size() >= M) break;
    bool good = true;
    for (uint32_t k : kept)
      if (h.dist(h.vec(k), h.vec(c.second)) < c.first) {
        good = false;
        break;
      }
    if (good) kept.push_back(c.second);
  }
}

uint32_t connect(Hnsw &h, uint32_t c, std::vector<Pair> &cands, int lvl) {
  const size_t Mmax = lvl == 0 ? h.maxM0 : h.maxM;
  std::vector<uint32_t> sel;
  if (cands.size() < h.M) {          // hnsw.h:486-488: fewer than M candidates are all kept
    for (const Pair &p : cands) sel.push_back(p.second);
  } else {
    select_heuristic(h, cands, h.M, sel);
  }
  {
    SpinLock &l = h.locks[c];
    l.lock();
    uint32_t *mine = h.list(c, lvl, nullptr, nullptr);
    for (size_t i = 0; i < sel.size(); ++i) mine[i] = sel[i];
    h.set_count(c, lvl, (uint32_t)sel.size());
    l.unlock();
  }
  std::vector<Pair> tmp;
  std::vector<uint32_t> kept;
  for (uint32_t s : sel) {
    SpinLock &l = h.locks[s];
    l.lock();
    const uint32_t cnt = h.count(s, lvl);
    uint32_t *ids = h.list(s, lvl, nullptr, nullptr);
    bool present = false;
    for (uint32_t i = 0; i < cnt; ++i) present |= ids[i] == c;
    if (!present) {
      if (cnt < Mmax) {
        ids[cnt] = c;
        h.set_count(s, lvl, cnt + 1);
      } else {
        tmp.clear();
        tmp.emplace_back(h.dist(h.vec(s), h.vec(c)), c);
        for (uint32_t i = 0; i < cnt; ++i) tmp.emplace_back(h.dist(h.vec(s), h.vec(ids[i])), ids[i]);
        std::sort(tmp.begin(), tmp.end());
        select_heuristic(h, tmp, Mmax, kept);
        for (size_t i = 0; i < kept.size(); ++i) ids[i] = kept[i];
        h.set_count(s, lvl, (uint32_t)kept.size());
      }
    }
    l.unlock();
  }
  return cands.empty() ? c : cands.front().second;
}

void insert(Hnsw &h, uint32_t c, Visited &vis, std::vector<Pair> &cands) {
  const int lc = h.level[c];
  std::unique_lock<std::mutex> g(h.global);
  const int maxl = h.maxlevel.load();
  if (lc <= maxl) g.unlock();
  uint32_t cur = h.enter.load();
  if (cur == kInvalid) {             // first element
    h.enter = c;
    h.maxlevel = lc;
    return;
  }
  const float *q = h.vec(c);
  float curd = h.dist(q, h.vec(cur));
  std::vector<uint32_t> nb;
  for (int lvl = maxl; lvl > lc; --lvl) {      // greedy descent
    bool changed = true;
    while (changed) {
      changed = false;
      {
        SpinLock &l = h.locks[cur];
        l.lock();
        const uint32_t cnt = h.count(cur, lvl);
        const uint32_t *ids = h.clist(cur, lvl);
        nb.assign(ids, ids + cnt);
        l.unlock();
      }
      for (uint32_t id : nb) {
        const float d = h.dist(q, h.vec(id));
        if (d < curd) {
          curd = d;
          cur = id;
          changed = true;
        }
      }
    }
  }
  for (int lvl = std::min(lc, maxl); lvl >= 0; --lvl) {
    search_layer(h, q, cur, curd, lvl, h.efc, vis, cands);
    // the new point itself is not in the graph yet, so it cannot be among the candidates
    cur = connect(h, c, cands, lvl);
    curd = h.dist(q, h.vec(cur));
  }
  if (lc > maxl) {
    h.enter = c;
    h.maxlevel = lc;
  }
}

template <typename F>
void parallel_for(size_t begin, size_t end, int threads, F &&fn) {
  std::atomic<size_t> next{begin};
  auto worker = [&](int tid) {
    for (;;) {
      const size_t i0 = next.fetch_add(64);
      if (i0 >= end) break;
      const size_t i1 = std::min(end, i0 + 64);
      for (size_t i = i0; i < i1; ++i) fn(i, tid);
    }
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < threads; ++t) pool.emplace_back(worker, t);
  worker(0);
  for (auto &t : pool) t.join();
}

}  // namespace

namespace {

// HNSW construction + HNSW-Slim pruning: the pruned per-level out-lists of every node.
struct Pruned {
  Hnsw h;
  std::vector<std::vector<std::vector<uint32_t>>> nbr;
  int maxlevel = 0;
};

int build_pruned(const float *base, size_t n, size_t dim, int metric, size_t M, size_t ef_construction,
                 double branching, int threshold_level, float top_pct0, float top_pct, size_t top_M0,
                 size_t low_m0, size_t top_M, size_t low_m, int threads, uint64_t seed, Pruned *out,
                 bool prune = true) {
  if (!base || n == 0 || dim == 0 || M < 2 || M > 512 || branching <= 1.0 || n >= (1ull << 31)) {
    set_error("build_slim_graph: bad argument");
    return HS_ERR_ARG;
  }
  Hnsw &h = out->h;
  h.data = base;
  h.n = n;
  h.dim = dim;
  h.metric = metric;
  h.M = M;
  h.maxM = M;
  h.maxM0 = 2 * M;                                 // hnsw.h:108-109
  h.efc = std::max(ef_construction, M);            // hnsw.h:110
  const double mult = 1.0 / std::log(branching);   // hnsw.h:143-158
  h.level.resize(n);
  h.links0.assign(n * h.maxM0, 0);
  h.cnt0.assign(n, 0);
  h.up.resize(n);
  h.locks.reset(new SpinLock[n]);
  int top_level = 0;
  for (size_t i = 0; i < n; ++i) {
    const double u = ((mix64(seed * 0x9E3779B9ull + i) >> 11) + 1) * (1.0 / 9007199254740993.0);   // (0,1)
    int l = (int)(-std::log(u) * mult);                                                     // hnsw.h:203-207
    l = std::min(l, kMaxLevels - 2);
    h.level[i] = (int8_t)l;
    top_level = std::max(top_level, l);
    if (l > 0) h.up[i].assign((size_t)l * (h.maxM + 1), 0);
  }

  // ---- 1. HNSW construction ----
  // The first few thousand points go in one at a time: points inserted concurrently into a
  // near-empty graph see almost no candidates, end up with one or two links and can become
  // unreachable once their few neighbours turn into hubs and prune them (measured: 0.8 % of the
  // first 5000 nodes of a 50k graph with 8 threads, none with this serial prefix).
  const size_t serial_prefix = std::min<size_t>(n, 4096);
  {
    Visited v0(n);
    std::vector<Pair> c0;
    for (size_t i = 0; i < serial_prefix; ++i) insert(h, (uint32_t)i, v0, c0);
  }
  {
    std::vector<std::unique_ptr<Visited>> vis(threads);
    std::vector<std::vector<Pair>> cands(threads);
    parallel_for(serial_prefix, n, threads, [&](size_t i, int tid) {
      if (!vis[tid]) vis[tid].reset(new Visited(n));
      insert(h, (uint32_t)i, *vis[tid], cands[tid]);
    });
  }
  const int maxlevel = h.maxlevel.load();
  out->maxlevel = maxlevel;
  if (!prune) return HS_OK;          // hs_build_hnsw_graph: the un-pruned index is the product

  // ---- 2. HNSW-Slim pruning (slim.h:867-1108) ----
  // degree thresholds: a level's top `pct` nodes by out-degree keep top_M* neighbours, the rest
  // low_m*.  As in the reference, the level-0 population count is never accumulated
  // (slim.h:906-921 counts levels >= 1 only), so on level 0 topN = 0, the threshold lands on
  // maxM0 + 1 and EVERY node is pruned to low_m0 before reverse edges are added.
  std::vector<std::vector<size_t>> hist(maxlevel + 1, std::vector<size_t>(h.maxM0 + 2, 0));
  std::vector<size_t> level_cnt(maxlevel + 1, 0);
  for (size_t i = 0; i < n; ++i) {
    for (int l = 1; l <= h.level[i]; ++l) {
      level_cnt[l]++;
      hist[l][h.count((uint32_t)i, l)]++;
    }
    hist[0][h.count((uint32_t)i, 0)]++;
  }
  std::vector<size_t> deg_thr(maxlevel + 1, 0);
  for (int l = 0; l <= maxlevel; ++l) {
    const size_t topN = (size_t)(level_cnt[l] * (l == 0 ? top_pct0 : top_pct) + 0.5);
    size_t acc = 0;
    for (size_t d = hist[l].size() - 1; d > 0; --d) {
      acc += hist[l][d];
      if (acc >= topN) {
        deg_thr[l] = d;
        break;
      }
    }
  }
  // out-lists after the first prune, then with reverse edges merged in
  std::vector<std::vector<std::vector<uint32_t>>> &nbr = out->nbr;
  std::vector<std::vector<std::vector<uint32_t>>> rev(n);
  nbr.assign(n, {});
  parallel_for(0, n, threads, [&](size_t v, int) {
    const int lv = h.level[v];
    nbr[v].resize(lv + 1);
    rev[v].resize(lv + 1);
    std::vector<Pair> tmp;
    for (int l = 0; l <= lv; ++l) {
      const uint32_t cnt = h.count((uint32_t)v, l);
      const uint32_t *ids = h.clist((uint32_t)v, l);
      const size_t keep = l == 0 ? (cnt > deg_thr[l] ? top_M0 : low_m0) : (cnt > deg_thr[l] ? top_M : low_m);
      tmp.clear();
      for (uint32_t j = 0; j < cnt; ++j) tmp.emplace_back(h.dist(h.vec((uint32_t)v), h.vec(ids[j])), ids[j]);
      std::sort(tmp.begin(), tmp.end());
      select_heuristic(h, tmp, keep, nbr[v][l]);
    }
  });
  parallel_for(0, n, threads, [&](size_t v, int) {
    for (int l = 0; l <= h.level[v]; ++l)
      for (uint32_t u : nbr[v][l]) {
        h.locks[u].lock();
        rev[u][l].push_back((uint32_t)v);
        h.locks[u].unlock();
      }
  });
  parallel_for(0, n, threads, [&](size_t v, int) {
    std::vector<Pair> tmp;
    for (int l = 0; l <= h.level[v]; ++l) {
      auto &lst = nbr[v][l];
      lst.insert(lst.end(), rev[v][l].begin(), rev[v][l].end());
      std::sort(lst.begin(), lst.end());
      lst.erase(std::unique(lst.begin(), lst.end()), lst.end());
      const size_t limit = l == 0 ? h.maxM0 : h.maxM;
      if (lst.size() > limit) {                     // slim.h:1036-1058
        tmp.clear();
        for (uint32_t u : lst) tmp.emplace_back(h.dist(h.vec((uint32_t)v), h.vec(u)), u);
        std::sort(tmp.begin(), tmp.end());
        select_heuristic(h, tmp, limit, lst);
      }
      // hierarchical pruning (slim.h:1063-1084): away from the threshold level a neighbour
      // is kept only where that level is its own top level
      if (l != threshold_level) {
        size_t w = 0;
        for (uint32_t u : lst)
          if (h.level[u] == l) lst[w++] = u;
        lst.resize(w);
      }
    }
    rev[v].clear();
    rev[v].shrink_to_fit();
  });
  out->maxlevel = maxlevel;
  return HS_OK;
}

// per-node neighbour blobs, shared by both file formats (slim.h:741-748, slimq.h:1205-1214)
bool write_blobs(FILE *f, const Pruned &P) {
  const size_t n = P.h.n;
  auto put = [&](const void *p, size_t sz) { return std::fwrite(p, 1, sz, f) == sz; };
  bool ok = true;
  std::vector<uint8_t> blob;
  for (size_t i = 0; i < n && ok; ++i) {
    const int lv = P.h.level[i];
    uint32_t total = 0;
    for (auto &l : P.nbr[i]) total += (uint32_t)l.size();
    const uint32_t bsz = (uint32_t)(2 * lv + 4 * total);
    ok &= put(&bsz, 4);
    if (bsz == 0 || total == 0) continue;
    blob.resize(bsz);
    uint32_t run = 0;
    for (int l = 0; l < lv; ++l) {
      run += (uint32_t)P.nbr[i][l].size();
      const uint16_t o = (uint16_t)run;
      std::memcpy(&blob[2 * l], &o, 2);
    }
    size_t w = 2 * (size_t)lv;
    for (int l = 0; l <= lv; ++l)
      for (uint32_t u : P.nbr[i][l]) {
        std::memcpy(&blob[w], &u, 4);
        w += 4;
      }
    ok &= put(blob.data(), bsz);
  }
  return ok;
}

}  // namespace

int build_slim_graph(const float *base, size_t n, size_t dim, int metric, size_t M, size_t ef_construction,
                     double branching, int threshold_level, float top_pct0, float top_pct, size_t top_M0,
                     size_t low_m0, size_t top_M, size_t low_m, int threads, uint64_t seed,
                     const uint64_t *labels, const char *out_path) {
  if (!out_path) {
    set_error("build_slim_graph: bad argument");
    return HS_ERR_ARG;
  }
  if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
  Pruned P;
  int rc = build_pruned(base, n, dim, metric, M, ef_construction, branching, threshold_level, top_pct0, top_pct,
                        top_M0, low_m0, top_M, low_m, threads, seed, &P);
  if (rc != HS_OK) return rc;
  Hnsw &h = P.h;
  auto &nbr = P.nbr;
  const int maxlevel = P.maxlevel;

  // ---- 3. saveIndex format (slim.h:717-751) ----
  FILE *f = std::fopen(out_path, "wb");
  if (!f) {
    set_error(std::string("cannot open ") + out_path + " for writing");
    return HS_ERR_IO;
  }
  auto put = [&](const void *p, size_t sz) { return std::fwrite(p, 1, sz, f) == sz; };
  bool ok = true;
  const uint64_t rec = 24 + 4 * dim;
  const uint64_t hdr[6] = {n, rec, 8, 4, 24, 16};
  ok &= put(hdr, sizeof hdr);
  const int32_t ml = maxlevel, thr = threshold_level;
  const uint32_t ep = h.enter.load();
  ok &= put(&ml, 4) && put(&thr, 4) && put(&ep, 4);
  const uint64_t ms[4] = {h.maxM, h.maxM0, h.M, h.efc};
  ok &= put(ms, sizeof ms);
  const uint8_t has_deleted = 0;
  ok &= put(&has_deleted, 1);
  std::vector<uint8_t> record(rec);
  for (size_t i = 0; i < n && ok; ++i) {
    uint32_t total = 0;
    for (auto &l : nbr[i]) total += (uint32_t)l.size();
    const int32_t lv = h.level[i];
    const uint64_t label = labels ? labels[i] : (uint64_t)i;
    const uint64_t stale_ptr = 0;
    std::memcpy(&record[0], &lv, 4);
    std::memcpy(&record[4], &total, 4);
    std::memcpy(&record[8], &label, 8);
    std::memcpy(&record[16], &stale_ptr, 8);
    std::memcpy(&record[24], h.vec((uint32_t)i), 4 * dim);
    ok &= put(record.data(), rec);
  }
  ok = ok && write_blobs(f, P);
  ok &= std::fclose(f) == 0;
  if (!ok) {
    set_error(std::string("write error on ") + out_path);
    return HS_ERR_IO;
  }
  return HS_OK;
}

// The un-pruned index of the `hnsw` strategy (hnsw_strategy.h:24-45): the same construction, saved
// in HierarchicalNSW::saveIndex's format (hnsw.h:748-779) — level-0 records
// [uint32 count][uint32 ids[maxM0]][float vec[dim]][uint64 label], then per node
// uint32 linkListSize + level lists of [uint32 count][uint32 ids[maxM]].
int build_hnsw_graph(const float *base, size_t n, size_t dim, int metric, size_t M, size_t ef_construction,
                     double branching, int threads, uint64_t seed, const uint64_t *labels, const char *out_path) {
  if (!out_path) {
    set_error("build_hnsw_graph: bad argument");
    return HS_ERR_ARG;
  }
  if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
  Pruned P;
  int rc = build_pruned(base, n, dim, metric, M, ef_construction, branching, 0, 0.f, 0.f, 0, 0, 0, 0, threads, seed,
                        &P, false);
  if (rc != HS_OK) return rc;
  Hnsw &h = P.h;
  FILE *f = std::fopen(out_path, "wb");
  if (!f) {
    set_error(std::string("cannot open ") + out_path + " for writing");
    return HS_ERR_IO;
  }
  auto put = [&](const void *p, size_t sz) { return std::fwrite(p, 1, sz, f) == sz; };
  bool ok = true;
  const uint64_t links0 = 4 + 4 * h.maxM0, links = 4 + 4 * h.maxM, rec = links0 + 4 * dim + 8;
  const uint64_t hdr[6] = {0 /*offsetLevel0*/, n /*max_elements*/, n, rec, links0 + 4 * dim /*label_offset*/,
                           links0 /*offsetData*/};
  ok &= put(hdr, sizeof hdr);
  const int32_t ml = P.maxlevel;
  const uint32_t ep = h.enter.load();
  ok &= put(&ml, 4) && put(&ep, 4);
  const uint64_t ms[3] = {h.maxM, h.maxM0, h.M};
  ok &= put(ms, sizeof ms);
  const double mult = 1.0 / std::log(branching);
  const uint64_t efc = h.efc;
  ok &= put(&mult, 8) && put(&efc, 8);
  std::vector<uint8_t> record(rec);
  for (size_t i = 0; i < n && ok; ++i) {
    std::fill(record.begin(), record.end(), 0);
    const uint32_t c = h.count((uint32_t)i, 0);
    std::memcpy(&record[0], &c, 4);
    std::memcpy(&record[4], h.clist((uint32_t)i, 0), 4 * (size_t)c);
    std::memcpy(&record[links0], h.vec((uint32_t)i), 4 * dim);
    const uint64_t label = labels ? labels[i] : (uint64_t)i;
    std::memcpy(&record[links0 + 4 * dim], &label, 8);
    ok &= put(record.data(), rec);
  }
  std::vector<uint8_t> lists;
  for (size_t i = 0; i < n && ok; ++i) {
    const int lvl = h.level[i];
    const uint32_t lsz = (uint32_t)(lvl * links);
    ok &= put(&lsz, 4);
    if (!lsz) continue;
    lists.assign(lsz, 0);
    for (int l = 1; l <= lvl; ++l) {
      const uint32_t c = h.count((uint32_t)i, l);
      std::memcpy(&lists[(size_t)(l - 1) * links], &c, 4);
      std::memcpy(&lists[(size_t)(l - 1) * links + 4], h.clist((uint32_t)i, l), 4 * (size_t)c);
    }
    ok &= put(lists.data(), lsz);
  }
  ok &= std::fclose(f) == 0;
  if (!ok) {
    set_error(std::string("write error on ") + out_path);
    return HS_ERR_IO;
  }
  return HS_OK;
}

// ------------------------------------------------------------------------------------------
// hnsw_slimq builder: the same HNSW + HNSW-Slim pruning over the raw floats, node payload =
// 1-bit RaBitQ codes + factors, written in HierarchicalNSWSlimQ::saveIndex's format
// (slimq.h:1161-1216) so both hs_load and the reference's loadIndex read it.
namespace {
void host_fwht(float *buf, size_t len) {          // natural order, butterfly distance 1, 2, 4, ...
  for (size_t h = 1; h < len; h *= 2)
    for (size_t j = 0; j < len; j += 2 * h)
      for (size_t k = 0; k < h; ++k) {
        const float u = buf[j + k], v = buf[j + k + h];
        buf[j + k] = u + v;
        buf[j + k + h] = u - v;
      }
}

}  // namespace

// FhtKacRotator::rotate (rabitqlib/utils/rotator.hpp:370-423)
void host_rotate(const float *x, size_t dim, size_t pd, size_t td, const uint8_t *flip, float *out) {
  const float fac = 1.0f / std::sqrt((float)td);
  std::memcpy(out, x, 4 * dim);
  std::fill(out + dim, out + pd, 0.f);
  const bool pow2 = td == pd;
  const size_t start = pd - td;
  for (int r = 0; r < 4; ++r) {
    const uint8_t *fl = flip + (size_t)r * pd / 8;
    for (size_t i = 0; i < pd; ++i)
      if ((fl[i >> 3] >> (i & 7)) & 1u) out[i] = -out[i];
    float *seg = (!pow2 && (r & 1)) ? out + start : out;
    host_fwht(seg, td);
    for (size_t i = 0; i < td; ++i) seg[i] *= fac;
    if (!pow2)
      for (size_t i = 0; i < pd / 2; ++i) {
        const float a = out[i], b = out[i + pd / 2];
        out[i] = a + b;
        out[i + pd / 2] = a - b;
      }
  }
  if (!pow2)
    for (size_t i = 0; i < pd; ++i) out[i] *= 0.25f;
}

// Lloyd k-means over the raw rows (the reference reads *_centroids_16.fvecs and
// *_clusterids_16.ivecs that no code in it produces, hnsw_slimq_strategy.h:42-45)
void host_kmeans(const float *base, size_t n, size_t dim, size_t k, int iters, uint64_t seed, int threads,
                 std::vector<float> &cent, std::vector<uint32_t> &ids) {
  if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
  cent.assign(k * dim, 0.f);
  ids.assign(n, 0);
  for (size_t c = 0; c < k; ++c) {
    const size_t pick = (size_t)(mix64(seed * 7919 + c) % n);
    std::memcpy(&cent[c * dim], base + pick * dim, 4 * dim);
  }
  const size_t sample = std::min<size_t>(n, 200000), stride = std::max<size_t>(1, n / sample);
  auto assign = [&](size_t i) {
    float best = std::numeric_limits<float>::max();
    uint32_t arg = 0;
    for (size_t c = 0; c < k; ++c) {
      const float d = l2sqr(base + i * dim, &cent[c * dim], dim);
      if (d < best) {
        best = d;
        arg = (uint32_t)c;
      }
    }
    return arg;
  };
  for (int it = 0; it < iters; ++it) {
    std::vector<std::vector<double>> sum(threads, std::vector<double>(k * dim, 0.0));
    std::vector<std::vector<size_t>> cnt(threads, std::vector<size_t>(k, 0));
    parallel_for(0, (n + stride - 1) / stride, threads, [&](size_t s, int tid) {
      const size_t i = s * stride;
      const uint32_t a = assign(i);
      cnt[tid][a]++;
      for (size_t d = 0; d < dim; ++d) sum[tid][a * dim + d] += base[i * dim + d];
    });
    for (size_t c = 0; c < k; ++c) {
      size_t tot = 0;
      for (int t = 0; t < threads; ++t) tot += cnt[t][c];
      if (!tot) continue;
      for (size_t d = 0; d < dim; ++d) {
        double v = 0;
        for (int t = 0; t < threads; ++t) v += sum[t][c * dim + d];
        cent[c * dim + d] = (float)(v / (double)tot);
      }
    }
  }
  parallel_for(0, n, threads, [&](size_t i, int) { ids[i] = assign(i); });
}

int build_slimq_graph(const float *base, size_t n, size_t dim, size_t M, size_t ef_construction, double branching,
                      int threshold_level, float top_pct0, float top_pct, size_t top_M0, size_t low_m0,
                      size_t top_M, size_t low_m, int threads, uint64_t seed, const float *centroids,
                      size_t num_cluster, const uint32_t *cluster_ids, const uint64_t *labels,
                      const char *out_path) {
  if (!out_path || num_cluster == 0 || num_cluster > 4096 || (centroids && !cluster_ids)) {
    set_error("build_slimq_graph: bad argument");
    return HS_ERR_ARG;
  }
  if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
  Pruned P;
  int rc = build_pruned(base, n, dim, HS_METRIC_L2, M, ef_construction, branching, threshold_level, top_pct0,
                        top_pct, top_M0, low_m0, top_M, low_m, threads, seed, &P);
  if (rc != HS_OK) return rc;
  const Hnsw &h = P.h;

  std::vector<float> cent_own;
  std::vector<uint32_t> cid_own;
  if (!centroids) {
    host_kmeans(base, n, dim, num_cluster, 8, seed, threads, cent_own, cid_own);
    centroids = cent_own.data();
    cluster_ids = cid_own.data();
  }
  // rotator: 4 x padded_dim random sign bits (rotator.hpp:217-229 draws them from random_device)
  const size_t pd = (dim + 63) / 64 * 64, words = pd / 64;     // rabitqlib/index/hnsw/hnsw.hpp:424-427
  size_t td = 1;
  while (td * 2 <= dim) td *= 2;                                // rotator.hpp:233-235
  if (td < 64 || td > 2048) {
    set_error("build_slimq_graph: dim must be in [64, 4095] (FhtKacRotator, rotator.hpp:237-258)");
    return HS_ERR_UNSUPPORTED;
  }
  std::vector<uint8_t> flip(4 * pd / 8);
  for (size_t i = 0; i < flip.size(); ++i) flip[i] = (uint8_t)(mix64(seed * 0xD1B54A32D192ED03ull + i) >> 56);
  std::vector<float> rcent(num_cluster * pd);
  for (size_t c = 0; c < num_cluster; ++c) host_rotate(centroids + c * dim, dim, pd, td, flip.data(), &rcent[c * pd]);

  // one_bit_code_with_factor (rabitq_impl.hpp:76-135, L2 metric) per node, in double
  std::vector<uint64_t> codes(n * words, 0);
  std::vector<float> fac(3 * n);                                // f_add, f_rescale, f_error
  parallel_for(0, n, threads, [&](size_t i, int) {
    std::vector<float> rot(pd);
    host_rotate(base + i * dim, dim, pd, td, flip.data(), rot.data());
    const float *cen = &rcent[(size_t)cluster_ids[i] * pd];
    double l2 = 0, ip_resi = 0, ip_cent = 0;
    uint64_t *code = &codes[i * words];
    for (size_t d = 0; d < pd; ++d) {
      const float r = rot[d] - cen[d];
      const int bit = r > 0.f ? 1 : 0;
      const double xu = bit - 0.5;
      l2 += (double)r * r;
      ip_resi += (double)r * xu;
      ip_cent += (double)cen[d] * xu;
      if (bit) code[d / 64] |= 1ull << (63 - (d % 64));      // pack_binary, space.hpp:272-286
    }
    if (ip_resi == 0) ip_resi = std::numeric_limits<double>::infinity();
    const double l2n = std::sqrt(l2);
    const double tmp_err =
        l2n * 1.9 * std::sqrt(std::max(0.0, (l2 * ((double)pd * 0.25) / (ip_resi * ip_resi) - 1.0) / (double)(pd - 1)));
    fac[3 * i] = (float)(l2 + 2 * l2 * ip_cent / ip_resi);
    fac[3 * i + 1] = (float)(-2 * l2 / ip_resi);
    fac[3 * i + 2] = (float)(2 * tmp_err);
  });

  SlimqHead head;
  head.n = n;
  head.maxlevel = P.maxlevel;
  head.threshold_level = threshold_level;
  head.enterpoint = h.enter.load();
  head.maxM = h.maxM;
  head.maxM0 = h.maxM0;
  head.M = h.M;
  head.ef_construction = h.efc;
  head.num_cluster = num_cluster;
  head.dim = dim;
  head.padded_dim = pd;
  head.ex_bits = 3;
  head.size_ex = pd * 3 / 8 + 8;                                // data_layout.hpp
  head.centroids = rcent.data();
  head.flip = flip.data();
  return write_slimq_file(
      out_path, head,
      [&](size_t i0, size_t cnt, SlimqNode *out) -> int {
        for (size_t j = 0; j < cnt; ++j) {
          const size_t i = i0 + j;
          SlimqNode &nd = out[j];
          nd.level = h.level[i];
          nd.total = 0;
          for (auto &l : P.nbr[i]) nd.total += (uint32_t)l.size();
          nd.label = labels ? labels[i] : (uint64_t)i;
          nd.cluster = cluster_ids[i];
          nd.code = &codes[i * words];
          nd.f_add = fac[3 * i];
          nd.f_rescale = fac[3 * i + 1];
          nd.f_error = fac[3 * i + 2];
        }
        return HS_OK;
      },
      [&](FILE *f) { return write_blobs(f, P); });
}

int write_slimq_file(const char *path, const SlimqHead &h,
                     const std::function<int(size_t i0, size_t cnt, SlimqNode *out)> &nodes,
                     const std::function<bool(FILE *f)> &blobs) {
  // record layout (slimq.h:1498-1505): [level][total][label][ptr][cluster @24][bin @28][ex]
  const size_t words = h.padded_dim / 64;
  const uint64_t size_bin = h.padded_dim / 8 + 12;             // data_layout.hpp
  const uint64_t off_bin = 28, off_ex = off_bin + size_bin, rec = off_ex + h.size_ex;
  FILE *f = std::fopen(path, "wb");
  if (!f) {
    set_error(std::string("cannot open ") + path + " for writing");
    return HS_ERR_IO;
  }
  auto put = [&](const void *p, size_t sz) { return std::fwrite(p, 1, sz, f) == sz; };
  bool ok = true;
  const uint64_t hdr[6] = {h.n, rec, 8, 4, off_bin /* offsetData_ = offset_bin_data_, slimq.h:1503 */, 16};
  ok &= put(hdr, sizeof hdr);
  ok &= put(&h.maxlevel, 4) && put(&h.threshold_level, 4) && put(&h.enterpoint, 4);
  const uint64_t ms[4] = {h.maxM, h.maxM0, h.M, h.ef_construction};
  ok &= put(ms, sizeof ms);
  const uint8_t has_deleted = 0;
  ok &= put(&has_deleted, 1);
  const uint64_t meta[9] = {h.num_cluster, h.dim, h.padded_dim, 24, off_bin, off_ex, size_bin, h.size_ex, h.ex_bits};
  ok &= put(meta, sizeof meta);
  const uint8_t metric_type = 0;   // rabitqlib::METRIC_L2
  ok &= put(&metric_type, 1);
  ok &= put(h.centroids, h.num_cluster * h.padded_dim * 4);
  ok &= put(h.flip, 4 * h.padded_dim / 8);
  const size_t slab = std::max<size_t>(1, (64u << 20) / rec);
  std::vector<SlimqNode> nd(std::min<size_t>(slab, h.n));
  std::vector<uint8_t> buf(nd.size() * rec);
  for (size_t i0 = 0; i0 < h.n && ok; i0 += slab) {
    const size_t cnt = std::min<size_t>(slab, h.n - i0);
    const int rc = nodes(i0, cnt, nd.data());
    if (rc != HS_OK) {
      std::fclose(f);
      return rc;
    }
    std::fill(buf.begin(), buf.end(), 0);
    for (size_t j = 0; j < cnt; ++j) {
      uint8_t *e = &buf[j * rec];
      std::memcpy(e, &nd[j].level, 4);
      std::memcpy(e + 4, &nd[j].total, 4);
      std::memcpy(e + 8, &nd[j].label, 8);
      std::memcpy(e + 24, &nd[j].cluster, 4);
      std::memcpy(e + off_bin, nd[j].code, 8 * words);
      std::memcpy(e + off_bin + 8 * words, &nd[j].f_add, 4);
      std::memcpy(e + off_bin + 8 * words + 4, &nd[j].f_rescale, 4);
      std::memcpy(e + off_bin + 8 * words + 8, &nd[j].f_error, 4);
    }
    ok &= put(buf.data(), cnt * rec);
  }
  ok = ok && blobs(f);
  ok &= std::fclose(f) == 0;
  if (!ok) {
    set_error(std::string("write error on ") + path);
    return HS_ERR_IO;
  }
  return HS_OK;
}

}  // namespace hs
