// GPU-side index construction: HNSW build + HNSW-Slim conversion, resident in HBM from the first
// row to the finished index (SURVEY.md §8(f) rank 3; the host-side counterpart is graph_build.cpp).
//
//  Phase 1 — HNSW construction.  The algorithm is hnswlib's (addPoint hnsw.h:1248-1376,
//  searchBaseLayer :326-479, getNeighborsByHeuristic2 :481-523, mutuallyConnectNewElement :525-660),
//  arranged for a GPU: levels are drawn up front (hnsw.h:203-207), the layers are built one after
//  the other from the top (a layer's graph only needs the layers above it for entry points), and a
//  layer grows by BATCHES of points: one warp per new point runs the ef_construction beam search
//  over the graph built so far (the traversal kernel's pool, visited hash and row scorer) and picks
//  its M neighbours with the relative-neighbourhood heuristic; the reverse edges of the whole batch
//  are then sorted by target (cub radix sort) and one warp per target appends them or — when its
//  list overflows — re-selects maxM of {old list + newcomers} with the same heuristic.  Batches are
//  at most 1/16 of the layer built so far, so a point misses few of its true neighbours by sharing
//  a batch with them (the reference's OpenMP build has the same blindness between its threads).
//
//  Phase 2 — HNSW-Slim conversion = convertFromHNSW (slim.h:867-1108): per node and level,
//  distance-sort the list and prune it with PruneByHeuristic (:836-865) to low_m / top_M (degree
//  histogram thresholds, :905-947); merge the reverse edges of the pruned lists in (:985-1011);
//  re-prune lists longer than maxM0 / maxM (:1036-1058); away from threshold_level keep only
//  neighbours whose own top level is this level (:1063-1084).  One warp per (node, level) for each
//  step, reverse edges through one radix sort per level.
//
// The result is an hs_index like the one hs_load makes; hs_save_index writes it in the reference's
// saveIndex format (slim.h:717-751) so that the reference — and the CPU baseline — load it.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cub/cub.cuh>
#include <memory>
#include <string>
#include <vector>

#include "hs_index.h"
#include "traverse_common.cuh"

namespace hs {
namespace {

#define GB_CUDA(call)                                                                 \
  do {                                                                                \
    cudaError_t e__ = (call);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      set_error(std::string(#call) + ": " + cudaGetErrorString(e__));                 \
      return HS_ERR_CUDA;                                                             \
    }                                                                                 \
  } while (0)

constexpr int kHashBits = 12;                  // visited table of the construction search (per warp)
constexpr uint32_t kMergeCap = 2048;           // candidates one node can carry into the re-prune

// ---- the point a warp measures distances FROM: registers (8-lane teams, CPL float4 per lane)
//      or shared memory (large dims), exactly the two forms of the traversal kernel ----
template <int CPL, int METRIC>
struct Probe {
  float4 q[CPL > 0 ? CPL : 1];
  float4 *qs;
  const float4 *vec;
  uint32_t row_chunks;
  int lane;
  __device__ __forceinline__ void init(const float4 *vec_, uint32_t rc, float4 *qs_, int lane_) {
    vec = vec_;
    row_chunks = rc;
    qs = qs_;
    lane = lane_;
  }
  __device__ __forceinline__ void load(uint32_t node) {
    const float4 *row = vec + (size_t)node * row_chunks;
    if constexpr (CPL > 0) {
      float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);     // row_chunks = 8 * CPL <= 32
      if ((uint32_t)lane < row_chunks) mine = __ldg(row + lane);
      const int t8 = lane & 7;
#pragma unroll
      for (int j = 0; j < CPL; ++j) {
        q[j].x = __shfl_sync(FULL, mine.x, t8 + 8 * j);
        q[j].y = __shfl_sync(FULL, mine.y, t8 + 8 * j);
        q[j].z = __shfl_sync(FULL, mine.z, t8 + 8 * j);
        q[j].w = __shfl_sync(FULL, mine.w, t8 + 8 * j);
      }
    } else {
      __syncwarp();
      for (uint32_t ch = lane; ch < row_chunks; ch += 32) qs[ch] = __ldg(row + ch);
      __syncwarp();
    }
  }
  // distances to `count` (<= 32) rows: lane j passes id j and receives d_j
  __device__ __forceinline__ float eval(uint32_t my_id, int count) const {
    if constexpr (CPL > 0) {
      return eval_rows_reg<CPL, METRIC, 1>(vec, row_chunks, q, my_id, count, lane);
    } else {
      return eval_rows_smem<METRIC>(vec, row_chunks, qs, my_id, count, lane);
    }
  }
};

// Relative-neighbourhood selection over candidates handed out in ascending (distance, id) order by
// next() (NONE when exhausted): keep a candidate unless an already kept one is strictly closer to it
// than the base point is (hnsw.h:481-523, slim.h:836-865).  Kept ids end in lane registers: lane j
// holds kept[j] in sel0 (j < 32) / kept[32 + j] in sel1.  The probe is overwritten.
template <int CPL, int METRIC, typename Next>
__device__ __forceinline__ uint32_t select_rng(Probe<CPL, METRIC> &pr, Next &&next, uint32_t want, bool take_all,
                                               uint32_t &sel0, uint32_t &sel1, float &seld0, float &seld1) {
  const int lane = pr.lane;
  uint32_t nsel = 0;
  sel0 = sel1 = kInvalid;
  seld0 = seld1 = 0.f;
  while (nsel < want) {
    const uint64_t key = next();
    if (key == NONE) break;
    const uint32_t c = (uint32_t)key;
    const float dc = ord2f((uint32_t)(key >> 32));
    bool good = true;
    if (nsel > 0 && !take_all) {
      pr.load(c);
      const float d0 = pr.eval(sel0 == kInvalid ? 0u : sel0, (int)min(nsel, 32u));
      bool closer = (uint32_t)lane < min(nsel, 32u) && d0 < dc;
      if (nsel > 32) {
        const float d1 = pr.eval(sel1 == kInvalid ? 0u : sel1, (int)(nsel - 32));
        closer |= (uint32_t)lane < nsel - 32 && d1 < dc;
      }
      good = !__any_sync(FULL, closer);
    }
    if (good) {
      if (nsel < 32) {
        if ((uint32_t)lane == nsel) {
          sel0 = c;
          seld0 = dc;
        }
      } else if ((uint32_t)lane == nsel - 32) {
        sel1 = c;
        seld1 = dc;
      }
      ++nsel;
    }
  }
  return nsel;
}

// bitonic sort of n2 (power of two) 64-bit keys in shared memory by one warp
__device__ __forceinline__ void warp_bitonic(uint64_t *a, uint32_t n2, int lane) {
  for (uint32_t k = 2; k <= n2; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      __syncwarp();
      for (uint32_t i = lane; i < n2; i += 32) {
        const uint32_t x = i ^ j;
        if (x > i) {
          const uint64_t u = a[i], v = a[x];
          const bool up = (i & k) == 0;
          if ((u > v) == up) {
            a[i] = v;
            a[x] = u;
          }
        }
      }
    }
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// Phase 1 kernels
// ---------------------------------------------------------------------------------------------
struct InsertParams {
  const float4 *vec;
  uint32_t row_chunks, n;
  uint32_t *adj;                                // rows of the layer under construction, kInvalid-padded
  uint32_t stride;
  const int32_t *slot;                          // node -> row on layers >= 1 (-1: level-0-only node)
  int layer, maxlevel;
  const uint32_t *upper_adj[kMaxLevels];        // complete layers above `layer`, stride ustride
  uint32_t ustride;
  uint32_t ep;                                  // the node with the highest level: first in every layer
  const uint32_t *order;                        // insertion order of this layer: position -> node
  uint32_t frontier, batch;                     // this launch inserts positions [frontier, frontier + batch)
  uint32_t M, efc;
  uint32_t *req_target, *req_src;               // batch x M reverse-edge requests (kInvalid = none)
  float *req_dist;
};

template <int CPL, int METRIC>
__global__ void __launch_bounds__(32) insert_kernel(const __grid_constant__ InsertParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint32_t *hash = reinterpret_cast<uint32_t *>(smem);
  uint32_t *stage_ids = hash + (1u << kHashBits);
  float4 *qs = reinterpret_cast<float4 *>(stage_ids + 32);
  const int lane = threadIdx.x;
  const uint32_t w = blockIdx.x;
  const uint32_t node = p.order[p.frontier + w];
  constexpr uint32_t hbits = kHashBits, hsize = 1u << kHashBits, hmask = hsize - 1, hlimit = hsize - hsize / 4;

  Probe<CPL, METRIC> pr;
  pr.init(p.vec, p.row_chunks, qs, lane);
  pr.load(node);
  hash_clear(hash, hsize, lane);
  __syncwarp();

  // greedy descent through the complete layers above (hnsw.h:1276-1303), restricted to nodes that are
  // already part of the layer under construction: on every layer those are the slots below `frontier`
  // (a layer is filled in slot order = level descending, and nodes found above have slots)
  uint32_t cur = p.ep;
  float curdist = __shfl_sync(FULL, pr.eval(cur, 1), 0);
  for (int level = p.maxlevel; level > p.layer; --level) {
    const uint32_t *ladj = p.upper_adj[level];
    bool changed = true;
    while (changed) {
      changed = false;
      const uint32_t *row = ladj + (size_t)__ldg(p.slot + cur) * p.ustride;
      for (uint32_t seg = 0; seg < p.ustride; seg += 32) {
        uint32_t id = (seg + lane < p.ustride) ? __ldg(row + seg + lane) : kInvalid;
        if (__ballot_sync(FULL, id != kInvalid) == 0) break;
        if (id != kInvalid && (uint32_t)__ldg(p.slot + id) >= p.frontier) id = kInvalid;
        const unsigned vm = __ballot_sync(FULL, id != kInvalid);
        if (vm == 0) continue;
        const int count = __popc(vm);
        if (id != kInvalid) stage_ids[__popc(vm & ((1u << lane) - 1))] = id;
        __syncwarp();
        const uint32_t cid = lane < count ? stage_ids[lane] : 0u;
        __syncwarp();
        const float d = pr.eval(cid, count);
        uint64_t key = lane < count ? (((uint64_t)f2ord(d) << 32) | (uint32_t)lane) : ~0ull;
        key = warp_min_u64(key);
        const float best = ord2f((uint32_t)(key >> 32));
        const uint32_t best_id = __shfl_sync(FULL, cid, (int)(key & 31));
        if (best < curdist) {
          curdist = best;
          cur = best_id;
          changed = true;
        }
      }
    }
  }

  // ef_construction beam search on the layer under construction (hnsw.h:326-479)
  RegPool32<8> pool;
  pool.init(nullptr, p.efc, lane);
  pool.seed(make_key(curdist, cur));
  uint32_t hcount = 1;
  if (lane == 0) visited_test_and_set(hash, hbits, hmask, cur);
  __syncwarp();
  for (;;) {
    const uint32_t x = pool.pop_closest_unexpanded();
    if (x == kInvalid) break;
    const uint32_t xrow = p.layer == 0 ? x : (uint32_t)__ldg(p.slot + x);
    const uint32_t *row = p.adj + (size_t)xrow * p.stride;
    if (hcount + p.stride > hlimit) {
      __syncwarp();
      hash_clear(hash, hsize, lane);
      __syncwarp();
      pool.for_each_id([&](uint32_t pid) { visited_test_and_set(hash, hbits, hmask, pid); });
      hcount = pool.size;
      __syncwarp();
    }
    for (uint32_t seg = 0; seg < p.stride; seg += 32) {
      // rows change between batches only, but stay away from the read-only path: another launch wrote them
      const uint32_t id = *reinterpret_cast<const volatile uint32_t *>(row + seg + lane);
      const unsigned vm = __ballot_sync(FULL, id != kInvalid);
      if (vm == 0) break;
      bool fresh = false;
      if (id != kInvalid) fresh = !visited_test_and_set(hash, hbits, hmask, id);
      if (fresh) {
        const char *r = reinterpret_cast<const char *>(p.vec + (size_t)id * p.row_chunks);
        for (uint32_t off = 0; off < p.row_chunks * 16u; off += 128) prefetch_l2(r + off);
      }
      const unsigned fm = __ballot_sync(FULL, fresh);
      const int count = __popc(fm);
      if (count == 0) continue;
      hcount += (uint32_t)count;
      if (fresh) stage_ids[__popc(fm & ((1u << lane) - 1))] = id;
      __syncwarp();
      const uint32_t cid = lane < count ? stage_ids[lane] : 0u;
      __syncwarp();
      const float d = pr.eval(cid, count);
      pool.admit(lane < count, make_key(d, cid));
    }
  }

  // neighbour selection (hnsw.h:481-523): fewer than M candidates are all kept (:486-488)
  uint64_t last = 0;
  auto next = [&]() -> uint64_t {
    if (last == NONE) return NONE;
    const uint64_t mine = pool.col_next_above(last);
    const int o = warp_argmin_key(mine);
    last = o >= 0 ? __shfl_sync(FULL, mine, o) : NONE;
    return last;
  };
  uint32_t sel0, sel1;
  float seld0, seld1;
  const uint32_t nsel = select_rng(pr, next, p.M, pool.size < p.M, sel0, sel1, seld0, seld1);

  const uint32_t myrow = p.layer == 0 ? node : (uint32_t)__ldg(p.slot + node);
  uint32_t *out = p.adj + (size_t)myrow * p.stride;
  for (uint32_t seg = 0; seg < p.stride; seg += 32) {
    uint32_t v = kInvalid;
    if (seg == 0 && (uint32_t)lane < nsel) v = sel0;
    if (seg == 32 && (uint32_t)lane + 32 < nsel) v = sel1;
    out[seg + lane] = v;
  }
  for (uint32_t j = lane; j < p.M; j += 32) {
    const bool have = j < nsel;
    const size_t at = (size_t)w * p.M + j;
    p.req_target[at] = have ? (j < 32 ? sel0 : sel1) : kInvalid;
    p.req_src[at] = node;
    p.req_dist[at] = have ? (j < 32 ? seld0 : seld1) : 0.f;
  }
}

struct BacklinkParams {
  const float4 *vec;
  uint32_t row_chunks;
  uint32_t *adj;
  uint32_t stride;
  const int32_t *slot;
  int layer;
  uint32_t Mmax;
  const uint32_t *keys;        // request targets, sorted ascending (kInvalid last)
  const uint32_t *vals;        // request index of every sorted position
  const uint32_t *req_src;
  const float *req_dist;
  uint32_t nreq;
};

// One warp per sorted request; the warp at the head of a target's run does the whole run
// (mutuallyConnectNewElement, hnsw.h:566-647, for all newcomers of the batch at once).
template <int CPL, int METRIC>
__global__ void __launch_bounds__(128) backlink_kernel(const __grid_constant__ BacklinkParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float4 *qs = reinterpret_cast<float4 *>(smem) + (size_t)wid * p.row_chunks;
  const uint32_t i = blockIdx.x * (blockDim.x >> 5) + wid;
  if (i >= p.nreq) return;
  const uint32_t t = p.keys[i];
  if (t == kInvalid || (i > 0 && p.keys[i - 1] == t)) return;
  // newcomers of this target: at most 64 (a longer run keeps its first 64 in batch order)
  uint32_t s0 = kInvalid, s1 = kInvalid;
  float sd0 = 0.f, sd1 = 0.f;
  const bool in0 = i + lane < p.nreq && p.keys[i + lane] == t;
  const bool in1 = i + 32 + lane < p.nreq && p.keys[i + 32 + lane] == t;
  if (in0) {
    const uint32_t r = p.vals[i + lane];
    s0 = p.req_src[r];
    sd0 = p.req_dist[r];
  }
  if (in1) {
    const uint32_t r = p.vals[i + 32 + lane];
    s1 = p.req_src[r];
    sd1 = p.req_dist[r];
  }
  const unsigned m0 = __ballot_sync(FULL, in0), m1 = m0 == FULL ? __ballot_sync(FULL, in1) : 0u;
  if (m0 != FULL) s1 = kInvalid;
  const uint32_t r_new = (uint32_t)__popc(m0) + (uint32_t)__popc(m1);     // runs are contiguous: masks are prefixes

  const uint32_t trow = p.layer == 0 ? t : (uint32_t)__ldg(p.slot + t);
  uint32_t *row = p.adj + (size_t)trow * p.stride;
  uint32_t e0 = row[lane], e1 = p.stride > 32 ? row[32 + lane] : kInvalid;
  const uint32_t c0 = (uint32_t)__popc(__ballot_sync(FULL, e0 != kInvalid));
  const uint32_t c1 = (uint32_t)__popc(__ballot_sync(FULL, e1 != kInvalid));
  const uint32_t cnt = c0 + c1;
  if (cnt + r_new <= p.Mmax) {                  // room for everyone: append (hnsw.h:583-587)
    // lane j holds newcomer j in s0 and newcomer 32 + j in s1
    for (uint32_t j = lane; j < r_new; j += 32) row[cnt + j] = j < 32 ? s0 : s1;
    return;
  }
  // overflow: maxM of {old list + newcomers}, closest first, relative-neighbourhood rule (hnsw.h:588-640)
  Probe<CPL, METRIC> pr;
  pr.init(p.vec, p.row_chunks, qs, lane);
  pr.load(t);
  uint64_t k[4] = {NONE, NONE, NONE, NONE};
  {
    const float d0 = pr.eval(e0 == kInvalid ? 0u : e0, (int)c0);
    if ((uint32_t)lane < c0) k[0] = make_key(d0, e0);
    if (c1) {
      const float d1 = pr.eval(e1 == kInvalid ? 0u : e1, (int)c1);
      if ((uint32_t)lane < c1) k[1] = make_key(d1, e1);
    }
    if (s0 != kInvalid) k[2] = make_key(sd0, s0);
    if (s1 != kInvalid) k[3] = make_key(sd1, s1);
  }
  uint64_t last = 0;
  auto next = [&]() -> uint64_t {
    if (last == NONE) return NONE;
    uint64_t m = NONE;
#pragma unroll
    for (int j = 0; j < 4; ++j) m = (k[j] > last && k[j] < m) ? k[j] : m;
    const int o = warp_argmin_key(m);
    last = o >= 0 ? __shfl_sync(FULL, m, o) : NONE;
    return last;
  };
  uint32_t sel0, sel1;
  float seld0, seld1;
  const uint32_t nsel = select_rng(pr, next, p.Mmax, false, sel0, sel1, seld0, seld1);
  row[lane] = (uint32_t)lane < nsel ? sel0 : kInvalid;
  if (p.stride > 32) row[32 + lane] = (uint32_t)lane + 32 < nsel ? sel1 : kInvalid;
}

// ---------------------------------------------------------------------------------------------
// Phase 2 kernels (convertFromHNSW, slim.h:867-1108)
// ---------------------------------------------------------------------------------------------
struct PruneParams {
  const float4 *vec;
  uint32_t row_chunks;
  const uint32_t *adj;          // HNSW lists of this level
  uint32_t stride, rows;
  const uint32_t *node_of_row;  // nullptr on level 0 (row == node)
  uint32_t keep_low, keep_top, deg_threshold;   // slim.h:971-976
  uint32_t *nbr1;               // rows x nstride: the pruned lists
  uint32_t nstride;
  uint32_t *req_target, *req_src;   // rows x keep_cap reverse-edge requests
  uint32_t keep_cap;
};

template <int CPL, int METRIC>
__global__ void __launch_bounds__(128) prune_kernel(const __grid_constant__ PruneParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float4 *qs = reinterpret_cast<float4 *>(smem) + (size_t)wid * p.row_chunks;
  const uint32_t r = blockIdx.x * (blockDim.x >> 5) + wid;
  if (r >= p.rows) return;
  const uint32_t node = p.node_of_row ? p.node_of_row[r] : r;
  const uint32_t *row = p.adj + (size_t)r * p.stride;
  const uint32_t e0 = row[lane], e1 = p.stride > 32 ? row[32 + lane] : kInvalid;
  const uint32_t c0 = (uint32_t)__popc(__ballot_sync(FULL, e0 != kInvalid));
  const uint32_t c1 = (uint32_t)__popc(__ballot_sync(FULL, e1 != kInvalid));
  const uint32_t cnt = c0 + c1;
  const uint32_t keep = cnt > p.deg_threshold ? p.keep_top : p.keep_low;
  Probe<CPL, METRIC> pr;
  pr.init(p.vec, p.row_chunks, qs, lane);
  uint32_t nsel = 0, sel0 = kInvalid, sel1 = kInvalid;
  float seld0, seld1;
  if (cnt) {
    pr.load(node);
    uint64_t k[2] = {NONE, NONE};
    const float d0 = pr.eval(e0 == kInvalid ? 0u : e0, (int)c0);
    if ((uint32_t)lane < c0) k[0] = make_key(d0, e0);
    if (c1) {
      const float d1 = pr.eval(e1 == kInvalid ? 0u : e1, (int)c1);
      if ((uint32_t)lane < c1) k[1] = make_key(d1, e1);
    }
    uint64_t last = 0;
    auto next = [&]() -> uint64_t {
      if (last == NONE) return NONE;
      uint64_t m = NONE;
#pragma unroll
      for (int j = 0; j < 2; ++j) m = (k[j] > last && k[j] < m) ? k[j] : m;
      const int o = warp_argmin_key(m);
      last = o >= 0 ? __shfl_sync(FULL, m, o) : NONE;
      return last;
    };
    nsel = select_rng(pr, next, keep, false, sel0, sel1, seld0, seld1);
  }
  for (uint32_t seg = 0; seg < p.nstride; seg += 32) {
    uint32_t v = kInvalid;
    if (seg == 0 && (uint32_t)lane < nsel) v = sel0;
    if (seg == 32 && (uint32_t)lane + 32 < nsel) v = sel1;
    p.nbr1[(size_t)r * p.nstride + seg + lane] = v;
  }
  for (uint32_t j = lane; j < p.keep_cap; j += 32) {
    const size_t at = (size_t)r * p.keep_cap + j;
    p.req_target[at] = j < nsel ? (j < 32 ? sel0 : sel1) : kInvalid;
    p.req_src[at] = node;
  }
}

// first / one-past-last sorted position of every target (targets without requests keep 0 / 0)
__global__ void segment_bounds_kernel(const uint32_t *__restrict__ keys, uint32_t nreq, uint32_t *seg_begin,
                                      uint32_t *seg_end) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nreq) return;
  const uint32_t t = keys[i];
  if (t == kInvalid) return;
  if (i == 0 || keys[i - 1] != t) seg_begin[t] = i;
  if (i + 1 == nreq || keys[i + 1] != t) seg_end[t] = i + 1;
}

struct MergeParams {
  const float4 *vec;
  uint32_t row_chunks, rows;
  const uint32_t *node_of_row;          // nullptr on level 0
  const uint32_t *nbr1;                 // pruned lists
  uint32_t nstride;
  const uint32_t *seg_begin, *seg_end;  // per NODE: its run in rev_src
  const uint32_t *rev_src;              // request sources in target order (vals-permuted)
  uint32_t limit;                       // maxM0 / maxM (slim.h:1036)
  const int8_t *levels;
  int level, threshold_level;
  uint32_t *out;                        // rows x ostride final lists
  uint32_t ostride;
  unsigned long long *sum_deg;          // [0] total degree [1] overflow count
  uint32_t *max_deg;
};

template <int CPL, int METRIC>
__global__ void __launch_bounds__(32) merge_kernel(const __grid_constant__ MergeParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t *keys = reinterpret_cast<uint64_t *>(smem);                  // kMergeCap
  float4 *qs = reinterpret_cast<float4 *>(keys + kMergeCap);
  const int lane = threadIdx.x;
  const uint32_t r = blockIdx.x;
  const uint32_t node = p.node_of_row ? p.node_of_row[r] : r;
  // union of the pruned list and the reverse edges, sorted by id, duplicates dropped (slim.h:1002-1010)
  const uint32_t b = p.seg_begin[node], e = p.seg_end[node];
  uint32_t nrev = e - b;
  uint32_t m = 0;
  for (uint32_t seg = 0; seg < p.nstride; seg += 32) {
    const uint32_t id = p.nbr1[(size_t)r * p.nstride + seg + lane];
    const unsigned vm = __ballot_sync(FULL, id != kInvalid);
    if (id != kInvalid) keys[m + __popc(vm & ((1u << lane) - 1))] = id;
    m += (uint32_t)__popc(vm);
  }
  if (m + nrev > kMergeCap) {
    if (lane == 0) atomicAdd(p.sum_deg + 1, 1ull);
    nrev = kMergeCap - m;
  }
  for (uint32_t j = lane; j < nrev; j += 32) keys[m + j] = p.rev_src[b + j];
  m += nrev;
  uint32_t n2 = 1;
  while (n2 < m) n2 <<= 1;
  for (uint32_t j = m + lane; j < n2; j += 32) keys[j] = NONE;
  __syncwarp();
  warp_bitonic(keys, n2, lane);
  uint32_t u = 0;                                         // unique count; compaction in place (u <= read position)
  for (uint32_t base = 0; base < m; base += 32) {
    const uint32_t j = base + lane;
    const uint64_t v = j < m ? keys[j] : NONE;
    const bool keepit = j < m && (j == 0 || keys[j - 1] != v);
    __syncwarp();
    const unsigned km = __ballot_sync(FULL, keepit);
    if (keepit) keys[u + __popc(km & ((1u << lane) - 1))] = v;
    u += (uint32_t)__popc(km);
    __syncwarp();
  }
  m = u;

  uint32_t nsel = 0, sel0 = kInvalid, sel1 = kInvalid;
  if (m > p.limit) {                                      // re-prune (slim.h:1036-1058)
    Probe<CPL, METRIC> pr;
    pr.init(p.vec, p.row_chunks, qs, lane);
    pr.load(node);
    for (uint32_t base = 0; base < m; base += 32) {
      const uint32_t j = base + lane;
      const uint32_t id = j < m ? (uint32_t)keys[j] : 0u;
      const float d = pr.eval(id, (int)min(32u, m - base));
      __syncwarp();
      if (j < m) keys[j] = make_key(d, id);
    }
    n2 = 1;
    while (n2 < m) n2 <<= 1;
    for (uint32_t j = m + lane; j < n2; j += 32) keys[j] = NONE;
    __syncwarp();
    warp_bitonic(keys, n2, lane);
    uint32_t pos = 0;
    auto next = [&]() -> uint64_t { return pos < m ? keys[pos++] : NONE; };
    float seld0, seld1;
    nsel = select_rng(pr, next, p.limit, false, sel0, sel1, seld0, seld1);
  } else {
    nsel = m;
    if ((uint32_t)lane < m) sel0 = (uint32_t)keys[lane];
    if ((uint32_t)lane + 32 < m) sel1 = (uint32_t)keys[lane + 32];
  }
  // hierarchical pruning (slim.h:1063-1084)
  bool k0 = (uint32_t)lane < nsel, k1 = (uint32_t)lane + 32 < nsel;
  if (p.level != p.threshold_level) {
    k0 = k0 && p.levels[sel0] == p.level;
    k1 = k1 && p.levels[sel1] == p.level;
  }
  const unsigned b0 = __ballot_sync(FULL, k0), b1 = __ballot_sync(FULL, k1);
  const uint32_t n0 = (uint32_t)__popc(b0), deg = n0 + (uint32_t)__popc(b1);
  uint32_t *out = p.out + (size_t)r * p.ostride;
  for (uint32_t j = lane; j < p.ostride; j += 32) out[j] = kInvalid;
  __syncwarp();
  if (k0) out[__popc(b0 & ((1u << lane) - 1))] = sel0;
  if (k1) out[n0 + __popc(b1 & ((1u << lane) - 1))] = sel1;
  if (lane == 0) {
    atomicAdd(p.sum_deg, (unsigned long long)deg);
    atomicMax(p.max_deg, deg);
  }
}

__global__ void gather_u32_kernel(const uint32_t *__restrict__ src, const uint32_t *__restrict__ idx, uint32_t n,
                                  uint32_t *__restrict__ dst) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}
__global__ void iota_kernel(uint32_t *a, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = i;
}
__global__ void restride_kernel(const uint32_t *__restrict__ src, uint32_t sstride, uint32_t *__restrict__ dst,
                                uint32_t dstride, size_t rows) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * dstride) return;
  const size_t r = i / dstride;
  const uint32_t c = (uint32_t)(i % dstride);
  dst[i] = c < sstride ? src[r * sstride + c] : kInvalid;
}
__global__ void pad_rows_kernel(const float *__restrict__ src, uint32_t dim, float *__restrict__ dst, uint32_t dim_padded,
                                size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * dim_padded) return;
  const size_t r = i / dim_padded;
  const uint32_t c = (uint32_t)(i % dim_padded);
  dst[i] = c < dim ? src[r * dim + c] : 0.f;
}

// ---------------------------------------------------------------------------------------------
// hnsw_slimq payload: cluster assignment, FHT-Kac rotation, 1-bit RaBitQ code + factors per node
// (the host builder's loop, graph_build.cpp build_slimq_graph; one_bit_code_with_factor,
// rabitqlib/quantization/rabitq_impl.hpp:76-135; rotator.hpp:370-423; pack_binary, space.hpp:272-286)
// ---------------------------------------------------------------------------------------------
struct PayloadParams {
  const float *vec;               // n x dim_padded raw rows
  uint32_t n, dim, dim_padded, pd, td, words, num_cluster;
  const float *cent;              // num_cluster x dim   raw centroids (cluster assignment)
  const float *rcent;             // num_cluster x pd    rotated centroids
  const uint8_t *flip;            // 4 * pd / 8
  float fac;                      // 1 / sqrt(td)
  uint2 *qrec;                    // n x (words + 2)
  float *f_error;                 // n (the file's third factor; the search does not read it)
};

__global__ void __launch_bounds__(128) slimq_payload_kernel(const __grid_constant__ PayloadParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float *buf = reinterpret_cast<float *>(smem) + (size_t)wid * p.pd;
  const uint32_t i = blockIdx.x * (blockDim.x >> 5) + wid;
  if (i >= p.n) return;
  const float *row = p.vec + (size_t)i * p.dim_padded;
  for (uint32_t d = lane; d < p.pd; d += 32) buf[d] = d < p.dim ? row[d] : 0.f;
  __syncwarp();
  // nearest raw centroid, first minimum (host_kmeans assign)
  uint32_t cluster = 0;
  {
    float best = 3.402823466e+38f;
    for (uint32_t c0 = 0; c0 < p.num_cluster; c0 += 32) {
      const uint32_t c = c0 + lane;
      float d = 3.402823466e+38f;
      if (c < p.num_cluster) {
        const float *cv = p.cent + (size_t)c * p.dim;
        float acc = 0.f;
        for (uint32_t k = 0; k < p.dim; ++k) {
          const float t = buf[k] - cv[k];
          acc = fmaf(t, t, acc);
        }
        d = acc;
      }
      uint64_t key = ((uint64_t)f2ord(d) << 32) | c;
      key = warp_min_u64(key);
      const float bd = ord2f((uint32_t)(key >> 32));
      if (bd < best) {
        best = bd;
        cluster = (uint32_t)key;
      }
    }
  }
  // FhtKacRotator::rotate, operation for operation as host_rotate (graph_build.cpp)
  const bool pow2 = p.td == p.pd;
  const uint32_t start = p.pd - p.td;
  for (int r = 0; r < 4; ++r) {
    const uint8_t *fl = p.flip + (size_t)r * p.pd / 8;
    for (uint32_t d = lane; d < p.pd; d += 32)
      if ((fl[d >> 3] >> (d & 7)) & 1u) buf[d] = -buf[d];
    __syncwarp();
    float *seg = (!pow2 && (r & 1)) ? buf + start : buf;
    for (uint32_t h = 1; h < p.td; h *= 2) {
      for (uint32_t idx = lane; idx < p.td / 2; idx += 32) {
        const uint32_t j = (idx / h) * 2 * h + (idx % h);
        const float u = seg[j], v = seg[j + h];
        seg[j] = u + v;
        seg[j + h] = u - v;
      }
      __syncwarp();
    }
    for (uint32_t d = lane; d < p.td; d += 32) seg[d] *= p.fac;
    __syncwarp();
    if (!pow2) {
      for (uint32_t d = lane; d < p.pd / 2; d += 32) {
        const float a = buf[d], b = buf[d + p.pd / 2];
        buf[d] = a + b;
        buf[d + p.pd / 2] = a - b;
      }
      __syncwarp();
    }
  }
  if (!pow2) {
    for (uint32_t d = lane; d < p.pd; d += 32) buf[d] *= 0.25f;
    __syncwarp();
  }
  // residual against the rotated centroid: sign bits + the three sums of one_bit_code_with_factor, in double
  const float *cen = p.rcent + (size_t)cluster * p.pd;
  uint2 *rec = p.qrec + (size_t)i * (p.words + 2);
  double l2 = 0, ip_resi = 0, ip_cent = 0;
  for (uint32_t w = 0; w < p.words; ++w) {
    uint32_t half[2];
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const uint32_t d = 64 * w + 32 * hh + lane;
      const float rr = buf[d] - cen[d];
      const bool bit = rr > 0.f;
      const double xu = bit ? 0.5 : -0.5;
      l2 += (double)rr * rr;
      ip_resi += (double)rr * xu;
      ip_cent += (double)cen[d] * xu;
      half[hh] = __brev(__ballot_sync(FULL, bit));      // dimension 64w + j  <->  bit 63 - j (MSB first)
    }
    if (lane == 0) rec[w] = make_uint2(half[1], half[0]);   // (low 32 bits, high 32 bits) of the code word
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    l2 += __shfl_xor_sync(FULL, l2, off);
    ip_resi += __shfl_xor_sync(FULL, ip_resi, off);
    ip_cent += __shfl_xor_sync(FULL, ip_cent, off);
  }
  if (lane == 0) {
    if (ip_resi == 0) ip_resi = __longlong_as_double(0x7ff0000000000000ll);
    const float f_add = (float)(l2 + 2 * l2 * ip_cent / ip_resi);
    const float f_rescale = (float)(-2 * l2 / ip_resi);
    const double tmp_err =
        sqrt(l2) * 1.9 * sqrt(fmax(0.0, (l2 * ((double)p.pd * 0.25) / (ip_resi * ip_resi) - 1.0) / (double)(p.pd - 1)));
    rec[p.words] = make_uint2(__float_as_uint(f_add), __float_as_uint(f_rescale));
    rec[p.words + 1] = make_uint2(cluster, 0u);
    p.f_error[i] = (float)(2 * tmp_err);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct DevBuf {                       // frees on scope exit unless released
  void *p = nullptr;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  template <typename T>
  T *as() const { return static_cast<T *>(p); }
  int alloc(size_t bytes) {
    if (p) cudaFree(p);
    p = nullptr;
    if (bytes == 0) bytes = 4;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();
      set_error("cudaMalloc(" + std::to_string(bytes) + "): " + cudaGetErrorString(e));
      return e == cudaErrorMemoryAllocation ? HS_ERR_NOMEM : HS_ERR_CUDA;
    }
    return HS_OK;
  }
  void *release() {
    void *q = p;
    p = nullptr;
    return q;
  }
};

inline uint64_t mix64(uint64_t x) {            // the host builder's per-node level stream (graph_build.cpp)
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

inline uint32_t round_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

template <typename F>
int dispatch_cm(uint32_t row_chunks, int metric, F &&f) {
  const uint32_t cpl = row_chunks / kTeam;
  const int c = (cpl == 3 || cpl == 4) ? (int)cpl : 0;
#define GB_CASE(C, M) \
  if (c == C && metric == M) return f(std::integral_constant<int, C>{}, std::integral_constant<int, M>{});
  GB_CASE(0, HS_METRIC_L2) GB_CASE(3, HS_METRIC_L2) GB_CASE(4, HS_METRIC_L2)
  GB_CASE(0, HS_METRIC_IP) GB_CASE(3, HS_METRIC_IP) GB_CASE(4, HS_METRIC_IP)
#undef GB_CASE
  set_error("graph_gpu: unknown metric");
  return HS_ERR_ARG;
}

// radix sort of (target, request index) pairs; returns sorted keys / vals in out buffers
struct Sorter {
  DevBuf temp, keys_out, vals_out, iota;
  size_t temp_bytes = 0, cap = 0;
  int prepare(size_t max_items, cudaStream_t st) {
    cap = max_items;
    int rc;
    if ((rc = keys_out.alloc(max_items * 4)) != HS_OK || (rc = vals_out.alloc(max_items * 4)) != HS_OK ||
        (rc = iota.alloc(max_items * 4)) != HS_OK)
      return rc;
    iota_kernel<<<(unsigned)((max_items + 255) / 256), 256, 0, st>>>(iota.as<uint32_t>(), (uint32_t)max_items);
    GB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                            (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)max_items, 0, 32, st));
    return temp.alloc(temp_bytes);
  }
  int sort(const uint32_t *keys_in, size_t items, int end_bit, cudaStream_t st) {
    GB_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, temp_bytes, keys_in, keys_out.as<uint32_t>(), iota.as<uint32_t>(),
                                            vals_out.as<uint32_t>(), (int)items, 0, end_bit, st));
    return HS_OK;
  }
};

struct GpuHnsw {                       // phase-1 result, device resident
  uint32_t n = 0, n_upper = 0;
  int maxlevel = 0;
  uint32_t ep = 0;
  uint32_t M = 0, maxM = 0, maxM0 = 0, efc = 0;
  uint32_t stride0 = 0, ustride = 0;
  std::vector<int8_t> levels;          // host copy
  std::vector<uint32_t> level_count;   // [maxlevel + 1]
  std::vector<int32_t> h_slot;         // host copy of upper_slot
  std::vector<uint32_t> h_order_up;    // slot -> node
  DevBuf adj0, slot, order_up, d_levels;
  DevBuf up[kMaxLevels];
};

int draw_levels(GpuHnsw &g, size_t n, double branching, uint64_t seed) {
  const double mult = 1.0 / std::log(branching);   // hnsw.h:143-158
  g.levels.resize(n);
  int top = 0;
  for (size_t i = 0; i < n; ++i) {
    const double u = ((mix64(seed * 0x9E3779B9ull + i) >> 11) + 1) * (1.0 / 9007199254740993.0);   // (0,1)
    int l = (int)(-std::log(u) * mult);                                                              // hnsw.h:203-207
    l = std::min(l, kMaxLevels - 2);
    g.levels[i] = (int8_t)l;
    top = std::max(top, l);
  }
  g.maxlevel = top;
  return HS_OK;
}

// slots of the nodes with level > 0, level descending then id ascending (the loader's order, graph_loader.cpp)
int assign_slots(GpuHnsw &g) {
  const size_t n = g.levels.size();
  g.n = (uint32_t)n;
  g.level_count.assign(g.maxlevel + 2, 0);
  std::vector<uint32_t> &up = g.h_order_up;
  up.clear();
  for (size_t i = 0; i < n; ++i) {
    for (int l = 0; l <= g.levels[i]; ++l) g.level_count[l]++;
    if (g.levels[i] > 0) up.push_back((uint32_t)i);
  }
  std::stable_sort(up.begin(), up.end(), [&](uint32_t a, uint32_t b) { return g.levels[a] > g.levels[b]; });
  g.n_upper = (uint32_t)up.size();
  g.h_slot.assign(n, -1);
  for (uint32_t s = 0; s < up.size(); ++s) g.h_slot[up[s]] = (int32_t)s;
  g.ep = up.empty() ? 0u : up[0];
  int rc;
  if ((rc = g.slot.alloc(n * 4)) != HS_OK || (rc = g.order_up.alloc(std::max<size_t>(1, up.size()) * 4)) != HS_OK ||
      (rc = g.d_levels.alloc(n)) != HS_OK)
    return rc;
  GB_CUDA(cudaMemcpy(g.slot.p, g.h_slot.data(), n * 4, cudaMemcpyHostToDevice));
  if (!up.empty()) GB_CUDA(cudaMemcpy(g.order_up.p, up.data(), up.size() * 4, cudaMemcpyHostToDevice));
  GB_CUDA(cudaMemcpy(g.d_levels.p, g.levels.data(), n, cudaMemcpyHostToDevice));
  return HS_OK;
}

int build_hnsw_gpu(const float4 *d_vec, uint32_t row_chunks, size_t n, int metric, size_t M, size_t efc_in,
                   double branching, uint64_t seed, cudaStream_t st, GpuHnsw *out) {
  GpuHnsw &g = *out;
  g.M = (uint32_t)M;
  g.maxM = (uint32_t)M;
  g.maxM0 = (uint32_t)(2 * M);                       // hnsw.h:108-109
  g.efc = (uint32_t)std::max(efc_in, M);             // hnsw.h:110
  if (M < 2 || M > 32 || g.efc > 256) {
    set_error("GPU builder: needs 2 <= M <= 32 and ef_construction <= 256 (use the host builder otherwise)");
    return HS_ERR_UNSUPPORTED;
  }
  int rc;
  if ((rc = draw_levels(g, n, branching, seed)) != HS_OK || (rc = assign_slots(g)) != HS_OK) return rc;
  g.stride0 = round_up(g.maxM0, 32);
  g.ustride = round_up(g.maxM, 32);
  if ((rc = g.adj0.alloc(n * (size_t)g.stride0 * 4)) != HS_OK) return rc;
  GB_CUDA(cudaMemsetAsync(g.adj0.p, 0xff, n * (size_t)g.stride0 * 4, st));
  for (int l = 1; l <= g.maxlevel; ++l) {
    if ((rc = g.up[l].alloc((size_t)g.level_count[l] * g.ustride * 4)) != HS_OK) return rc;
    GB_CUDA(cudaMemsetAsync(g.up[l].p, 0xff, (size_t)g.level_count[l] * g.ustride * 4, st));
  }
  // insertion order of level 0: the nodes with slots first (slot order), then the level-0-only nodes by id
  DevBuf order0;
  {
    std::vector<uint32_t> o(n);
    std::copy(g.h_order_up.begin(), g.h_order_up.end(), o.begin());
    size_t w = g.h_order_up.size();
    for (size_t i = 0; i < n; ++i)
      if (g.levels[i] == 0) o[w++] = (uint32_t)i;
    if ((rc = order0.alloc(n * 4)) != HS_OK) return rc;
    GB_CUDA(cudaMemcpy(order0.p, o.data(), n * 4, cudaMemcpyHostToDevice));
  }
  constexpr uint32_t kBatchMax = 16384;
  DevBuf req_target, req_src, req_dist;
  const size_t req_cap = (size_t)kBatchMax * g.M;
  if ((rc = req_target.alloc(req_cap * 4)) != HS_OK || (rc = req_src.alloc(req_cap * 4)) != HS_OK ||
      (rc = req_dist.alloc(req_cap * 4)) != HS_OK)
    return rc;
  Sorter sorter;
  if ((rc = sorter.prepare(req_cap, st)) != HS_OK) return rc;
  int key_bits = 1;
  while ((1ull << key_bits) < n) ++key_bits;
  // kInvalid targets must sort last: sort on all 32 bits when the batch may contain empty requests
  const int end_bit = 32;
  (void)key_bits;

  return dispatch_cm(row_chunks, metric, [&](auto C, auto Mt) -> int {
    constexpr int CPL = decltype(C)::value, MET = decltype(Mt)::value;
    auto ins = insert_kernel<CPL, MET>;
    auto back = backlink_kernel<CPL, MET>;
    const size_t qbytes = CPL == 0 ? (size_t)row_chunks * 16 : 0;
    const size_t ins_smem = (4u << kHashBits) + 128 + qbytes;
    const size_t back_smem = 4 * qbytes;
    GB_CUDA(cudaFuncSetAttribute(ins, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ins_smem));
    GB_CUDA(cudaFuncSetAttribute(back, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(back_smem, 16)));
    for (int layer = g.maxlevel; layer >= 0; --layer) {
      const uint32_t members = layer == 0 ? (uint32_t)n : g.level_count[layer];
      InsertParams ip{};
      ip.vec = d_vec;
      ip.row_chunks = row_chunks;
      ip.n = (uint32_t)n;
      ip.adj = layer == 0 ? g.adj0.as<uint32_t>() : g.up[layer].as<uint32_t>();
      ip.stride = layer == 0 ? g.stride0 : g.ustride;
      ip.slot = g.slot.as<int32_t>();
      ip.layer = layer;
      ip.maxlevel = g.maxlevel;
      for (int l = 1; l <= g.maxlevel; ++l) ip.upper_adj[l] = g.up[l].as<uint32_t>();
      ip.ustride = g.ustride;
      ip.ep = g.ep;
      ip.order = layer == 0 ? order0.as<uint32_t>() : g.order_up.as<uint32_t>();
      ip.M = g.M;
      ip.efc = g.efc;
      ip.req_target = req_target.as<uint32_t>();
      ip.req_src = req_src.as<uint32_t>();
      ip.req_dist = req_dist.as<float>();
      BacklinkParams bp{};
      bp.vec = d_vec;
      bp.row_chunks = row_chunks;
      bp.adj = ip.adj;
      bp.stride = ip.stride;
      bp.slot = ip.slot;
      bp.layer = layer;
      bp.Mmax = layer == 0 ? g.maxM0 : g.maxM;
      bp.keys = sorter.keys_out.as<uint32_t>();
      bp.vals = sorter.vals_out.as<uint32_t>();
      bp.req_src = ip.req_src;
      bp.req_dist = ip.req_dist;
      uint32_t frontier = 1;                       // position 0 (the entry point) starts every layer alone
      while (frontier < members) {
        const uint32_t batch = std::min({members - frontier, kBatchMax, std::max(1u, frontier / 16)});
        ip.frontier = frontier;
        ip.batch = batch;
        ins<<<batch, 32, ins_smem, st>>>(ip);
        const uint32_t nreq = batch * g.M;
        int rc2 = sorter.sort(ip.req_target, nreq, end_bit, st);
        if (rc2 != HS_OK) return rc2;
        bp.nreq = nreq;
        back<<<(nreq + 3) / 4, 128, std::max<size_t>(back_smem, 16), st>>>(bp);
        frontier += batch;
      }
      GB_CUDA(cudaGetLastError());
    }
    GB_CUDA(cudaStreamSynchronize(st));
    return HS_OK;
  });
}

// A device-resident slim graph (phase-2 result), in the engine's HBM layout
struct GpuSlim {
  DevBuf adj0;
  DevBuf up[kMaxLevels];
  uint32_t deg0_stride = 32, upper_stride = 8, max_deg0 = 0, max_deg_up = 0;
  uint64_t sum_deg0 = 0;
};

struct ConvertParams {
  int threshold_level;
  float top_pct0, top_pct;
  uint32_t top_M0, low_m0, top_M, low_m;
};

// convertFromHNSW on the device.  h_adj / strides describe the HNSW lists (kInvalid-padded rows).
int convert_gpu(const float4 *d_vec, uint32_t row_chunks, int metric, const GpuHnsw &g, const uint32_t *h0,
                uint32_t h0_stride, const uint32_t *const *hup, uint32_t hup_stride, const ConvertParams &cp,
                cudaStream_t st, GpuSlim *out) {
  const uint32_t n = g.n;
  int rc;
  DevBuf stats, maxdeg;
  if ((rc = stats.alloc(16)) != HS_OK || (rc = maxdeg.alloc(4)) != HS_OK) return rc;
  // degree thresholds of the upper levels (slim.h:905-947); level 0: the population count is never
  // accumulated there (:908-921 counts levels >= 1 only), so topN = 0, the threshold lands on maxM0 + 1
  // and every level-0 list is pruned to low_m0
  std::vector<uint32_t> deg_thr(g.maxlevel + 1, 0);
  deg_thr[0] = g.maxM0 + 1;
  for (int l = 1; l <= g.maxlevel; ++l) {
    const size_t rows = g.level_count[l];
    std::vector<uint32_t> rowsh(rows * hup_stride);
    GB_CUDA(cudaMemcpyAsync(rowsh.data(), hup[l], rowsh.size() * 4, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaStreamSynchronize(st));
    std::vector<size_t> hist(g.maxM0 + 2, 0);
    for (size_t r = 0; r < rows; ++r) {
      uint32_t c = 0;
      for (uint32_t j = 0; j < hup_stride; ++j) c += rowsh[r * hup_stride + j] != kInvalid;
      hist[std::min<uint32_t>(c, g.maxM0 + 1)]++;
    }
    const size_t topN = (size_t)(rows * cp.top_pct + 0.5);
    size_t acc = 0;
    for (size_t d = hist.size() - 1; d > 0; --d) {
      acc += hist[d];
      if (acc >= topN) {
        deg_thr[l] = (uint32_t)d;
        break;
      }
    }
  }
  const uint32_t cap0 = round_up(std::max(g.maxM0, 1u), 32), capu = round_up(std::max(g.maxM, 1u), 32);
  if (cap0 > 64 || capu > 64 || cp.top_M0 > 64 || cp.low_m0 > 64 || cp.top_M > 64 || cp.low_m > 64) {
    set_error("GPU conversion: list capacities above 64 are not supported");
    return HS_ERR_UNSUPPORTED;
  }
  return dispatch_cm(row_chunks, metric, [&](auto C, auto Mt) -> int {
    constexpr int CPL = decltype(C)::value, MET = decltype(Mt)::value;
    auto prune = prune_kernel<CPL, MET>;
    auto merge = merge_kernel<CPL, MET>;
    const size_t qbytes = CPL == 0 ? (size_t)row_chunks * 16 : 0;
    const size_t prune_smem = std::max<size_t>(4 * qbytes, 16), merge_smem = kMergeCap * 8 + qbytes;
    GB_CUDA(cudaFuncSetAttribute(prune, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prune_smem));
    GB_CUDA(cudaFuncSetAttribute(merge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)merge_smem));
    DevBuf seg_begin, seg_end;
    int rc2;
    if ((rc2 = seg_begin.alloc((size_t)n * 4)) != HS_OK || (rc2 = seg_end.alloc((size_t)n * 4)) != HS_OK) return rc2;
    for (int l = 0; l <= g.maxlevel; ++l) {
      const uint32_t rows = l == 0 ? n : g.level_count[l];
      const uint32_t keep_low = l == 0 ? cp.low_m0 : cp.low_m, keep_top = l == 0 ? cp.top_M0 : cp.top_M;
      // level 0 never takes the top branch (threshold maxM0 + 1): its request table only needs keep_low columns
      const uint32_t keep_cap = l == 0 ? keep_low : std::max(keep_low, keep_top);
      const uint32_t nstride = round_up(std::max(keep_cap, 1u), 32);
      const size_t nreq = (size_t)rows * keep_cap;
      if (nreq >= (1ull << 31)) {
        set_error("GPU conversion: too many reverse-edge requests for one level");
        return HS_ERR_UNSUPPORTED;
      }
      DevBuf nbr1, req_target, req_src, rev_src;
      Sorter sorter;
      if ((rc2 = nbr1.alloc((size_t)rows * nstride * 4)) != HS_OK || (rc2 = req_target.alloc(nreq * 4)) != HS_OK ||
          (rc2 = req_src.alloc(nreq * 4)) != HS_OK || (rc2 = rev_src.alloc(nreq * 4)) != HS_OK ||
          (rc2 = sorter.prepare(std::max<size_t>(nreq, 1), st)) != HS_OK)
        return rc2;
      PruneParams pp{};
      pp.vec = d_vec;
      pp.row_chunks = row_chunks;
      pp.adj = l == 0 ? h0 : hup[l];
      pp.stride = l == 0 ? h0_stride : hup_stride;
      pp.rows = rows;
      pp.node_of_row = l == 0 ? nullptr : g.order_up.as<uint32_t>();
      pp.keep_low = keep_low;
      pp.keep_top = keep_top;
      pp.deg_threshold = deg_thr[l];
      pp.nbr1 = nbr1.as<uint32_t>();
      pp.nstride = nstride;
      pp.req_target = req_target.as<uint32_t>();
      pp.req_src = req_src.as<uint32_t>();
      pp.keep_cap = keep_cap;
      prune<<<(rows + 3) / 4, 128, prune_smem, st>>>(pp);
      if (nreq) {
        if ((rc2 = sorter.sort(req_target.as<uint32_t>(), nreq, 32, st)) != HS_OK) return rc2;
        gather_u32_kernel<<<(unsigned)((nreq + 255) / 256), 256, 0, st>>>(req_src.as<uint32_t>(), sorter.vals_out.as<uint32_t>(),
                                                                         (uint32_t)nreq, rev_src.as<uint32_t>());
      }
      GB_CUDA(cudaMemsetAsync(seg_begin.p, 0, (size_t)n * 4, st));
      GB_CUDA(cudaMemsetAsync(seg_end.p, 0, (size_t)n * 4, st));
      if (nreq)
        segment_bounds_kernel<<<(unsigned)((nreq + 255) / 256), 256, 0, st>>>(sorter.keys_out.as<uint32_t>(), (uint32_t)nreq,
                                                                             seg_begin.as<uint32_t>(), seg_end.as<uint32_t>());
      const uint32_t limit = l == 0 ? g.maxM0 : g.maxM;
      const uint32_t ocap = round_up(limit, 32);
      DevBuf wide;
      if ((rc2 = wide.alloc((size_t)rows * ocap * 4)) != HS_OK) return rc2;
      GB_CUDA(cudaMemsetAsync(stats.p, 0, 16, st));
      GB_CUDA(cudaMemsetAsync(maxdeg.p, 0, 4, st));
      MergeParams mp{};
      mp.vec = d_vec;
      mp.row_chunks = row_chunks;
      mp.rows = rows;
      mp.node_of_row = pp.node_of_row;
      mp.nbr1 = nbr1.as<uint32_t>();
      mp.nstride = nstride;
      mp.seg_begin = seg_begin.as<uint32_t>();
      mp.seg_end = seg_end.as<uint32_t>();
      mp.rev_src = rev_src.as<uint32_t>();
      mp.limit = limit;
      mp.levels = g.d_levels.as<int8_t>();
      mp.level = l;
      mp.threshold_level = cp.threshold_level;
      mp.out = wide.as<uint32_t>();
      mp.ostride = ocap;
      mp.sum_deg = stats.as<unsigned long long>();
      mp.max_deg = maxdeg.as<uint32_t>();
      merge<<<rows, 32, merge_smem, st>>>(mp);
      unsigned long long hstats[2] = {0, 0};
      uint32_t hmax = 0;
      GB_CUDA(cudaMemcpyAsync(hstats, stats.p, 16, cudaMemcpyDeviceToHost, st));
      GB_CUDA(cudaMemcpyAsync(&hmax, maxdeg.p, 4, cudaMemcpyDeviceToHost, st));
      GB_CUDA(cudaStreamSynchronize(st));
      GB_CUDA(cudaGetLastError());
      if (hstats[1]) {
        set_error("GPU conversion: " + std::to_string(hstats[1]) + " nodes have more than " + std::to_string(kMergeCap) +
                  " candidate neighbours after the reverse-edge merge");
        return HS_ERR_UNSUPPORTED;
      }
      if (l == 0) {
        out->max_deg0 = hmax;
        out->sum_deg0 = hstats[0];
        out->deg0_stride = std::max<uint32_t>(32, round_up(hmax, 32));
        if (out->deg0_stride == ocap) {
          out->adj0.p = wide.release();
        } else {
          if ((rc2 = out->adj0.alloc((size_t)rows * out->deg0_stride * 4)) != HS_OK) return rc2;
          const size_t tot = (size_t)rows * out->deg0_stride;
          restride_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(wide.as<uint32_t>(), ocap, out->adj0.as<uint32_t>(),
                                                                        out->deg0_stride, rows);
          GB_CUDA(cudaStreamSynchronize(st));
        }
      } else {
        out->max_deg_up = std::max(out->max_deg_up, hmax);
        out->up[l].p = wide.release();           // restrided once every level's maximum is known
      }
    }
    out->upper_stride = std::max<uint32_t>(8, round_up(out->max_deg_up, 8));
    for (int l = 1; l <= g.maxlevel; ++l) {
      const uint32_t rows = g.level_count[l], ocap = round_up(g.maxM, 32);
      if (out->upper_stride == ocap) continue;
      DevBuf narrow;
      if ((rc2 = narrow.alloc((size_t)rows * out->upper_stride * 4)) != HS_OK) return rc2;
      const size_t tot = (size_t)rows * out->upper_stride;
      restride_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(out->up[l].as<uint32_t>(), ocap, narrow.as<uint32_t>(),
                                                                    out->upper_stride, rows);
      GB_CUDA(cudaStreamSynchronize(st));
      std::swap(out->up[l].p, narrow.p);
    }
    GB_CUDA(cudaGetLastError());
    return HS_OK;
  });
}

}  // namespace

// ---- entry points used by hs_api.cu ----
namespace {

// phase 2 and the hand-over: convertFromHNSW over g's lists (adj0 / up[l], strides stride0 / ustride), then the
// vector store, the slots and the slim lists move into `dg`
int convert_into_device_graph(DevBuf &vec, size_t n, size_t dim, size_t dim_padded, int metric, GpuHnsw &g,
                              const hs_build_params *bp, cudaStream_t st, DeviceGraph *dg) {
  const uint32_t row_chunks = (uint32_t)(dim_padded / 4);
  ConvertParams cp{bp->threshold_level, bp->top_degree_percent0, bp->top_degree_percent, (uint32_t)bp->top_M0,
                   (uint32_t)bp->low_m0, (uint32_t)bp->top_M, (uint32_t)bp->low_m};
  GpuSlim s;
  const uint32_t *hup[kMaxLevels] = {};
  for (int l = 1; l <= g.maxlevel; ++l) hup[l] = g.up[l].as<uint32_t>();
  const int rc = convert_gpu(vec.as<float4>(), row_chunks, metric, g, g.adj0.as<uint32_t>(), g.stride0, hup, g.ustride, cp, st, &s);
  if (rc != HS_OK) return rc;
  dg->n = n;
  dg->dim = dim;
  dg->dim_padded = dim_padded;
  dg->metric = metric;
  dg->M = g.M;
  dg->maxM = g.maxM;
  dg->maxM0 = g.maxM0;
  dg->ef_construction = g.efc;
  dg->maxlevel = g.maxlevel;
  dg->threshold_level = bp->threshold_level;
  dg->enterpoint = g.ep;
  dg->deg0_stride = s.deg0_stride;
  dg->max_deg0 = s.max_deg0;
  dg->upper_stride = s.upper_stride;
  dg->n_upper = g.n_upper;
  dg->sum_deg0 = s.sum_deg0;
  for (int l = 0; l <= g.maxlevel; ++l) dg->level_count[l] = g.level_count[l];
  dg->d_vec = static_cast<float *>(vec.release());
  dg->d_adj0 = static_cast<uint32_t *>(s.adj0.release());
  dg->d_upper_slot = static_cast<int32_t *>(g.slot.release());
  for (int l = 1; l <= g.maxlevel; ++l) dg->d_upper_adj[l] = static_cast<uint32_t *>(s.up[l].release());
  return HS_OK;
}

// rows -> HNSW -> HNSW-Slim lists, all on the device; fills `dg` (ownership of the arrays moves to it)
int build_slim_device_graph(const float *base, size_t n, size_t dim, int metric, const hs_build_params *bp,
                            double branching, int device, cudaStream_t st, DeviceGraph *dg) {
  const size_t dim_padded = (dim + kRowAlignFloats - 1) / kRowAlignFloats * kRowAlignFloats;
  const uint32_t row_chunks = (uint32_t)(dim_padded / 4);
  int rc;
  // the vector store: 128-byte rows, zero padded (DESIGN.md "HBM layout")
  DevBuf vec;
  if ((rc = vec.alloc(n * dim_padded * 4)) != HS_OK) return rc;
  {
    cudaPointerAttributes a{};
    const bool on_device = cudaPointerGetAttributes(&a, base) == cudaSuccess &&
                           (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (dim_padded == dim) {
      GB_CUDA(cudaMemcpyAsync(vec.p, base, n * dim * 4, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    } else if (on_device) {
      const size_t tot = n * dim_padded;
      pad_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(base, (uint32_t)dim, vec.as<float>(), (uint32_t)dim_padded, n);
    } else {
      GB_CUDA(cudaMemsetAsync(vec.p, 0, n * dim_padded * 4, st));
      GB_CUDA(cudaMemcpy2DAsync(vec.p, dim_padded * 4, base, dim * 4, dim * 4, n, cudaMemcpyHostToDevice, st));
    }
    GB_CUDA(cudaStreamSynchronize(st));
  }
  GpuHnsw g;
  rc = build_hnsw_gpu(vec.as<float4>(), row_chunks, n, metric, bp->M, bp->ef_construction, branching, bp->seed, st, &g);
  if (rc != HS_OK) return rc;
  return convert_into_device_graph(vec, n, dim, dim_padded, metric, g, bp, st, dg);
}

// The un-pruned lists of an hs_build_hnsw_graph file as a phase-1 result: the file's levels, entry point and
// M / maxM / maxM0, the loader's slot order (= assign_slots'), and rows re-strided to the widths the phase-2
// kernels read (round_up(maxM0 | maxM, 32) ids, kInvalid-padded).
int device_hnsw_from_file(const HostGraph &h, cudaStream_t st, GpuHnsw *out) {
  GpuHnsw &g = *out;
  g.M = (uint32_t)h.M;
  g.maxM = (uint32_t)h.maxM;
  g.maxM0 = (uint32_t)h.maxM0;
  g.efc = (uint32_t)h.ef_construction;
  g.levels = h.levels;
  g.maxlevel = h.maxlevel;
  int rc;
  if ((rc = assign_slots(g)) != HS_OK) return rc;
  g.ep = h.enterpoint;
  g.stride0 = round_up(g.maxM0, 32);
  g.ustride = round_up(g.maxM, 32);
  auto upload_rows = [&](const std::vector<uint32_t> &src, uint32_t sstride, size_t rows, uint32_t dstride,
                         DevBuf &dst) -> int {
    std::vector<uint32_t> w(rows * dstride, kInvalid);
    const uint32_t c = std::min(sstride, dstride);
    for (size_t r = 0; r < rows; ++r) std::memcpy(&w[r * dstride], &src[r * sstride], 4 * (size_t)c);
    int rc2;
    if ((rc2 = dst.alloc(w.size() * 4)) != HS_OK) return rc2;
    GB_CUDA(cudaMemcpyAsync(dst.p, w.data(), w.size() * 4, cudaMemcpyHostToDevice, st));
    GB_CUDA(cudaStreamSynchronize(st));
    return HS_OK;
  };
  if ((rc = upload_rows(h.adj0, h.deg0_stride, h.n, g.stride0, g.adj0)) != HS_OK) return rc;
  for (int l = 1; l <= g.maxlevel; ++l)
    if ((rc = upload_rows(h.upper_adj[l], h.upper_stride, g.level_count[l], g.ustride, g.up[l])) != HS_OK) return rc;
  return HS_OK;
}

void free_device_graph(DeviceGraph &dg) {
  cudaFree(dg.d_vec);
  cudaFree(dg.d_adj0);
  cudaFree(dg.d_upper_slot);
  for (auto *p : dg.d_upper_adj) cudaFree(p);
  cudaFree(dg.d_qrec);
  cudaFree(dg.d_centroids);
  cudaFree(dg.d_flip);
  dg = DeviceGraph();
}

struct StreamGuard {
  cudaStream_t s;
  ~StreamGuard() { cudaStreamDestroy(s); }
};

}  // namespace

int gpu_build_slim_index(const float *base, size_t n, size_t dim, int metric, const hs_build_params *bp,
                         double branching, const uint64_t *labels, int device, hs_index **out_ix) {
  if (!base || n == 0 || dim == 0 || n >= (1ull << 31) || !bp || !out_ix) {
    set_error("hs_build_slim_index_gpu: bad argument");
    return HS_ERR_ARG;
  }
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  cudaStream_t st = nullptr;
  GB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  StreamGuard guard{st};
  DeviceGraph dg;
  if ((rc = build_slim_device_graph(base, n, dim, metric, bp, branching, device, st, &dg)) != HS_OK) {
    free_device_graph(dg);
    return rc;
  }
  std::vector<uint32_t> lab(n);
  for (size_t i = 0; i < n; ++i) lab[i] = labels ? (uint32_t)labels[i] : (uint32_t)i;     // truncated as slim.h:2129
  dg.h_labels = lab.data();
  return adopt_device_graph(dg, device, out_ix);
}

// phase 2 of gpu_build_slim_index over the lists of an hs_build_hnsw_graph file (hs_debug_convert_gpu)
int gpu_debug_convert(const char *hnsw_graph_path, size_t dim, int metric, const hs_build_params *bp, int device,
                      hs_index **out_ix) {
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  HostGraph h;
  {
    std::vector<uint8_t> bytes;
    if ((rc = read_file(hnsw_graph_path, &bytes)) != HS_OK) return rc;
    if ((rc = parse_graph(bytes.data(), bytes.size(), HS_KIND_HNSW, dim, &h)) != HS_OK) return rc;
  }
  if (h.n == 0) {
    set_error("hs_debug_convert_gpu: the index is empty");
    return HS_ERR_ARG;
  }
  cudaStream_t st = nullptr;
  GB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  StreamGuard guard{st};
  DeviceGraph dg;
  {
    DevBuf vec;
    GpuHnsw g;
    if ((rc = vec.alloc(h.vec.size() * 4)) != HS_OK) return rc;
    GB_CUDA(cudaMemcpyAsync(vec.p, h.vec.data(), h.vec.size() * 4, cudaMemcpyHostToDevice, st));
    if ((rc = device_hnsw_from_file(h, st, &g)) != HS_OK ||
        (rc = convert_into_device_graph(vec, h.n, dim, h.dim_padded, metric, g, bp, st, &dg)) != HS_OK) {
      free_device_graph(dg);
      return rc;
    }
  }
  dg.h_labels = h.labels.data();
  return adopt_device_graph(dg, device, out_ix);
}

// hnsw_slimq on the device: the hnsw_slim graph over the raw rows (as the host builder, graph_build.cpp), the
// centroids from Lloyd iterations on a host-side sample of the rows (the reference reads them from files no
// code of it produces, hnsw_slimq_strategy.h:42-45) or as given, and one kernel for every node's cluster id,
// rotation, 1-bit code and factors, written straight into the engine's 8-byte-word records.
int gpu_build_slimq_index(const float *base, size_t n, size_t dim, const hs_build_params *bp, double branching,
                          const float *centroids, size_t num_cluster, const uint64_t *labels, int device,
                          hs_index **out_ix) {
  if (!base || n == 0 || dim == 0 || n >= (1ull << 31) || !bp || !out_ix || num_cluster == 0 || num_cluster > 4096) {
    set_error("hs_build_slimq_index_gpu: bad argument");
    return HS_ERR_ARG;
  }
  const size_t pd = (dim + 63) / 64 * 64, words = pd / 64;     // rabitqlib/index/hnsw/hnsw.hpp:424-427
  size_t td = 1;
  while (td * 2 <= dim) td *= 2;                                // rotator.hpp:233-235
  if (td < 64 || pd > 2048) {
    set_error("hs_build_slimq_index_gpu: dim must be in [64, 2048] (FhtKacRotator, rotator.hpp:237-258)");
    return HS_ERR_UNSUPPORTED;
  }
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  cudaStream_t st = nullptr;
  GB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  StreamGuard guard{st};
  DeviceGraph dg;
  if ((rc = build_slim_device_graph(base, n, dim, HS_METRIC_L2, bp, branching, device, st, &dg)) != HS_OK) {
    free_device_graph(dg);
    return rc;
  }
  auto fail = [&](int code) {
    free_device_graph(dg);
    return code;
  };
  // centroids: given, or k-means over an evenly spaced sample of at most 200k rows
  std::vector<float> cent(num_cluster * dim);
  if (centroids) {
    std::memcpy(cent.data(), centroids, cent.size() * 4);
  } else {
    const size_t sample = std::min<size_t>(n, 200000), stride = n / sample;
    std::vector<float> rows(sample * dim);
    if (cudaMemcpy2D(rows.data(), dim * 4, dg.d_vec, dg.dim_padded * 4 * stride, dim * 4, sample, cudaMemcpyDeviceToHost) !=
        cudaSuccess) {
      set_error(std::string("hs_build_slimq_index_gpu: sample download: ") + cudaGetErrorString(cudaGetLastError()));
      return fail(HS_ERR_CUDA);
    }
    std::vector<uint32_t> ids;
    host_kmeans(rows.data(), sample, dim, num_cluster, 8, bp->seed, 0, cent, ids);
  }
  std::vector<uint8_t> flip(4 * pd / 8);          // the host builder's sign bits (graph_build.cpp)
  for (size_t i = 0; i < flip.size(); ++i) flip[i] = (uint8_t)(mix64(bp->seed * 0xD1B54A32D192ED03ull + i) >> 56);
  std::vector<float> rcent(num_cluster * pd);
  for (size_t c = 0; c < num_cluster; ++c) host_rotate(&cent[c * dim], dim, pd, td, flip.data(), &rcent[c * pd]);
  DevBuf d_cent, d_rcent, d_flip, d_qrec, d_ferr;
  if ((rc = d_cent.alloc(cent.size() * 4)) != HS_OK || (rc = d_rcent.alloc(rcent.size() * 4)) != HS_OK ||
      (rc = d_flip.alloc(flip.size())) != HS_OK || (rc = d_qrec.alloc(n * (words + 2) * 8)) != HS_OK ||
      (rc = d_ferr.alloc(n * 4)) != HS_OK)
    return fail(rc);
  if (cudaMemcpyAsync(d_cent.p, cent.data(), cent.size() * 4, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(d_rcent.p, rcent.data(), rcent.size() * 4, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(d_flip.p, flip.data(), flip.size(), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    set_error(std::string("hs_build_slimq_index_gpu: upload: ") + cudaGetErrorString(cudaGetLastError()));
    return fail(HS_ERR_CUDA);
  }
  PayloadParams pp{};
  pp.vec = dg.d_vec;
  pp.n = (uint32_t)n;
  pp.dim = (uint32_t)dim;
  pp.dim_padded = (uint32_t)dg.dim_padded;
  pp.pd = (uint32_t)pd;
  pp.td = (uint32_t)td;
  pp.words = (uint32_t)words;
  pp.num_cluster = (uint32_t)num_cluster;
  pp.cent = d_cent.as<float>();
  pp.rcent = d_rcent.as<float>();
  pp.flip = d_flip.as<uint8_t>();
  pp.fac = 1.0f / std::sqrt((float)td);
  pp.qrec = d_qrec.as<uint2>();
  pp.f_error = d_ferr.as<float>();
  const size_t smem = 4 * pd * 4;
  if (cudaFuncSetAttribute(slimq_payload_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(HS_ERR_CUDA);
  slimq_payload_kernel<<<(unsigned)((n + 3) / 4), 128, smem, st>>>(pp);
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
    set_error(std::string("slimq_payload_kernel: ") + cudaGetErrorString(cudaGetLastError()));
    return fail(HS_ERR_CUDA);
  }
  // f_error stays on the host (hs_save_index writes it); d_ferr is freed on return
  dg.h_f_error.resize(n);
  if (cudaMemcpy(dg.h_f_error.data(), d_ferr.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
    set_error(std::string("hs_build_slimq_index_gpu: f_error download: ") + cudaGetErrorString(cudaGetLastError()));
    return fail(HS_ERR_CUDA);
  }
  dg.kind = HS_KIND_SLIMQ;
  dg.padded_dim_q = pd;
  dg.num_cluster = num_cluster;
  dg.trunc_dim = (uint32_t)td;
  dg.d_qrec = static_cast<uint2 *>(d_qrec.release());
  dg.d_centroids = static_cast<float *>(d_rcent.release());
  dg.d_flip = static_cast<uint8_t *>(d_flip.release());
  std::vector<uint32_t> lab(n);
  for (size_t i = 0; i < n; ++i) lab[i] = labels ? (uint32_t)labels[i] : (uint32_t)i;
  dg.h_labels = lab.data();
  return adopt_device_graph(dg, device, out_ix);
}

}  // namespace hs
