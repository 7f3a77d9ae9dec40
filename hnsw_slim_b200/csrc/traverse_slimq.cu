// hnsw_slimq graph traversal on sm_100a: one warp per query.
//
// Replaces, for a whole query batch, HierarchicalNSWSlimQ<float>::searchKnn
// (slimq.h:1810-1924):
//   1. per-query preparation (slimq.h:1816-1847): FHT-Kac rotation
//      (rq/utils/rotator.hpp:370-423), 4-bit scalar quantisation of the rotated query and
//      its bit-plane transpose (rq/index/query.hpp:127-156, rq/quantization/rabitq_impl.hpp:
//      379-432,534-581, rq/utils/space.hpp:1405-1516), distances to the cluster centroids;
//   2. greedy descent over the upper levels on ESTIMATED distances (slimq.h:1862-1901);
//   3. the sorted-buffer beam search of searchBaseLayerST (slimq.h:688-759): every level-0
//      neighbour of the expanded node is scored with the 1-bit RaBitQ estimator
//      (get_bin_est slimq.h:408-440 -> split_single_estdist rq/index/estimator.hpp:164-188 ->
//      warmup_ip_x0_q rq/utils/warmup_space.hpp:8-102: popcounts of code & query bit planes),
//      the expanded node itself is re-ranked with its exact fp32 distance (slimq.h:747-757).
//
// One lane scores one neighbour: its 32-byte record (two 64-bit code words, f_add, f_rescale,
// cluster id) is one sector, the query's bit planes sit in registers, so a hop reads
// 128 B of adjacency + deg x 32 B of codes + one raw row.  The reference's sorted buffer is the
// unsorted REDUX pool of the fp32 kernel (traverse_common.cuh) with duplicate entries allowed,
// exactly as SearchBuffer allows them (SURVEY.md §8a Q4); "visited" (marked on expansion,
// slimq.h:700-704) is "a flagged copy of the key is in the pool" — an expanded entry that left
// the pool is worse than the pool's worst from then on and is rejected by is_full() anyway.
// Results equal the reference's sequential algorithm except where two estimates (or two
// exact distances at the k-th boundary) tie bit for bit.
//
// Floating point: every operation is an explicit round-to-nearest intrinsic in the
// association oracle/hs_oracle_slimq.c spells out ("warp order" reductions), so the
// preparation, the estimates and the results are bit-identical to the oracle.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <type_traits>

#include "traverse_common.cuh"
#include "traverse_slimq.cuh"

namespace hs {
namespace {

#ifndef HS_SLIMQ_MIN_CTAS
#define HS_SLIMQ_MIN_CTAS 8
#endif
#ifndef HS_SLIMQ_EST32
#define HS_SLIMQ_EST32 1           // popcount sums of the estimator in 32-bit integers (one I2F each)
#endif
#ifndef HS_SLIMQ_BLOOM
#define HS_SLIMQ_BLOOM 1           // a 1024-bit Bloom word set (32 bits per lane) of the expanded nodes in front of the pool's duplicate scan
#endif
#ifndef HS_SLIMQ_TOPCACHE
#define HS_SLIMQ_TOPCACHE 0        // keep the exact-distance heap's worst distance in a register and skip the heap code
#endif

template <int SLOTS> struct QPoolSel { using type = RegPool32<SLOTS>; };
template <> struct QPoolSel<0> { using type = SmemPool; };

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = __fadd_rn(v, __shfl_xor_sync(FULL, v, off));
  return v;
}

// ---- the 1-bit estimator: one lane, one neighbour ----
// planes in registers (WREG == 2 words) or shared memory (any word count)
template <int WREG>
struct Planes {
  unsigned long long r[WREG > 0 ? WREG * 4 : 1];
  const unsigned long long *s;
};

template <int WREG>
__device__ __forceinline__ float estimate(const TraverseQParams &p, const Planes<WREG> &pl, float delta,
                                          float vl, float k1xsumq, const float *g2c, uint32_t id) {
  // popcount sums stay far below 2^24 (<= 15 * padded_dim, padded_dim <= 2048: hs_load): 32-bit integers, ONE
  // int-to-float conversion each (a 64-bit source would cost a multi-instruction conversion per estimate)
#if HS_SLIMQ_EST32
  uint32_t ip = 0, ppc = 0;
#else
  unsigned long long ip = 0, ppc = 0;
#endif
  float f_add, f_rescale;
  uint32_t cluster;
  if constexpr (WREG == 2) {
    const uint4 *rec = reinterpret_cast<const uint4 *>(p.qrec) + 2 * (size_t)id;
    const uint4 a = __ldg(rec), b = __ldg(rec + 1);
    const unsigned long long x0 = ((unsigned long long)a.y << 32) | a.x;
    const unsigned long long x1 = ((unsigned long long)a.w << 32) | a.z;
    ppc = (uint32_t)(__popcll(x0) + __popcll(x1));
#pragma unroll
    for (int j = 0; j < 4; ++j) ip += (uint32_t)(__popcll(x0 & pl.r[j]) + __popcll(x1 & pl.r[4 + j])) << j;
    f_add = __uint_as_float(b.x);
    f_rescale = __uint_as_float(b.y);
    cluster = b.z;
  } else {
    const uint2 *rec = p.qrec + (size_t)id * p.rec_words;
    for (uint32_t w = 0; w < p.words; ++w) {
      const uint2 c = __ldg(rec + w);
      const unsigned long long x = ((unsigned long long)c.y << 32) | c.x;
      ppc += (uint32_t)__popcll(x);
#pragma unroll
      for (int j = 0; j < 4; ++j) ip += (uint32_t)__popcll(x & pl.s[w * 4 + j]) << j;
    }
    const uint2 f = __ldg(rec + p.words), c = __ldg(rec + p.words + 1);
    f_add = __uint_as_float(f.x);
    f_rescale = __uint_as_float(f.y);
    cluster = c.x;
  }
  // warmup_space.hpp:101, estimator.hpp:185 (one rounding per operation, as the oracle)
  const float ipf = __fadd_rn(__fmul_rn(delta, (float)ip), __fmul_rn(vl, (float)ppc));
  return __fadd_rn(__fadd_rn(f_add, g2c[cluster]), __fmul_rn(f_rescale, __fadd_rn(ipf, k1xsumq)));
}

// ---- per-query preparation, whole warp; buf = padded_dim floats of shared memory ----
// Leaves the ROTATED query in buf, g2c[c] = ||q' - C_c||^2 (as sqrt then square, slimq.h:
// 1825-1832,428-437) in shared memory, the planes in pl, returns (delta, vl, k1xsumq).
template <int WREG>
__device__ __forceinline__ void prepare_query(const TraverseQParams &p, const float *qptr, float *buf,
                                              float *g2c, unsigned long long *planes_s, Planes<WREG> &pl,
                                              float &delta, float &vl, float &k1xsumq, int lane,
                                              float *dump_q2c) {
  const uint32_t pd = p.padded_dim, td = p.trunc_dim;
  for (uint32_t i = lane; i < pd; i += 32) buf[i] = i < p.dim ? __ldg(qptr + i) : 0.f;
  __syncwarp();
  // FhtKacRotator::rotate, rotator.hpp:370-423
  const bool pow2 = td == pd;
  const uint32_t start = pd - td;
  for (int r = 0; r < 4; ++r) {
    const uint8_t *fl = p.flip + (size_t)r * pd / 8;
    for (uint32_t i = lane; i < pd; i += 32)          // flip_sign, rotator.hpp:100-205
      if ((__ldg(fl + (i >> 3)) >> (i & 7)) & 1u) buf[i] = -buf[i];
    __syncwarp();
    float *seg = (!pow2 && (r & 1)) ? buf + start : buf;
    for (uint32_t h = 1; h < td; h <<= 1) {           // FWHT, butterfly distance 1, 2, 4, ...
      for (uint32_t idx = lane; idx < td / 2; idx += 32) {
        const uint32_t j = (idx / h) * 2 * h + (idx % h);
        const float u = seg[j], v = seg[j + h];
        seg[j] = __fadd_rn(u, v);
        seg[j + h] = __fsub_rn(u, v);
      }
      __syncwarp();
    }
    for (uint32_t i = lane; i < td; i += 32) seg[i] = __fmul_rn(seg[i], p.fht_fac);
    __syncwarp();
    if (!pow2) {                                       // kacs_walk, rotator.hpp:299-368
      for (uint32_t i = lane; i < pd / 2; i += 32) {
        const float x = buf[i], y = buf[i + pd / 2];
        buf[i] = __fadd_rn(x, y);
        buf[i + pd / 2] = __fsub_rn(x, y);
      }
      __syncwarp();
    }
  }
  if (!pow2) {
    for (uint32_t i = lane; i < pd; i += 32) buf[i] = __fmul_rn(buf[i], 0.25f);
    __syncwarp();
  }

  // SplitSingleQuery ctor (query.hpp:127-156) -> rabitq_scalar_impl (rabitq_impl.hpp:534-581)
  float s_sum = 0.f, s_nd = 0.f;
  for (uint32_t i = lane; i < pd; i += 32) {
    const float r = buf[i];
    s_sum = __fadd_rn(s_sum, r);
    s_nd = __fmaf_rn(r, r, s_nd);
  }
  const float sumq = warp_sum_f(s_sum);
  const float norm_data = __fsqrt_rn(warp_sum_f(s_nd));
  float s_uu = 0.f, s_ru = 0.f;
  for (uint32_t t = 0; t * 32 < pd; ++t) {
    const uint32_t i = t * 32 + lane;
    const float r = buf[i];
    const float o = norm_data > 0.f ? __fdiv_rn(fabsf(r), norm_data) : fabsf(r);
    int c = (int)__dadd_rn(__dmul_rn(p.t_const, (double)o), 1e-5);     // rabitq_impl.hpp:386-390
    c = c >= 8 ? 7 : c;
    if (r < 0.f) c = (~c) & 7;                                           // :424-429
    const int u = c + (r > 0.f ? 8 : 0);                                 // :51, :553-555
    const float ucb = __fadd_rn((float)u, -7.5f);
    s_uu = __fmaf_rn(ucb, ucb, s_uu);
    s_ru = __fmaf_rn(r, ucb, s_ru);
    // new_transpose_bin, space.hpp:1405-1516: dim 64 w + l  <->  bit 63 - l of word w
    const uint32_t w = t >> 1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned long long half = (unsigned long long)__brev(__ballot_sync(FULL, (u >> j) & 1));
      if constexpr (WREG > 0) {
#pragma unroll
        for (int ww = 0; ww < WREG; ++ww)
          if ((int)w == ww) pl.r[ww * 4 + j] = (t & 1) ? (pl.r[ww * 4 + j] | half) : (half << 32);
      } else {
        if (lane == 0) planes_s[w * 4 + j] = (t & 1) ? (planes_s[w * 4 + j] | half) : (half << 32);
      }
    }
  }
  const float norm_quan = __fsqrt_rn(warp_sum_f(s_uu));
  // norm_data == 0 (an all-zero query, or one whose squares underflow): the reference computes cosv = 0 / 0, so
  // delta, vl and every estimate are NaN, and a NaN key, f2ord(0x7fffffff) == 0xffffffff, is the pool's
  // "expanded / empty" marker: the base-layer search would stop at once and return one result and padding.
  // This departs from the reference on purpose and takes the limit cosv = 0 (delta = vl = 0): the estimate is
  // then f_add + ||c||^2, RaBitQ's estimate of ||x||^2, which is the distance to a zero query.  The oracle agrees.
  const float cosv = norm_data > 0.f ? __fdiv_rn(warp_sum_f(s_ru), __fmul_rn(norm_data, norm_quan)) : 0.f;
  delta = __fmul_rn(__fdiv_rn(norm_data, norm_quan), cosv);            // :567
  vl = __fmul_rn(delta, -7.5f);                                         // :574
  k1xsumq = __fmul_rn(sumq, -0.5f);                                     // query.hpp:133,138
  if constexpr (WREG == 0) pl.s = planes_s;

  for (uint32_t c = 0; c < p.num_cluster; ++c) {                        // slimq.h:1825-1832
    const float *cen = p.centroids + (size_t)c * pd;
    float acc = 0.f;
    for (uint32_t i = lane; i < pd; i += 32) {
      const float d = __fsub_rn(buf[i], __ldg(cen + i));
      acc = __fmaf_rn(d, d, acc);
    }
    const float norm = __fsqrt_rn(warp_sum_f(acc));
    if (lane == 0) {
      g2c[c] = __fmul_rn(norm, norm);
      if (dump_q2c) dump_q2c[c] = norm;
    }
  }
  __syncwarp();
}

template <int WREG, int SLOTS, int KREG>
__global__ void __launch_bounds__(128, HS_SLIMQ_MIN_CTAS)
traverse_slimq_kernel(const __grid_constant__ TraverseQParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  unsigned char *wbase = smem + (size_t)wid * p.smem_per_warp;
  float *buf = reinterpret_cast<float *>(wbase + p.off_buf);
  float *g2c = reinterpret_cast<float *>(wbase + p.off_g2c);
  unsigned long long *planes_s = reinterpret_cast<unsigned long long *>(wbase + p.off_planes);
  const uint32_t ef = p.ef;
  if (p.overlap) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // see traverse_fp32.cu

  bool acked = false;
  for (;;) {
    uint32_t qi = 0;
    if (lane == 0) qi = next_ticket(p.work_counter, p.launch_tag);
    qi = __shfl_sync(FULL, qi, 0);
    if (qi >= p.nq) break;
    if (!acked) {              // shard group: the table slot this launch writes must have been merged everywhere
      scatter_wait_acks(p.scatter, lane);
      acked = true;
    }
    const float *qptr = p.queries + (size_t)qi * p.dim;

    Planes<WREG> pl;
    float delta, vl, k1;
    prepare_query<WREG>(p, qptr, buf, g2c, planes_s, pl, delta, vl, k1, lane,
                        p.prep_q2c ? p.prep_q2c + (size_t)qi * p.num_cluster : nullptr);
    if (p.prep_rotated) {                               // hs_slimq_prepare: dump and stop
      for (uint32_t i = lane; i < p.padded_dim; i += 32) p.prep_rotated[(size_t)qi * p.padded_dim + i] = buf[i];
      if (lane == 0) {
        for (uint32_t w = 0; w < p.words * 4; ++w) {
          unsigned long long v;
          if constexpr (WREG > 0) {
            v = 0;
#pragma unroll
            for (int ww = 0; ww < WREG * 4; ++ww) v = ((int)w == ww) ? pl.r[ww] : v;
          } else {
            v = planes_s[w];
          }
          p.prep_planes[(size_t)qi * p.words * 4 + w] = v;
        }
        p.prep_scal[(size_t)qi * 3 + 0] = delta;
        p.prep_scal[(size_t)qi * 3 + 1] = vl;
        p.prep_scal[(size_t)qi * 3 + 2] = k1;
      }
      __syncwarp();
      continue;
    }
    // the raw query replaces the rotated one: only the exact rerank needs floats from here on
    __syncwarp();
    for (uint32_t i = lane; i < p.row_chunks * 4; i += 32) buf[i] = i < p.dim ? __ldg(qptr + i) : 0.f;
    __syncwarp();
    const float4 *qs = reinterpret_cast<const float4 *>(buf);

    auto est = [&](uint32_t id) -> float { return estimate<WREG>(p, pl, delta, vl, k1, g2c, id); };

    uint32_t ne = 0, nh = 0, nr = 0;

    // ---- entry point and greedy descent on estimates, slimq.h:1849-1901 ----
    uint32_t cur = p.enterpoint;
    float curdist = est(cur);
    ne = 1;
    for (int level = p.maxlevel; level > p.threshold_level; --level) {
      const uint32_t *ladj = p.upper_adj[level];
      bool changed = true;
      while (changed) {
        changed = false;
        const int slot = __ldg(p.upper_slot + cur);
        if (slot < 0) break;
        const uint32_t *row = ladj + (size_t)slot * p.upper_stride;
        bool any = false;
        for (uint32_t seg = 0; seg < p.upper_stride; seg += 32) {
          const uint32_t id = (seg + lane < p.upper_stride) ? __ldg(row + seg + lane) : kInvalid;
          const unsigned vm = __ballot_sync(FULL, id != kInvalid);
          if (vm == 0) break;                       // rows are packed front to back
          const int count = __popc(vm);
          any = true;
          const float d = id != kInvalid ? est(id) : 0.f;
          ne += (uint32_t)count;
          // sequential scan with strict '<' == first-index argmin
          uint64_t key = lane < count ? (((uint64_t)f2ord(d) << 32) | (uint32_t)lane) : ~0ull;
          key = warp_min_u64(key);
          const float best = ord2f((uint32_t)(key >> 32));
          const uint32_t best_id = __shfl_sync(FULL, id, (int)(key & 31));
          if (best < curdist) {
            curdist = best;
            cur = best_id;
            changed = true;
          }
        }
        if (any) nh++;
      }
    }

    // ---- base layer, slimq.h:688-759 ----
    typename QPoolSel<SLOTS>::type pool;
    pool.init(reinterpret_cast<uint64_t *>(wbase), ef, lane);
    pool.seed(make_key(curdist, cur));                  // search_pool_.insert(currObj, curdist), :1914
    using TopK = typename std::conditional<KREG != 0, RegPool<1>, SmemPool>::type;
    TopK top;
    top.init(reinterpret_cast<uint64_t *>(wbase + p.off_topk), p.k, lane);
    bool top_seeded = false;
#if HS_SLIMQ_TOPCACHE
    uint32_t top_worst_d = 0xffffffffu;       // distance word of the heap's worst key once it holds k entries
#endif
    // the exact-distance heap changes on few hops once it is full: its worst key is kept here and an expanded
    // node that cannot enter (slimq.h:750-757: pushed, then the heap is trimmed back to K) skips the heap code

    // "Was this neighbour expanded already?" is, for the pool, a scan of all its entries per admitted candidate
    // (admit_q).  Almost every answer is no: a 1024-bit Bloom filter of the expanded nodes — bit b of the set lives
    // in lane b / 32, so ONE shuffle hands every lane the word its own candidate hashes to — says so without the
    // scan; only a set bit (an expanded node, or one of the ~10 % false positives at ~100 expansions) goes on to
    // the exact test.  No false negatives, so results and counters are unchanged.  Measured on 1M x 96
    // (profiles/r02_probe_slimq_bloom.txt): ef=100 +1.2 %, ef=200 +5 %, ef=300 (shared-memory pool) +21 %, but
    // -2 % at ef=50, where the two-slot pool's scan is cheaper than the filter: not used there.
    constexpr bool kBloom = HS_SLIMQ_BLOOM && SLOTS != 2;
    uint32_t bloom = 0;
    auto bloom_bit = [](uint32_t id) { return (id * 0x9E3779B1u) >> 22; };
    for (;;) {
      const uint32_t node = pool.pop_closest_unexpanded_dups();
      if (node == kInvalid) break;
      if constexpr (kBloom) {
        const uint32_t b = bloom_bit(node);
        if ((uint32_t)lane == (b >> 5)) bloom |= 1u << (b & 31u);
      }
      const uint32_t *row = p.adj0 + (size_t)node * p.deg0_stride;
      uint32_t id = __ldg(row + lane);
      // the expanded node's raw row, for the exact rerank below (slimq.h:747-749): issued now so
      // that its DRAM latency hides behind the estimates and the pool update.  Lane t owns the
      // 4-float chunks t, t+32, ... (the oracle's HSO_ORDER_GPU association with team = 32).
      const float4 *xrow = p.vec + (size_t)node * p.row_chunks;
      float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f);
      if ((uint32_t)lane < p.row_chunks) x0 = __ldg(xrow + lane);

      bool any = false;
      for (uint32_t seg = 0; seg < p.deg0_stride; seg += 32) {
        if (seg) id = __ldg(row + seg + lane);
        const bool valid = id != kInvalid;
        const unsigned vm = __ballot_sync(FULL, valid);
        if (vm == 0) break;
        any = true;
        ne += (uint32_t)__popc(vm);
        const float d = valid ? est(id) : 0.f;
        unsigned maybe = FULL;
        if constexpr (kBloom) {
          const uint32_t hb = bloom_bit(id);
          const uint32_t bw = __shfl_sync(FULL, bloom, hb >> 5);
          maybe = __ballot_sync(FULL, valid && ((bw >> (hb & 31u)) & 1u));
        }
        const unsigned entered = pool.admit_q(valid, make_key(d, id), maybe);
        if ((entered >> lane) & 1u) prefetch_l2(p.adj0 + (size_t)id * p.deg0_stride);
      }
      if (p.flags & 1u) {
        // speculation: the entry that is now the closest unexpanded one is the likeliest next
        // pop; its adjacency row is (mostly) in L2 since its admission — pull the code records
        // of its neighbours towards L2 while this hop finishes
        const uint32_t nxt = pool.peek_closest_unexpanded();
        if (nxt != kInvalid) {
          const uint32_t nid = __ldg(p.adj0 + (size_t)nxt * p.deg0_stride + lane);
          if (nid != kInvalid) prefetch_l2(p.qrec + (size_t)nid * p.rec_words);
        }
      }
      if (!any) continue;                               // slimq.h:708-715: no neighbours, no rerank
      nh++;
      nr++;
      acc2_t acc2 = 0ull;
      if ((uint32_t)lane < p.row_chunks) acc2 = acc4<HS_METRIC_L2>(acc2, qs[lane], x0);
      for (uint32_t c = lane + 32; c < p.row_chunks; c += 32) acc2 = acc4<HS_METRIC_L2>(acc2, qs[c], __ldg(xrow + c));
      const float dx = warp_sum_f(sum2(acc2));
      const uint64_t xk = make_key(dx, node);
      if (!top_seeded) {
        top.seed(xk);
        top_seeded = true;
#if HS_SLIMQ_TOPCACHE
        if (p.k == 1) top_worst_d = (uint32_t)(xk >> 32);
      } else if ((uint32_t)(xk >> 32) <= top_worst_d) {       // ties on the distance word go through the exact test
        top.admit(lane == 0, xk);
        if (top.size >= p.k) top_worst_d = (uint32_t)(top.worst_key() >> 32);
      }
#else
      } else {
        top.admit(lane == 0, xk);
      }
#endif
    }

    // ---- results: the k closest expanded nodes by exact distance, ascending ----
    __syncwarp();
    {
      // lane i keeps result i; one coalesced store per row for k <= 32 (see traverse_fp32.cu)
      uint64_t last = 0;
      uint64_t mine_out = NONE;
      for (uint32_t i = 0; i < p.k; ++i) {
        const uint64_t mine = (last == NONE || !top_seeded) ? NONE : top.col_next_above(last);
        const int o = warp_argmin_key(mine);
        last = o >= 0 ? __shfl_sync(FULL, mine, o) : NONE;
        if ((uint32_t)lane == (i & 31u)) mine_out = last;
        if ((i & 31u) == 31u || i + 1 == p.k) {
          const uint32_t r = (i & ~31u) + (uint32_t)lane;
          if (r <= i) {
            const bool have = mine_out != NONE;
            const uint32_t out_l = have ? __ldg(p.labels + (uint32_t)mine_out) : 0xFFFFFFFFu;
            const float out_d = have ? ord2f((uint32_t)(mine_out >> 32)) : __int_as_float(0x7f800000);
            if (p.out_labels) p.out_labels[(size_t)qi * p.k + r] = out_l;
            if (p.out_dists) p.out_dists[(size_t)qi * p.k + r] = out_d;
            // sharded path: the same row goes straight into every rank's gather buffer
            for (uint32_t t = 0; t < p.scatter.n; ++t) {
              const size_t at = ((size_t)p.scatter.row0 + qi) * p.k + r;
              p.scatter.labels[t][at] = out_l;
              p.scatter.dists[t][at] = out_d;
            }
          }
          mine_out = NONE;
        }
      }
    }
    if (lane == 0) {
      atomicAdd(p.stats + 0, (unsigned long long)ne);
      atomicAdd(p.stats + 1, (unsigned long long)nh);
      atomicAdd(p.stats + 2, (unsigned long long)nr);
      if (p.per_query) {
        p.per_query[2 * (size_t)qi + 0] = ne;
        p.per_query[2 * (size_t)qi + 1] = nh;
      }
    }
    __syncwarp();
  }
  scatter_signal_done(p.scatter, lane);
}

inline int wreg_variant(uint32_t words) { return words == 2 ? 2 : 0; }
inline int slots_variant(uint32_t ef) { return ef <= 64 ? 2 : (ef <= 128 ? 4 : (ef <= 256 ? 8 : 0)); }
inline int kreg_variant(uint32_t k) { return k <= 32 ? 1 : 0; }

template <typename F>
int dispatch(int wreg, int slots, int kreg, F &&f) {
#define HS_CASE(W, S, K) \
  if (wreg == W && slots == S && kreg == K) return f(std::integral_constant<int, W>{}, std::integral_constant<int, S>{}, std::integral_constant<int, K>{});
#define HS_CASES_K(W, S) HS_CASE(W, S, 0) HS_CASE(W, S, 1)
#define HS_CASES_S(W) HS_CASES_K(W, 0) HS_CASES_K(W, 2) HS_CASES_K(W, 4) HS_CASES_K(W, 8)
  HS_CASES_S(0) HS_CASES_S(2)
#undef HS_CASES_S
#undef HS_CASES_K
#undef HS_CASE
  set_error("no hnsw_slimq kernel variant for this configuration");
  return HS_ERR_UNSUPPORTED;
}

inline uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

}  // namespace

int plan_traverse_slimq(TraverseQParams &p, int sm_count, int nq, TraverseQLaunch *out) {
  const int slv = slots_variant(p.ef), krv = kreg_variant(p.k), wrv = wreg_variant(p.words);
  const uint32_t pool_bytes = slv ? 0u : align_up(p.ef * 8u, 16);
  const uint32_t topk_bytes = krv ? 0u : align_up(p.k * 8u, 16);
  const uint32_t buf_floats = p.padded_dim > p.row_chunks * 4 ? p.padded_dim : p.row_chunks * 4;
  p.off_topk = pool_bytes;
  p.off_buf = p.off_topk + topk_bytes;
  p.off_g2c = p.off_buf + buf_floats * 4;
  p.off_planes = align_up(p.off_g2c + p.num_cluster * 4, 16);
  p.smem_per_warp = align_up(p.off_planes + (wrv ? 0u : p.words * 4 * 8), 16);
  if (p.smem_per_warp > 227u * 1024u) {
    set_error("ef / dim too large for the per-warp shared-memory working set");
    return HS_ERR_UNSUPPORTED;
  }
  // CTA shape: the smallest CTA that does not cost resident warps (see plan_traverse, traverse_fp32.cu)
  auto occupancy = [&](int w) {
    const size_t smem = (size_t)w * p.smem_per_warp;
    if (smem > 227u * 1024u) return 0;
    return dispatch(wrv, slv, krv, [&](auto W, auto S, auto K) {
      auto kern = traverse_slimq_kernel<decltype(W)::value, decltype(S)::value, decltype(K)::value>;
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, w * 32, smem) != cudaSuccess) nb = 0;
      return nb;
    });
  };
  int wpc = 1, per_sm = occupancy(1);
  for (int w = 2; w <= 4; w *= 2) {
    const int o = occupancy(w);
    if (o * w > per_sm * wpc) {
      wpc = w;
      per_sm = o;
    }
  }
  if (const char *w = std::getenv("HS_WPC")) {          // tuning knob
    wpc = std::max(1, std::min(4, std::atoi(w)));
    per_sm = occupancy(wpc);
  }
  out->warps_per_cta = wpc;
  out->smem_bytes = (size_t)wpc * p.smem_per_warp;
  if (per_sm <= 0) {
    set_error("traverse_slimq_kernel does not fit on an SM (cudaOccupancyMaxActiveBlocksPerMultiprocessor)");
    return HS_ERR_CUDA;
  }
  const int resident = sm_count * per_sm;
  const int need = (nq + wpc - 1) / wpc;
  out->grid = need < resident ? (need > 0 ? need : 1) : resident;
  return HS_OK;
}

int launch_traverse_slimq(const TraverseQParams &p, const TraverseQLaunch &l, cudaStream_t stream) {
  return dispatch(wreg_variant(p.words), slots_variant(p.ef), kreg_variant(p.k), [&](auto W, auto S, auto K) {
    auto kern = traverse_slimq_kernel<decltype(W)::value, decltype(S)::value, decltype(K)::value>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem_bytes);
    // HS_SLIMQ_CARVEOUT (tuning knob): preferred shared-memory carve-out in percent; the rest of the
    // 256 KB array is L1, which serves about half of this kernel's sector requests
    static const int carve = [] { const char *c = std::getenv("HS_SLIMQ_CARVEOUT"); return c ? std::atoi(c) : -2; }();
    if (carve >= -1) cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    if (e != cudaSuccess) {
      set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
      return (int)HS_ERR_CUDA;
    }
    cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(l.grid);
  cfg.blockDim = dim3(l.warps_per_cta * 32);
  cfg.dynamicSmemBytes = l.smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = p.overlap ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, p);
    e = cudaGetLastError();
    if (e != cudaSuccess) {
      set_error(std::string("traverse_slimq_kernel launch: ") + cudaGetErrorString(e));
      return (int)HS_ERR_CUDA;
    }
    return (int)HS_OK;
  });
}

}  // namespace hs
