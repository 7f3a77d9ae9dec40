// fp32 graph traversal for hnsw_slim on sm_100a: one warp per query.
//
// Replaces, for a whole query batch, HierarchicalNSWSlim<float>::searchKnn
// (slim.h:2030-2131): entry distance, greedy descent over the thinned upper levels
// (slim.h:2040-2078), then the ef-bounded best-first search of searchBaseLayerST<true>
// (slim.h:321-457) with L2Sqr / InnerProductDistance (space_l2.h:25-54, space_ip.h:146-204).
//
// Equivalence with the CPU algorithm (DESIGN.md "Sequential semantics"): the reference
// keeps a min-heap of candidates and an ef-bounded max-heap of results and tightens
// lowerBound after every admitted neighbour.  Here both are ONE pool of at most ef
// (distance,id) keys with an "expanded" bit; a hop scores all unvisited neighbours of the
// closest unexpanded entry at once and admits each one iff it beats the pool's current
// worst entry (which it replaces) — the reference's `top_size < ef || lowerBound > dist`
// followed by the trim to ef.  An entry pushed out of the pool can never be expanded by
// the reference either (its distance exceeds lowerBound from then on), so visited sets,
// distance counts and results coincide except where two distances tie bit-for-bit.
//
// The pool is UNSORTED and column-distributed (lane l owns entries l, l+32, ...), in registers
// for ef <= 256 (RegPool32: 32-bit distance words, one VIMNMX3 per lane + one REDUX per warp for
// the closest unexpanded / worst entry), in shared memory above (SmemPool); a hop needs no binary
// search and no shifting.  Per-warp shared memory: an open-addressing visited hash (replaces the
// N-entry tag array of visited_list_pool.h; it moves to global memory — traverse_fp32_g.cu — when
// it would cost too many resident warps), 32 staging ids and, for large dims, the query.  Vector
// rows are read with 128-bit loads, 8 lanes per row (4 rows per warp instruction), two packed
// fp32 FMA chains per lane (FADD2/FFMA2), xor-shuffle reduction 4,2,1.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstdint>
#include <type_traits>

#include "traverse_common.cuh"
#include "traverse_fp32.cuh"

// This file is compiled three times: as is (visited hash in shared memory), through traverse_fp32_g.cu with
// HS_GHASH = 1 (visited hash in global memory, L2-resident) and through traverse_fp32_c.cu with HS_CVTAB = 1
// (compact 16-bit visited table in shared memory, traverse_common.cuh cv_test_and_set: ef 129..256 at small dims).
#ifndef HS_GHASH
#define HS_GHASH 0
#endif
#ifndef HS_CVTAB
#define HS_CVTAB 0
#endif

namespace hs {
namespace {

// tuning knobs (see profiles/ for the measurements behind the defaults)
#ifndef HS_TRAVERSE_MIN_CTAS
#define HS_TRAVERSE_MIN_CTAS 6     // 128-thread CTAs per SM the register budget must allow
#endif
#ifndef HS_TRAVERSE_MIN_CTAS_BIG
#define HS_TRAVERSE_MIN_CTAS_BIG 6 // same for the pools of 5..8 register slots per lane (ef 129..256)
#endif
#ifndef HS_TRAVERSE_U
#define HS_TRAVERSE_U 2            // x4 rows whose loads are in flight per warp (kernels with the query in shared memory)
#endif
#ifndef HS_ROW_RING
#define HS_ROW_RING 0              // > 0: rows go through a shared-memory ring of this many rows (cp.async), see eval_rows_ring
#endif
#ifndef HS_POOL_COMPACT
#define HS_POOL_COMPACT 1          // pools of 5..8 slots per lane keep the expanded mark in the id word (RegPool32C)
#endif

template <int SLOTS> struct PoolSel {
  using type = std::conditional_t<(SLOTS >= 5 && HS_POOL_COMPACT), RegPool32C<SLOTS>, RegPool32<SLOTS>>;
};
template <> struct PoolSel<0> { using type = SmemPool; };

// Where a kernel keeps the query.  Shared memory for the generic path (CPL 0) and for the ef <= 128 register pools
// (2 / 4 slots): there the 4 x CPL query registers per lane pay for a second row group in eval_rows_sq (8 rows in
// flight instead of 4), which turns the 2 to 3 load rounds of a typical hop (about 9 fresh rows at ef = 100) into 1
// to 2.  Registers for CPL 3 / 4 with the larger pools (5..8 slots, ef 129..256) and the shared-memory pool: those
// keep 4 rows in flight.  plan_traverse sizes the shared-memory carve-out by the same rule.
constexpr bool query_in_smem(int cpl, int slots) { return cpl == 0 || slots == 2 || slots == 4; }

template <int CPL, int METRIC, int SLOTS>
__global__ void __launch_bounds__(128, SLOTS >= 5 ? HS_TRAVERSE_MIN_CTAS_BIG : HS_TRAVERSE_MIN_CTAS)
traverse_kernel(const __grid_constant__ TraverseParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  unsigned char *wbase = smem + (size_t)wid * p.smem_per_warp;
  // the visited table: shared memory, or (HS_GHASH) this warp's slice of a global scratch array.
  // A hop's probes then cost an L2 round trip instead of a shared-memory one, which is nothing
  // next to the row reads of a large-dim / large-ef hop, and the shared memory it frees is what
  // bounds the number of resident warps there.
  uint32_t *hash;
  if constexpr (HS_GHASH) {
    hash = p.ghash + ((size_t)(blockIdx.x * (blockDim.x >> 5) + wid) << p.hash_bits);
  } else {
    hash = reinterpret_cast<uint32_t *>(wbase + p.off_hash);
  }
  uint32_t *stage_ids = reinterpret_cast<uint32_t *>(wbase + p.off_stage);
  uint32_t *ghosts = stage_ids + 32;        // 16 words: exact-tie side list (traverse_common.cuh ghost_append)
  constexpr bool QSMEM = query_in_smem(CPL, SLOTS);
  float4 *qs = reinterpret_cast<float4 *>(wbase + p.off_query);

  if (p.overlap) {
    // consecutive batches may overlap (programmatic dependent launch): this grid needs nothing
    // from its predecessor, so the next launch may fill SM slots as soon as they free up
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }

  const uint32_t hbits = p.hash_bits, hsize = 1u << hbits, hmask = hsize - 1;     // HS_CVTAB: 2^12 16-bit cells
  // HS_CVTAB test knobs: traverse_flags bit 4 resets the table at 1/8 load instead of 3/4, bit 5 gives every id
  // ONE candidate bucket — both make the rare paths (reset, unrecorded id) common; results must not change
  const uint32_t hlimit = (HS_CVTAB && (p.flags & 16u)) ? hsize / 8 : hsize - hsize / 4;
  const bool cv_single = HS_CVTAB && (p.flags & 32u);
  // the visited set behind one interface (the three compilations of this file)
  bool vis_overflow = false;      // HS_CVTAB: an id found both its buckets full and was not recorded
  auto vis_clear = [&]() {
    if constexpr (HS_CVTAB) cv_clear(hash, lane);
    else hash_clear<HS_GHASH != 0>(hash, hsize, lane);
  };
  auto vis_test_and_set = [&](uint32_t id) -> bool {       // true: seen before
    if constexpr (HS_CVTAB) {
      const int r = cv_test_and_set(hash, id, cv_single);
      vis_overflow |= r == 2;
      return r == 1;
    } else {
      return visited_test_and_set<HS_GHASH != 0>(hash, hbits, hmask, id);
    }
  };
  // the table must be rebuilt from the pool before this hop: nearly full, or (HS_CVTAB) an id went unrecorded.
  // Results are unchanged either way: a node scored before was rejected or displaced and will be again.
  auto vis_needs_reset = [&](uint32_t hcount_, uint32_t incoming) -> bool {
    if constexpr (HS_CVTAB) {
      if (__any_sync(FULL, vis_overflow)) {
        vis_overflow = false;
        return true;
      }
    }
    return hcount_ + incoming > hlimit;
  };
  const uint32_t ef = p.ef;
  const int t8 = lane & 7;
  constexpr int QN = CPL > 0 ? CPL : 1;
  const bool qvec = ((reinterpret_cast<uintptr_t>(p.queries) & 15u) == 0) && (p.dim & 3u) == 0;

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

    // ---- query (zero-padded past dim): each chunk is read ONCE per warp (one 16-byte load per
    //      lane when the batch is 16-byte aligned): the batch may sit in pinned host memory
    //      (zero-copy hs_search_batch), where every request crosses PCIe.  Into shared memory
    //      (QSMEM), or into registers, where lane t of each team owns chunks t, t+8, ... and the
    //      chunks are handed to the four teams by shuffles ----
    const float *qptr = p.queries + (size_t)qi * p.dim;
    auto load_chunk = [&](uint32_t ch) -> float4 {
      const uint32_t c = 4u * ch;
      float4 v;
      if (qvec && c + 3 < p.dim) {
        v = __ldg(reinterpret_cast<const float4 *>(qptr) + ch);
      } else {
        v.x = c + 0 < p.dim ? __ldg(qptr + c + 0) : 0.f;
        v.y = c + 1 < p.dim ? __ldg(qptr + c + 1) : 0.f;
        v.z = c + 2 < p.dim ? __ldg(qptr + c + 2) : 0.f;
        v.w = c + 3 < p.dim ? __ldg(qptr + c + 3) : 0.f;
      }
      return v;
    };
    float4 q[QN];
    if constexpr (!QSMEM) {
      const float4 mine = load_chunk((uint32_t)lane);      // row_chunks = 8 * CPL <= 32
#pragma unroll
      for (int j = 0; j < QN; ++j) {
        q[j].x = __shfl_sync(FULL, mine.x, t8 + 8 * j);
        q[j].y = __shfl_sync(FULL, mine.y, t8 + 8 * j);
        q[j].z = __shfl_sync(FULL, mine.z, t8 + 8 * j);
        q[j].w = __shfl_sync(FULL, mine.w, t8 + 8 * j);
      }
    } else {
      for (uint32_t ch = lane; ch < p.row_chunks; ch += 32) qs[ch] = load_chunk(ch);
    }
    vis_clear();
    vis_overflow = false;
    __syncwarp();

    auto eval = [&](uint32_t my_id, int count) -> float {
      if constexpr (CPL > 0) {
        const float4 *qsm = qs;
#if HS_ROW_RING > 0
        float4 *ring = qs + (QSMEM ? p.row_chunks : 0u);      // the ring follows the query (plan_traverse)
        if constexpr (QSMEM) return eval_rows_ring<QN, METRIC, HS_ROW_RING>(p.vec, p.row_chunks, qsm, ring, my_id, count, lane);
        else return eval_rows_ring<QN, METRIC, HS_ROW_RING>(p.vec, p.row_chunks, q, ring, my_id, count, lane);
#else
        if constexpr (QSMEM) return eval_rows_sq<QN, METRIC, HS_TRAVERSE_U>(p.vec, p.row_chunks, qsm, my_id, count, lane);
        else return eval_rows_reg<QN, METRIC, 1>(p.vec, p.row_chunks, q, my_id, count, lane);
#endif
      } else {
        return eval_rows_smem<METRIC>(p.vec, p.row_chunks, qs, my_id, count, lane);
      }
    };

    uint32_t nd = 0, nh = 0;

    // ---- entry point and greedy descent, slim.h:2033-2078 ----
    uint32_t cur = p.enterpoint;
    float curdist = __shfl_sync(FULL, eval(cur, 1), 0);
    nd = 1;
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
          const float d = eval(id, count);
          nd += (uint32_t)count;
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

    // ---- seed, slim.h:2100-2106 ----
    uint32_t hcount = 1;
    typename PoolSel<SLOTS>::type pool;
    pool.init(reinterpret_cast<uint64_t *>(wbase), ef, lane);
    pool.seed(make_key(curdist, cur));
    if (lane == 0) vis_test_and_set(cur);
    __syncwarp();

    // ---- layered beam for threshold_level > 0 (searchBaseLayer, slim.h:222-316, called for
    //      levels min(threshold, maxlevel) .. 1 at slim.h:2108-2113).  Every layer restarts
    //      from ALL pool entries (the candidate set is re-made from top_candidates, :228-233:
    //      the expanded flags are cleared) while the visited set carries over.  The stop rule
    //      `min(cand) > lowerBound && |top| == ef` (:236-238) is "no unexpanded entry left in the
    //      pool", as on level 0: a candidate outside the pool implies a full pool. ----
    for (int layer = min(p.threshold_level, p.maxlevel); layer > 0; --layer) {
      const uint32_t *ladj = p.upper_adj[layer];
      if (lane == 0) ghosts[0] = 0;         // the candidate set is re-made from the results on every layer
      __syncwarp();
      for (;;) {
        uint32_t node = pool.pop_closest_unexpanded();
        if (node == kInvalid) node = pool.take_ghost(ghosts);
        if (node == kInvalid) break;
        const int slot = __ldg(p.upper_slot + node);
        // pool entries met on a lower layer may not exist on this one: the reference asserts
        // element_level >= layer (:247); such an entry has no row here
        if (slot < 0 || (uint32_t)slot >= p.level_count[layer]) continue;
        const uint32_t *row = ladj + (size_t)slot * p.upper_stride;
        if (vis_needs_reset(hcount, p.upper_stride)) {
          __syncwarp();
          vis_clear();
          __syncwarp();
          pool.for_each_id([&](uint32_t pid) { vis_test_and_set(pid); });
          hcount = pool.size;
          __syncwarp();
        }
        bool any = false;
        for (uint32_t seg = 0; seg < p.upper_stride; seg += 32) {
          const uint32_t id = (seg + lane < p.upper_stride) ? __ldg(row + seg + lane) : kInvalid;
          const unsigned vm = __ballot_sync(FULL, id != kInvalid);
          if (vm == 0) break;
          any = true;
          bool fresh = false;
          if (id != kInvalid) fresh = !vis_test_and_set(id);
          const unsigned fm = __ballot_sync(FULL, fresh);
          const int count = __popc(fm);
          if (count == 0) continue;
          hcount += (uint32_t)count;
          if (fresh) stage_ids[__popc(fm & ((1u << lane) - 1))] = id;
          __syncwarp();
          const uint32_t cid = lane < count ? stage_ids[lane] : 0u;
          __syncwarp();
          const float d = eval(cid, count);
          nd += (uint32_t)count;
          pool.admit(lane < count, make_key(d, cid), ghosts);
        }
        if (any) nh++;
      }
      pool.clear_flags();
    }

    // ---- base layer, slim.h:321-457 ----
    // evict_last on the adjacency prefetch: +1 % with 512-byte rows, -2 % with 3840-byte rows (200k x 960),
    // where the lines it pins compete with row lines that other queries would have hit: small dims only
    const bool opt_prefetch = p.flags & 1u, opt_spec = p.flags & 2u, opt_keep = (p.flags & 8u) && CPL > 0;
    uint32_t spec_node = kInvalid, spec_ids = kInvalid;
    if (lane == 0) ghosts[0] = 0;
    __syncwarp();
    for (;;) {
      if (p.flags & 4u) break;    // profiling aid (HS_TRAVERSE_FLAGS bit 2): time the descent alone
      // closest unexpanded entry (the reference pops its candidate min-heap, slim.h:335-354); once the pool
      // has none left, an entry that was trimmed while tying with the worst one (ghost_append)
      uint32_t node = pool.pop_closest_unexpanded();
      if (node == kInvalid) node = pool.take_ghost(ghosts);
      if (node == kInvalid) break;
      const uint32_t *row = p.adj0 + (size_t)node * p.deg0_stride;
      uint32_t id = node == spec_node ? spec_ids : __ldg(row + lane);
      // Speculation on the NEXT pop: unless this hop admits something closer, it is the entry that
      // is now the closest unexpanded one.  It usually entered the pool many hops ago, so the L2
      // prefetch of its adjacency row at admission time has long been evicted and the row would
      // cost a full DRAM round trip right after the pop; loading it now hides that behind this
      // hop.  Results do not depend on it: a wrong guess just loads the row on demand.
      if (opt_spec) {
        spec_node = pool.peek_closest_unexpanded();
        if (spec_node != kInvalid) {
          const uint32_t *srow = p.adj0 + (size_t)spec_node * p.deg0_stride;
          spec_ids = __ldg(srow + lane);
          if (p.deg0_stride > 32 && lane * 32u + 32u < p.deg0_stride) prefetch_l2(srow + 32 + lane * 32);
        }
      }

      if (vis_needs_reset(hcount, p.deg0_stride)) {
        // visited hash nearly full: keep only the pool entries (results are unchanged:
        // a node scored before was rejected or displaced and will be again)
        __syncwarp();
        vis_clear();
        __syncwarp();
        pool.for_each_id([&](uint32_t pid) { vis_test_and_set(pid); });
        hcount = pool.size;
        __syncwarp();
      }

      bool any = false;
      for (uint32_t seg = 0; seg < p.deg0_stride; seg += 32) {
        if (seg) id = __ldg(row + seg + lane);
        const unsigned vm = __ballot_sync(FULL, id != kInvalid);
        if (vm == 0) break;
        any = true;
        bool fresh = false;
        if (id != kInvalid) fresh = !vis_test_and_set(id);
        if (fresh && opt_prefetch) {
          // pull the whole row towards L2 now; the scoring loop below then mostly waits on L2
          const char *r = reinterpret_cast<const char *>(p.vec + (size_t)id * p.row_chunks);
          if constexpr (CPL > 0) {
#pragma unroll
            for (int j = 0; j < CPL; ++j) prefetch_l2(r + 128 * j);      // row = CPL x 128 B
          } else {
            for (uint32_t off = 0; off < p.row_chunks * 16u; off += 128) prefetch_l2(r + off);
          }
        }
        const unsigned fm = __ballot_sync(FULL, fresh);
        const int count = __popc(fm);
        if (count == 0) continue;
        hcount += (uint32_t)count;
        if (fresh) stage_ids[__popc(fm & ((1u << lane) - 1))] = id;
        __syncwarp();
        const uint32_t cid = lane < count ? stage_ids[lane] : 0u;
        __syncwarp();
        const float d = eval(cid, count);
        nd += (uint32_t)count;
        const unsigned entered = pool.admit(lane < count, make_key(d, cid), ghosts);
        if ((entered >> lane) & 1u) {
          if (opt_keep) prefetch_l2_keep(p.adj0 + (size_t)cid * p.deg0_stride);
          else prefetch_l2(p.adj0 + (size_t)cid * p.deg0_stride);
        }
      }
      if (any) nh++;
    }

    // ---- results: the k closest, ascending (the reference nth_element's the same set,
    //      slim.h:2126-2130): k rounds of warp-wide extract-min over the pool ----
    __syncwarp();
    {
      // lane i keeps result i; labels are looked up and rows written 32 results at a time
      // (one coalesced store per row for k <= 32: the output may be pinned host memory)
      uint64_t last = 0;   // every key is > 0 (f2ord(+0.0f) has the top bit set)
      uint64_t mine_out = NONE;
      for (uint32_t i = 0; i < p.k; ++i) {
        const uint64_t mine = last == NONE ? NONE : pool.col_next_above(last);
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
      atomicAdd(p.stats + 0, (unsigned long long)nd);
      atomicAdd(p.stats + 1, (unsigned long long)nh);
      if (p.per_query) {
        p.per_query[2 * (size_t)qi + 0] = nd;
        p.per_query[2 * (size_t)qi + 1] = nh;
      }
    }
    __syncwarp();
  }
  scatter_signal_done(p.scatter, lane);
}

template <int CPL, int METRIC, int SLOTS>
int launch_t(const TraverseParams &p, const TraverseLaunch &l, cudaStream_t stream) {
  auto kern = traverse_kernel<CPL, METRIC, SLOTS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem_bytes);
  if (e != cudaSuccess) {
    set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    return HS_ERR_CUDA;
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
    set_error(std::string("traverse_kernel launch: ") + cudaGetErrorString(e));
    return HS_ERR_CUDA;
  }
  return HS_OK;
}
template <int CPL, int METRIC, int SLOTS>
int occupancy_t(int threads, size_t smem) {
  auto kern = traverse_kernel<CPL, METRIC, SLOTS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, smem) != cudaSuccess) nb = 0;
  return nb;
}

template <typename F>
int dispatch(int cpl, int metric, int slots, F &&f) {
#define HS_CASE(C, M, S) \
  if (cpl == C && metric == M && slots == S) return f(std::integral_constant<int, C>{}, std::integral_constant<int, M>{}, std::integral_constant<int, S>{});
#if HS_CVTAB        // the compact table serves the register pools of 5..8 slots at small dims only (plan_traverse)
#define HS_CASES_S(C, M) HS_CASE(C, M, 5) HS_CASE(C, M, 6) HS_CASE(C, M, 7) HS_CASE(C, M, 8)
#define HS_CASES_M(C) HS_CASES_S(C, HS_METRIC_L2) HS_CASES_S(C, HS_METRIC_IP)
  HS_CASES_M(3) HS_CASES_M(4)
#else
#define HS_CASES_S(C, M) HS_CASE(C, M, 0) HS_CASE(C, M, 2) HS_CASE(C, M, 4) HS_CASE(C, M, 5) HS_CASE(C, M, 6) HS_CASE(C, M, 7) HS_CASE(C, M, 8)
#define HS_CASES_M(C) HS_CASES_S(C, HS_METRIC_L2) HS_CASES_S(C, HS_METRIC_IP)
  HS_CASES_M(0) HS_CASES_M(3) HS_CASES_M(4)
#endif
#undef HS_CASES_M
#undef HS_CASES_S
#undef HS_CASE
  set_error("no traversal kernel variant for this configuration");
  return HS_ERR_UNSUPPORTED;
}

}  // namespace

// one pair of entry points per copy of this file (shared-memory / global-memory / compact visited table)
#if HS_GHASH
#define HS_VARIANT(name) name##_g
#elif HS_CVTAB
#define HS_VARIANT(name) name##_c
#else
#define HS_VARIANT(name) name##_s
#endif
int HS_VARIANT(traverse_occupancy)(int cpl, int metric, int slots, int threads, size_t smem) {
  return dispatch(cpl, metric, slots, [&](auto C, auto M, auto S) {
    return occupancy_t<decltype(C)::value, decltype(M)::value, decltype(S)::value>(threads, smem);
  });
}
int HS_VARIANT(traverse_launch)(int cpl, int metric, int slots, const TraverseParams &p, const TraverseLaunch &l,
                                cudaStream_t stream) {
  return dispatch(cpl, metric, slots, [&](auto C, auto M, auto S) {
    return launch_t<decltype(C)::value, decltype(M)::value, decltype(S)::value>(p, l, stream);
  });
}

#if !HS_GHASH && !HS_CVTAB
int traverse_occupancy_g(int cpl, int metric, int slots, int threads, size_t smem);
int traverse_launch_g(int cpl, int metric, int slots, const TraverseParams &p, const TraverseLaunch &l,
                      cudaStream_t stream);
int traverse_occupancy_c(int cpl, int metric, int slots, int threads, size_t smem);
int traverse_launch_c(int cpl, int metric, int slots, const TraverseParams &p, const TraverseLaunch &l,
                      cudaStream_t stream);

namespace {
// kernel variants: CPL 3 (dim 96: DEEP/MSTuring), 4 (dim 128: SIFT) keep the query in
// registers, everything else runs the generic shared-memory-query path (CPL = 0);
// pool in registers for ef <= 64 / 128 / 160 / 192 / 224 / 256 (2 / 4 / 5 / 6 / 7 / 8 slots per lane), in shared memory above.
inline int cpl_variant(uint32_t row_chunks) {
  const uint32_t cpl = row_chunks / kTeam;
  return (cpl == 3 || cpl == 4) ? (int)cpl : 0;
}
// Register pools of 12 / 16 slots for ef 257..512 in the generic kernel (its query sits in shared memory) were
// measured and lose to the shared-memory pool there (GIST-shaped 200k x 960: ef=400 193 k vs 236 k QPS even with a
// 96-register budget, profiles/r02_probe_bigpool.txt): a large-dim hop is row traffic, and the pool's registers
// are taken from the loads in flight.
inline int slots_variant(uint32_t ef, int cplv, uint32_t flags = 0) {
  (void)cplv;
  if (flags & 64u) return 0;         // traverse_flags bit 6: the shared-memory pool whatever ef is (A/B runs, tests)
  return ef <= 64 ? 2 : (ef <= 128 ? 4 : (ef <= 160 ? 5 : (ef <= 192 ? 6 : (ef <= 224 ? 7 : (ef <= 256 ? 8 : 0)))));
}
inline uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }
constexpr uint32_t kSmemPerSm = 227u * 1024u;
}  // namespace

int plan_traverse(TraverseParams &p, int metric, int hash_bits_override, int ghash_mode, int sm_count, int nq,
                  TraverseLaunch *out) {
  // visited-hash capacity: ~16 slots per ef entry (measured ~12 evaluations per ef entry on
  // 1M x 128, SURVEY.md §8d); the kernel resets the table when it passes 75 % so a smaller table
  // only costs repeated evaluations, never correctness.  With threshold_level > 0 every layer of
  // the layered beam adds its own evaluations.
  const uint32_t layers = 1u + (uint32_t)std::max(0, std::min(p.threshold_level, p.maxlevel));
  const uint32_t min_slots = p.ef + 2 * std::max(p.deg0_stride, p.upper_stride) + 32;   // the reset must make room
  auto pick_bits = [&](uint32_t cap) {
    uint32_t bits = 10;
    while ((1u << bits) < 16u * p.ef * layers && bits < cap) ++bits;
    if (hash_bits_override > 0) bits = (uint32_t)hash_bits_override;
    if (bits < 8) bits = 8;
    if (bits > 16) bits = 16;
    while ((1u << bits) - (1u << bits) / 4 < min_slots && bits < 16) ++bits;
    return bits;
  };
  const int cplv = cpl_variant(p.row_chunks), slv = slots_variant(p.ef, cplv, p.flags);
  const int met = metric == HS_METRIC_IP ? HS_METRIC_IP : HS_METRIC_L2;
  const uint32_t list_bytes = slv ? 0u : align_up(p.ef * 8u, 16);
  const uint32_t stage_bytes = 32 * 4 + 16 * 4;       // staging ids + the exact-tie side list
  // the query where the kernel reads it from shared memory (query_in_smem), then, small dims with HS_ROW_RING, the
  // row ring (same carve-out, off_query)
  const uint32_t query_bytes = (query_in_smem(cplv, slv) ? p.row_chunks * 16u : 0u)
                               + (cplv == 0 ? 0u : (uint32_t)HS_ROW_RING * p.row_chunks * 16u);

  // Shared-memory tables first.  They bound the resident warps: 24 per SM (what the register file
  // allows) needs <= 9.4 KB per warp.  When the table of this ef (plus the query of a large dim)
  // pushes a warp past ~14 KB (fewer than 16 warps per SM), the tables move to global memory:
  // they stay L2-resident and a probe's extra latency is small next to a hop's row reads.
  const uint32_t bits_s = pick_bits(14);
  const uint32_t per_warp_s = align_up(list_bytes + (4u << bits_s) + stage_bytes + query_bytes, 16);
  bool ghash = ghash_mode == 1 || (ghash_mode < 0 && kSmemPerSm / per_warp_s < 16);
  if (per_warp_s > kSmemPerSm) ghash = true;
  // Compact table (traverse_fp32_c.cu): 4096 16-bit cells in 8 KB, exact for ids < 2^24.  It serves the case the
  // 32-bit table is too big for — the register pools of 5..8 slots (ef 129..256) at small dims, where 16 KB per
  // warp would halve the resident warps: with 8 KB they stay at 24 per SM and the probes stay in shared memory.
  // ~12 evaluations per ef entry (SURVEY.md §8d) fill it to ~60 % at ef=256; past 75 % it is reset like the others.
  // ghash_mode 2 asks for it explicitly, 3 is the automatic choice without it.
  const bool legacy_auto = ghash_mode == 3;
  if (legacy_auto) ghash = kSmemPerSm / per_warp_s < 16 || per_warp_s > kSmemPerSm;
  const bool cv_fits = cplv != 0 && slv >= 5 && p.n <= (1u << 24) && layers == 1 && hash_bits_override <= 0;
  const bool cvtab = cv_fits && (ghash_mode == 2 || ghash_mode < 0);
  if (cvtab) ghash = false;
  const uint32_t bits = cvtab ? 12u : (ghash ? pick_bits(16) : bits_s);
  p.hash_bits = bits;
  const uint32_t hash_bytes = cvtab ? (2u << bits) : (ghash ? 0u : (4u << bits));
  p.off_hash = list_bytes;
  p.off_stage = p.off_hash + hash_bytes;
  p.off_query = p.off_stage + stage_bytes;
  p.smem_per_warp = align_up(p.off_query + query_bytes, 16);
  if (p.smem_per_warp > kSmemPerSm) {
    set_error("ef / dim too large for the per-warp shared-memory working set");
    return HS_ERR_UNSUPPORTED;
  }
  // CTA shape.  Warps never cooperate, so a CTA is only a packaging unit — and the smaller the
  // better: an SM slot is handed to the next (overlapping) launch when a whole CTA exits, and a CTA
  // of 4 warps idles 3 of them while its last query drains.  One-warp CTAs are used whenever the
  // 32-CTAs-per-SM limit and the 1 KB of shared memory the system reserves per CTA do not cost
  // resident warps (measured +2.5 % at ef=100, +5 % at ef=50 on 1M x 128); else 2 or 4 warps.
  const int met_ = met;
  auto occupancy = [&](int w) {
    const size_t smem = (size_t)w * p.smem_per_warp;
    if (smem > kSmemPerSm) return 0;
    if (cvtab) return traverse_occupancy_c(cplv, met_, slv, w * 32, smem);
    return ghash ? traverse_occupancy_g(cplv, met_, slv, w * 32, smem) : traverse_occupancy_s(cplv, met_, slv, w * 32, smem);
  };
  int wpc = 1, per_sm = occupancy(1);
  for (int w = 2; w <= 4; w *= 2) {
    const int o = occupancy(w);
    // large dims (query in shared memory): four-warp CTAs measured better or equal (GIST-shaped
    // 200k x 960: ef=50 6.2 vs 7.3 ms per 10k queries, ef=100 equal), so they win ties there
    if (o * w > per_sm * wpc || (cplv == 0 && o * w >= per_sm * wpc)) {
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
    set_error("traverse_kernel does not fit on an SM (cudaOccupancyMaxActiveBlocksPerMultiprocessor)");
    return HS_ERR_CUDA;
  }
  out->resident = sm_count * per_sm;
  out->ghash = ghash;
  out->cvtab = cvtab;
  resize_traverse_launch(p, nq, out);
  return HS_OK;
}

// The only part of a launch plan that depends on the batch size: the grid (and what follows from it).  Everything
// else — kernel variant, shared-memory layout, CTA shape, occupancy — is a function of (index, ef, knobs), which is
// what makes a cached plan reusable for batches of any size (a server's batches differ in size every time, and the
// occupancy queries of a full plan cost tens of microseconds).
void resize_traverse_launch(const TraverseParams &p, int nq, TraverseLaunch *l) {
  const int wpc = l->warps_per_cta;
  const int need = (nq + wpc - 1) / wpc;
  l->grid = need < l->resident ? (need > 0 ? need : 1) : l->resident;
  l->ghash_bytes = l->ghash ? ((size_t)l->grid * wpc * 4) << p.hash_bits : 0;
  // two overlapping launches alternate between two scratch halves (hs_api.cu); a third launch can
  // only become resident next to them when a grid does not fill the GPU — no overlap then
  l->may_overlap = !l->ghash || l->grid == l->resident;
}

int launch_traverse(const TraverseParams &p, int metric, const TraverseLaunch &l, cudaStream_t stream) {
  const int cplv = cpl_variant(p.row_chunks), slv = slots_variant(p.ef, cplv, p.flags);
  const int met = metric == HS_METRIC_IP ? HS_METRIC_IP : HS_METRIC_L2;
  if (l.cvtab) return traverse_launch_c(cplv, met, slv, p, l, stream);
  return l.ghash ? traverse_launch_g(cplv, met, slv, p, l, stream) : traverse_launch_s(cplv, met, slv, p, l, stream);
}
#endif   // !HS_GHASH && !HS_CVTAB

}  // namespace hs
