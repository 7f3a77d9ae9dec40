// Device-side building blocks shared by the traversal kernels (traverse_fp32.cu,
// traverse_slimq.cu): order-preserving (distance,id) keys, warp-wide arg-min/max, the
// register / shared-memory candidate pools, the fp32 row scorer and the visited hash.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "hs_internal.h"

namespace hs {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t FLAG = 0x80000000u;             // "expanded" bit inside the id half of a key
constexpr uint64_t KEYMASK = ~(uint64_t)FLAG;
constexpr uint32_t EMPTY = 0xFFFFFFFFu;

// monotone float -> uint32 map (IP distances 1 - <a,b> can be negative)
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
__device__ __forceinline__ uint64_t make_key(float d, uint32_t id) {
  return ((uint64_t)f2ord(d) << 32) | id;
}

__device__ __forceinline__ uint64_t warp_min_u64(uint64_t v) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    uint64_t o = __shfl_xor_sync(FULL, v, off);
    v = o < v ? o : v;
  }
  return v;
}

// Per-lane partial sums live as TWO fp32 accumulators packed in one 64-bit register pair and are
// updated with the packed FADD2 / FFMA2 instructions of sm_100 (sub.rn.f32x2, fma.rn.f32x2: two
// IEEE fp32 operations per issue slot).  `lo` accumulates elements x and z of the lane's float4
// chunks, `hi` elements y and w, both in chunk order; the lane's sum is lo + hi.  The oracle's
// HSO_ORDER_GPU association (oracle/hs_oracle.c dist_gpu) restates exactly this.
typedef unsigned long long acc2_t;
__device__ __forceinline__ acc2_t pack2(float lo, float hi) {
  acc2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float sum2(acc2_t a) {
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
  return __fadd_rn(lo, hi);
}
__device__ __forceinline__ acc2_t sub2(acc2_t a, acc2_t b) {
  acc2_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ acc2_t fma2(acc2_t a, acc2_t b, acc2_t c) {
  acc2_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
template <int METRIC>
__device__ __forceinline__ acc2_t acc4(acc2_t acc, const float4 q, const float4 x) {
  const acc2_t q01 = pack2(q.x, q.y), q23 = pack2(q.z, q.w);
  const acc2_t x01 = pack2(x.x, x.y), x23 = pack2(x.z, x.w);
  if (METRIC == HS_METRIC_L2) {
    const acc2_t d01 = sub2(q01, x01), d23 = sub2(q23, x23);
    acc = fma2(d01, d01, acc);
    acc = fma2(d23, d23, acc);
  } else {
    acc = fma2(q01, x01, acc);
    acc = fma2(q23, x23, acc);
  }
  return acc;
}
template <int METRIC>
__device__ __forceinline__ float finish(float acc) {
  return METRIC == HS_METRIC_IP ? __fsub_rn(1.0f, acc) : acc;
}
__device__ __forceinline__ float team_reduce(float v) {
  v = __fadd_rn(v, __shfl_xor_sync(FULL, v, 4));
  v = __fadd_rn(v, __shfl_xor_sync(FULL, v, 2));
  v = __fadd_rn(v, __shfl_xor_sync(FULL, v, 1));
  return v;
}

// Distances from the query to `count` (<= 32) rows; lane j holds id j, gets d_j back.
// Register-resident query, CPL float4 chunks per lane, U x 4 rows in flight per warp.
template <int CPL, int METRIC, int U>
__device__ __forceinline__ float eval_rows_reg(const float4 *__restrict__ vec, uint32_t row_chunks,
                                               const float4 (&q)[CPL], uint32_t my_id, int count,
                                               int lane) {
  const int team = lane >> 3, t = lane & 7;
  float my_d = 0.f;
  for (int it0 = 0; it0 * 4 < count; it0 += U) {
    float4 x[U][CPL];
    bool act[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int src = (it0 + u) * 4 + team;
      const uint32_t id = __shfl_sync(FULL, my_id, src & 31);
      act[u] = src < count;
      if (act[u]) {
        const float4 *row = vec + (size_t)id * row_chunks + t;
#pragma unroll
        for (int j = 0; j < CPL; ++j) x[u][j] = __ldg(row + 8 * j);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      acc2_t acc2 = 0ull;
      if (act[u]) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) acc2 = acc4<METRIC>(acc2, q[j], x[u][j]);
      }
      const float acc = team_reduce(sum2(acc2));
      const float v = __shfl_sync(FULL, acc, (lane & 3) * 8);
      if ((lane >> 2) == it0 + u) my_d = finish<METRIC>(v);
    }
  }
  return my_d;
}

// Query chunk j of lane t of a team for eval_rows_ring: Q is either `float4[CPL]` (registers, as in eval_rows_reg) or
// `float4 *` (the query's chunks in shared memory, as in eval_rows_sq).
template <typename Q>
__device__ __forceinline__ float4 query_chunk(const Q &q, int j, int t) {
  if constexpr (std::is_pointer_v<Q>) return q[8 * j + t];
  else return q[j];
}

// One round of eval_rows_sq: G groups of 4 rows from row 4 * it0 on, each group with at least one row.  The loads of
// all G groups are issued before the first FMA.  A team without a row of its own re-reads the last row (an address
// its group loads anyway) instead of skipping its loads: loads that happen on some paths only leave the rows
// conditionally defined, and the kernel then spills hundreds of bytes.  Its sum is replaced by 0, as in eval_rows_reg.
// The query chunk is read with a volatile LDS.128 next to its FMAs: hoisted above the row loads, the chunks take the
// registers of the second group and ptxas delays that group's loads behind the first group's FMAs.
template <int CPL, int METRIC, int G>
__device__ __forceinline__ void eval_round_sq(const float4 *__restrict__ vec, uint32_t row_chunks, const float4 *qs,
                                              uint32_t my_id, int count, int it0, int lane, float &my_d) {
  const int team = lane >> 3, t = lane & 7;
  float4 x[G][CPL];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const uint32_t id = __shfl_sync(FULL, my_id, min((it0 + g) * 4 + team, count - 1));
    const float4 *row = vec + (size_t)id * row_chunks + t;
#pragma unroll
    for (int j = 0; j < CPL; ++j) x[g][j] = __ldg(row + 8 * j);
  }
  acc2_t acc2[G];
#pragma unroll
  for (int g = 0; g < G; ++g) acc2[g] = 0ull;
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    float4 qj;
    const unsigned a = (unsigned)__cvta_generic_to_shared(qs + 8 * j + t);
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(qj.x), "=f"(qj.y), "=f"(qj.z), "=f"(qj.w) : "r"(a));
#pragma unroll
    for (int g = 0; g < G; ++g) acc2[g] = acc4<METRIC>(acc2[g], qj, x[g][j]);
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const float acc = team_reduce(sum2((it0 + g) * 4 + team < count ? acc2[g] : 0ull));
    const float v = __shfl_sync(FULL, acc, (lane & 3) * 8);
    if ((lane >> 2) == it0 + g) my_d = finish<METRIC>(v);
  }
}

// Same as eval_rows_reg with the query in shared memory (`qs`: the query's row_chunks chunks; the four teams read the
// same 16 bytes, a broadcast, and a team reads 128 contiguous bytes, so a chunk is one conflict-free LDS.128).  That
// frees the 4 x CPL query registers for a second row group: U x 4 rows in flight per warp, so a hop of up to 8 fresh
// rows (U = 2) waits for one round of row loads instead of two.  Rounds of U groups while more than U - 1 groups of
// rows are left, then single groups.  Every group keeps its own FFMA2 chain in chunk order: the sums do not depend on
// U or on where the query is read from (bit-identical to eval_rows_reg).
template <int CPL, int METRIC, int U>
__device__ __forceinline__ float eval_rows_sq(const float4 *__restrict__ vec, uint32_t row_chunks, const float4 *qs,
                                              uint32_t my_id, int count, int lane) {
  float my_d = 0.f;
  int it0 = 0;
  if constexpr (U > 1) {
#pragma unroll 1
    for (; count - it0 * 4 > 4 * (U - 1); it0 += U) eval_round_sq<CPL, METRIC, U>(vec, row_chunks, qs, my_id, count, it0, lane, my_d);
  }
#pragma unroll 1
  for (; it0 * 4 < count; ++it0) eval_round_sq<CPL, METRIC, 1>(vec, row_chunks, qs, my_id, count, it0, lane, my_d);
  return my_d;
}

// Same through a per-warp shared-memory ring of R rows (R a multiple of 4): ALL rows of a chunk are put in flight at
// once with 16-byte cp.async copies (one per lane and row: a row of CPL x 8 chunks is at most 32 of them), then
// scored out of shared memory — the rows-in-flight count no longer depends on the register budget, and a hop waits
// for one memory round trip instead of one per 4 rows.  Same association as eval_rows_reg (bit-identical sums).
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
template <int CPL, int METRIC, int R, typename Q>
__device__ __forceinline__ float eval_rows_ring(const float4 *__restrict__ vec, uint32_t row_chunks, const Q &q,
                                                float4 *ring, uint32_t my_id, int count, int lane) {
  static_assert(R % 4 == 0 && R > 0, "ring rows must be a multiple of 4");
  const int team = lane >> 3, t = lane & 7;
  float my_d = 0.f;
  for (int base = 0; base < count; base += R) {
    const int n = min(R, count - base);
    for (int r = 0; r < n; ++r) {
      const uint32_t id = __shfl_sync(FULL, my_id, base + r);
      if (lane < CPL * 8) cp_async16(ring + r * (CPL * 8) + lane, vec + (size_t)id * row_chunks + lane);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    for (int it = 0; it * 4 < n; ++it) {
      const int src = it * 4 + team;
      acc2_t acc2 = 0ull;
      if (src < n) {
        const float4 *row = ring + src * (CPL * 8) + t;
#pragma unroll
        for (int j = 0; j < CPL; ++j) acc2 = acc4<METRIC>(acc2, query_chunk(q, j, t), row[8 * j]);
      }
      const float acc = team_reduce(sum2(acc2));
      const float v = __shfl_sync(FULL, acc, (lane & 3) * 8);
      if ((lane >> 2) == base / 4 + it) my_d = finish<METRIC>(v);
    }
    __syncwarp();                                  // the ring is rewritten by the next chunk / the next call
  }
  return my_d;
}

// Same with the query in shared memory and a run-time chunk count (large / odd dims).
template <int METRIC>
__device__ __forceinline__ float eval_rows_smem(const float4 *__restrict__ vec, uint32_t row_chunks,
                                                const float4 *qs, uint32_t my_id, int count, int lane) {
  const int team = lane >> 3, t = lane & 7;
  const int cpl = (int)(row_chunks >> 3);
  float my_d = 0.f;
  for (int it = 0; it * 4 < count; ++it) {
    const int src = it * 4 + team;
    const uint32_t id = __shfl_sync(FULL, my_id, src & 31);
    acc2_t acc2 = 0ull;
    if (src < count) {
      const float4 *row = vec + (size_t)id * row_chunks + t;
      const float4 *qq = qs + t;
      int j = 0;
      for (; j + 8 <= cpl; j += 8) {
        float4 x[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) x[jj] = __ldg(row + 8 * (j + jj));
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) acc2 = acc4<METRIC>(acc2, qq[8 * (j + jj)], x[jj]);
      }
      for (; j < cpl; ++j) acc2 = acc4<METRIC>(acc2, qq[8 * j], __ldg(row + 8 * j));
    }
    const float acc = team_reduce(sum2(acc2));
    const float v = __shfl_sync(FULL, acc, (lane & 3) * 8);
    if ((lane >> 2) == it) my_d = finish<METRIC>(v);
  }
  return my_d;
}

// visited set: open addressing, linear probing, 32-bit keys (replaces the per-thread
// uint16 tag array of visited_list_pool.h:10-31).  Returns true if id was already present.
template <bool GLOBAL_TABLE = false>
__device__ __forceinline__ bool visited_test_and_set(uint32_t *hash, uint32_t hbits, uint32_t hmask,
                                                     uint32_t id) {
  uint32_t h = (id * 0x9E3779B1u) >> (32 - hbits);
  if (GLOBAL_TABLE) {
    // table in global memory: look before the atomic (most probes of a long search end on an
    // occupied slot, and a load is cheaper than a compare-and-swap at L2)
    volatile uint32_t *vh = hash;
    for (;;) {
      const uint32_t v = vh[h];
      if (v == id) return true;
      if (v == EMPTY) {
        const uint32_t old = atomicCAS(hash + h, EMPTY, id);
        if (old == EMPTY) return false;
        if (old == id) return true;
      }
      h = (h + 1) & hmask;
    }
  }
  // table in shared memory: compare-and-swap FIRST — a fresh id whose home slot is empty (the
  // common case, the table is at most 75 % full) costs one shared-memory round trip instead of a
  // load, a branch and a CAS
  for (;;) {
    const uint32_t old = atomicCAS(hash + h, EMPTY, id);
    if (old == EMPTY) return false;
    if (old == id) return true;
    h = (h + 1) & hmask;
  }
}

// Callers follow with __syncwarp().  A table in global memory is probed with atomics that execute
// at L2: the clearing stores must have landed there first (GLOBAL_TABLE: device-scope fence).
template <bool GLOBAL_TABLE = false>
__device__ __forceinline__ void hash_clear(uint32_t *hash, uint32_t hsize, int lane) {
  const uint4 e = make_uint4(EMPTY, EMPTY, EMPTY, EMPTY);
  for (uint32_t i = lane * 4; i < hsize; i += 128) *reinterpret_cast<uint4 *>(hash + i) = e;
  if (GLOBAL_TABLE) __threadfence();
}

// ---- compact visited table: 4096 cells of 16 bits in 8 KB of shared memory (ids < 2^24) ----
// For ef 129..256 the 32-bit table above needs 16 KB per warp, which leaves 14 warps per SM (or sends the table
// to global memory); halving the cell halves that.  A 16-bit cell cannot hold an id, so the table stores
// REMAINDERS: 512 buckets of 8 cells (one 16-byte bucket = one LDS.128); an id has two candidate buckets, each
// from a bijection of the 24-bit id space (multiplication by an odd constant mod 2^24) whose top 9 bits pick the
// bucket and whose low 15 bits are the cell value — bit 15 of the cell says which of the two bijections it came
// from, so (bucket, cell) identifies the id exactly: no false positives, which bit-exact parity with the
// reference's visited array (visited_list_pool.h:10-31) needs.  0xFFFF marks an empty cell (the one id whose
// second-choice cell would be 0xFFFF simply has no second choice).  A bucket fills front to back, an insertion goes
// to the emptier of the two buckets (two-choice balancing keeps 8-cell buckets from overflowing far beyond the
// 75 % load at which the caller resets the table anyway), by compare-and-swap on the 32-bit word that holds the
// cell; a lane that loses the race looks again.  Returns 0: was absent, now recorded; 1: present; 2: absent and
// NOT recorded (both buckets full) — the caller then resets the table before the next hop, exactly as it does
// when the table passes its load limit (results unchanged, see the reset comment in the kernel).
constexpr uint32_t kCvWords = 2048;            // 32-bit words: 512 buckets x 4
__device__ __forceinline__ void cv_clear(uint32_t *tab, int lane) {
  const uint4 e = make_uint4(EMPTY, EMPTY, EMPTY, EMPTY);
  for (uint32_t i = lane * 4; i < kCvWords; i += 128) *reinterpret_cast<uint4 *>(tab + i) = e;
}
// nonzero iff some 16-bit half of x is zero
__device__ __forceinline__ uint32_t cv_haszero(uint32_t x) { return (x - 0x00010001u) & ~x & 0x80008000u; }
// one bucket: a 16-byte shared-memory load that is re-issued on every call (the loop below re-reads after a lost CAS)
__device__ __forceinline__ uint4 cv_bucket(const uint32_t *p) {
  uint4 v;
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
// `single` (a test knob, traverse_flags bit 5) withholds the second choice so that buckets do overflow.
__device__ __forceinline__ int cv_test_and_set(uint32_t *tab, uint32_t id, bool single = false) {
  const uint32_t m1 = (id * 0x9E3779B1u) & 0xFFFFFFu, m2 = (id * 0x85EBCA6Bu) & 0xFFFFFFu;
  const uint32_t b1 = m1 >> 15, b2 = m2 >> 15;
  const uint32_t c1 = m1 & 0x7FFFu, c2 = (m2 & 0x7FFFu) | 0x8000u;
  const bool ok2 = c2 != 0xFFFFu && b2 != b1 && !single;
  const uint32_t p1 = c1 * 0x00010001u, p2 = c2 * 0x00010001u;
  for (;;) {
    const uint4 w1 = cv_bucket(tab + 4 * b1), w2 = cv_bucket(tab + 4 * b2);
    uint32_t hit = cv_haszero(w1.x ^ p1) | cv_haszero(w1.y ^ p1) | cv_haszero(w1.z ^ p1) | cv_haszero(w1.w ^ p1);
    if (ok2) hit |= cv_haszero(w2.x ^ p2) | cv_haszero(w2.y ^ p2) | cv_haszero(w2.z ^ p2) | cv_haszero(w2.w ^ p2);
    if (hit) return 1;
    // buckets fill front to back: a word is full iff its high half is used (word < 0xFFFF0000)
    const uint32_t T = 0xFFFF0000u;
    const int f1 = (w1.x < T) + (w1.y < T) + (w1.z < T) + (w1.w < T);
    const int f2 = ok2 ? (w2.x < T) + (w2.y < T) + (w2.z < T) + (w2.w < T) : 4;
    const uint32_t t1 = f1 == 0 ? w1.x : (f1 == 1 ? w1.y : (f1 == 2 ? w1.z : w1.w));     // first word with room (if f < 4)
    const uint32_t t2 = f2 == 0 ? w2.x : (f2 == 1 ? w2.y : (f2 == 2 ? w2.z : w2.w));
    const int occ1 = 2 * f1 + (f1 < 4 && (t1 & 0xFFFFu) != 0xFFFFu), occ2 = 2 * f2 + (f2 < 4 && (t2 & 0xFFFFu) != 0xFFFFu);
    if (occ1 >= 8 && occ2 >= 8) return 2;
    const bool second = occ2 < occ1;
    const uint32_t old = second ? t2 : t1, c = second ? c2 : c1;
    uint32_t *at = tab + 4 * (second ? b2 : b1) + (second ? f2 : f1);
    const uint32_t neu = (old & 0xFFFFu) == 0xFFFFu ? ((old & 0xFFFF0000u) | c) : ((old & 0x0000FFFFu) | (c << 16));
    if (atomicCAS(at, old, neu) == old) return 0;
  }
}

__device__ __forceinline__ void prefetch_l2(const void *p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
// same, asking L2 to evict the line last: adjacency rows of pool entries are needed again when the
// entry is popped, typically long after the streaming row reads would have pushed them out
__device__ __forceinline__ void prefetch_l2_keep(const void *p) {
  asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(p));
}
constexpr uint64_t NONE = ~0ull;

// Dynamic work distribution: the next query index of THIS launch.  The counter is one slot of a
// ring that the host walks (hs_api.cu), tagged in its high half with the launch sequence number,
// so it never needs a reset between launches — which lets consecutive launches overlap
// (hs_set_overlap) without a memset node between them.  The first warp of a launch to arrive
// finds a foreign tag and claims the slot.
__device__ __forceinline__ uint32_t next_ticket(unsigned long long *ctr, uint32_t tag) {
  unsigned long long old = atomicAdd(ctr, 1ull);
  while ((uint32_t)(old >> 32) != tag) {
    const unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(ctr);
    if ((uint32_t)(cur >> 32) == tag) {
      old = atomicAdd(ctr, 1ull);
    } else if (atomicCAS(ctr, cur, ((unsigned long long)tag << 32) | 1ull) == cur) {
      old = (unsigned long long)tag << 32;       // ticket 0 is mine
    } else {
      old = cur;                                  // lost the race: look again
    }
  }
  return (uint32_t)old;
}

// ---- shard-group completion protocol (ScatterDst, hs_internal.h) ----
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Called by a whole warp before its first row store of a launch: the destination slot of every rank
// must have been merged (ack words are written by the ranks' merge streams).  Sequence numbers are
// compared as signed differences so that they may wrap.  The host never launches a batch before THIS
// rank's merge of batch seq - depth has completed (hs_shardgroup_submit), so a warp only ever waits
// here for OTHER ranks' merge streams — it cannot hold the SM slot its own merge kernel needs.  A wait
// that exceeds sc.ack_timeout_ns (a dead or wedged peer) is recorded in *sc.status and abandoned: the
// batch's rows are then unreliable, which hs_shardgroup_wait reports, but the GPU does not hang.
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void scatter_wait_acks(const ScatterDst &sc, int lane) {
  if (sc.ack_need == 0) return;
  if ((uint32_t)lane < sc.n_acks) {
    if ((int32_t)(ld_acquire_sys(sc.acks + lane) - sc.ack_need) < 0) {
      const unsigned long long t0 = global_ns();
      while ((int32_t)(ld_acquire_sys(sc.acks + lane) - sc.ack_need) < 0) {
        __nanosleep(512);
        if (global_ns() - t0 > sc.ack_timeout_ns) {
          if (sc.status) atomicMax(sc.status, 1u);
          break;
        }
      }
    }
  }
  __syncwarp();
}
// Called by every warp of a launch exactly once, after its last row store.
__device__ __forceinline__ void scatter_signal_done(const ScatterDst &sc, int lane) {
  if (sc.done_ctr == nullptr) return;
  __syncwarp();
  if (lane == 0) {
    __threadfence_system();                        // this warp's rows (local and peer memory) before the count
    const unsigned int old = atomicAdd(sc.done_ctr, 1u);
    if (old + 1u == sc.done_target) {
      atomicExch(sc.done_ctr, 0u);                 // ready for the batch that reuses this counter
      __threadfence_system();                      // every counted warp's rows before the flags
      for (uint32_t t = 0; t < sc.n_flags; ++t) st_release_sys(sc.flags[t], sc.seq);
    }
  }
}

// lane holding the warp-wide smallest `key` ((dist,id) order; NONE = no entry); -1 if none
__device__ __forceinline__ int warp_argmin_key(uint64_t key) {
  const uint32_t hi = (uint32_t)(key >> 32);
  const uint32_t ghi = __reduce_min_sync(FULL, hi);
  if (ghi == 0xffffffffu) return -1;
  unsigned b = __ballot_sync(FULL, hi == ghi);
  if (b & (b - 1)) {   // equal distances in several lanes: smaller id first
    const uint32_t lo = hi == ghi ? (uint32_t)key : 0xffffffffu;
    const uint32_t glo = __reduce_min_sync(FULL, lo);
    b = __ballot_sync(FULL, hi == ghi && lo == glo);
  }
  return __ffs(b) - 1;
}
// lane holding the warp-wide largest `key` (0 = no entry)
__device__ __forceinline__ int warp_argmax_key(uint64_t key) {
  const uint32_t hi = (uint32_t)(key >> 32);
  const uint32_t ghi = __reduce_max_sync(FULL, hi);
  unsigned b = __ballot_sync(FULL, hi == ghi);
  if (b & (b - 1)) {
    const uint32_t lo = hi == ghi ? (uint32_t)key : 0u;
    const uint32_t glo = __reduce_max_sync(FULL, lo);
    b = __ballot_sync(FULL, hi == ghi && lo == glo);
  }
  return __ffs(b) - 1;
}

// ---- "ghost" candidates: exact distance ties at the ef boundary ----
// The reference keeps candidates and results in two heaps.  An entry trimmed from the result heap stays in
// the candidate heap, and the reference still EXPANDS it when it comes up unless its distance is strictly
// beyond lowerBound (slim.h:237, :339-340: `>`).  A trimmed entry is the worst one, so that only happens
// when another entry with the bit-identical distance stays behind as the new worst — an exact fp32 tie.
// The pool drops a displaced entry, so the tie case is kept on the side: when the entry being displaced is
// unexpanded and ties with another column's worst, it is appended to a small per-warp list in shared
// memory (g[0] = count, then (distance word, id) pairs); when the pool runs out of unexpanded entries the
// list is consulted: a ghost whose distance still equals the pool's worst is expanded like the reference
// would, everything else in it is dead (lowerBound only shrinks).  Cost on the hot path: one AND and one
// uniform branch per displacement.  Not caught: a tie whose two members sit in the SAME pool column and no
// other (1 in 32 of an event that needs two bit-equal fp32 distances at the boundary).
constexpr uint32_t kGhostCap = 7;            // pairs; the list occupies 16 words per warp
__device__ __forceinline__ void ghost_append(uint32_t *g, uint32_t dword, uint32_t id) {
  const uint32_t c = g[0];
  if (c < kGhostCap) {
    g[2 + 2 * c] = dword;
    g[3 + 2 * c] = id;
    g[0] = c + 1;
  }
}
// the next ghost that the reference would still expand (distance word == worst of a FULL pool), or kInvalid
__device__ __forceinline__ uint32_t ghost_take(uint32_t *g, uint32_t worst, bool full, int lane) {
  const uint32_t cnt = g[0];
  if (cnt == 0) return kInvalid;
  uint32_t gd = 0, gi = kInvalid;
  if ((uint32_t)lane < cnt) {
    gd = g[2 + 2 * lane];
    gi = g[3 + 2 * lane];
  }
  const unsigned alive = __ballot_sync(FULL, full && (uint32_t)lane < cnt && gd == worst);
  __syncwarp();
  if (alive == 0) {
    if (lane == 0) g[0] = 0;
    __syncwarp();
    return kInvalid;
  }
  const int o = __ffs(alive) - 1;
  if (lane == o) g[2 + 2 * o] = 0;          // taken (0 is no distance word of a used slot)
  __syncwarp();
  return __shfl_sync(FULL, gi, o);
}

// The candidate/result pool: at most ef keys, unsorted, column-distributed (entry e lives in
// lane e % 32).  Two storages with one interface:
//   RegPool<SLOTS>  ef <= 32*SLOTS: the column sits in registers; column min/max are a few
//                   compare-selects recomputed on demand by all lanes at once
//   SmemPool        any ef: the column sits in shared memory, with cached column statistics
// Interface: seed(), pop_closest_unexpanded(), admit(), for_each_id(), kth().
template <int SLOTS>
struct RegPool {
  uint64_t k[SLOTS];     // empty slots hold NONE (flag set => never "unexpanded", and skipped for max)
  uint32_t size, ef;
  int lane;

  __device__ __forceinline__ void init(uint64_t *, uint32_t ef_, int lane_) {
    ef = ef_;
    lane = lane_;
    size = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) k[s] = NONE;
  }
  __device__ __forceinline__ void put(uint32_t e, uint64_t key) {   // called by the owner lane only
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) k[s] = ((int)(e >> 5) == s) ? key : k[s];   // select, not k[e>>5] = ..: keeps k in registers
  }
  __device__ __forceinline__ void seed(uint64_t key) {
    if (lane == 0) k[0] = key;
    size = 1;
  }
  __device__ __forceinline__ uint64_t col_min_un(int &slot) const {
    uint64_t m = NONE;
    slot = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const bool un = !((uint32_t)k[s] & FLAG);
      if (un && k[s] < m) {
        m = k[s];
        slot = s;
      }
    }
    return m;
  }
  __device__ __forceinline__ uint64_t col_max(int &slot) const {
    uint64_t m = 0;
    slot = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const uint64_t km = k[s] & KEYMASK;
      const bool used = (uint32_t)(s * 32 + lane) < size;
      if (used && km >= m) {
        m = km;
        slot = s;
      }
    }
    return m;
  }
  // closest unexpanded entry: marks it expanded and returns its node id, kInvalid if none
  __device__ __forceinline__ uint32_t pop_closest_unexpanded() {
    int slot;
    const uint64_t m = col_min_un(slot);
    const int o = warp_argmin_key(m);
    if (o < 0) return kInvalid;
    if (lane == o) {
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) k[s] = (s == slot) ? (k[s] | (uint64_t)FLAG) : k[s];
    }
    return (uint32_t)__shfl_sync(FULL, (uint32_t)m, o);
  }
  // admit scored neighbours, one per lane; returns the ballot of lanes whose key entered
  __device__ __forceinline__ unsigned admit(bool valid, uint64_t key) {
    unsigned entered = 0;
    const unsigned vmask = __ballot_sync(FULL, valid);
    if (vmask == 0) return 0;
    unsigned todo = vmask;
    if (size < ef) {   // room left: the first (ef - size) candidates are appended unconditionally
      const uint32_t room = ef - size;
      const uint32_t n_app = min(room, (uint32_t)__popc(vmask));
      for (uint32_t j = 0; j < n_app; ++j) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint64_t ck = __shfl_sync(FULL, key, src);
        const uint32_t e = size + j;
        if ((int)(e & 31) == lane) put(e, ck);
        entered |= 1u << src;
      }
      size += n_app;
      if (todo == 0) return entered;
    }
    int slot;
    uint64_t cm = col_max(slot);
    int owner = warp_argmax_key(cm);
    uint64_t worst = __shfl_sync(FULL, cm, owner);
    todo &= __ballot_sync(FULL, valid && key < worst);   // the worst only gets smaller
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t ck = __shfl_sync(FULL, key, src);
      if (ck < worst) {
        if (lane == owner) {
#pragma unroll
          for (int s = 0; s < SLOTS; ++s) k[s] = (s == slot) ? ck : k[s];
        }
        entered |= 1u << src;
        if (todo) {
          cm = col_max(slot);
          owner = warp_argmax_key(cm);
          worst = __shfl_sync(FULL, cm, owner);
        }
      }
    }
    return entered;
  }
  // the largest key of the pool (0 if empty), warp-uniform
  __device__ __forceinline__ uint64_t worst_key() const {
    int slot;
    const uint64_t cm = col_max(slot);
    return __shfl_sync(FULL, cm, warp_argmax_key(cm));
  }
  // every entry becomes unexpanded again (a new layer of the layered beam, slim.h:228-233)
  __device__ __forceinline__ void clear_flags() {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) k[s] = ((uint32_t)(s * 32 + lane) < size) ? (k[s] & KEYMASK) : k[s];
  }
  // ---- hnsw_slimq pool semantics (SearchBuffer, slimq.h:80-151): the same (dist,id) may sit
  //      in the pool several times; "visited" == some copy carries the expanded flag ----
  // closest unexpanded entry; flags EVERY copy of it (the reference pops the later copies
  // and skips them as visited, slimq.h:700-702 — a no-op)
  __device__ __forceinline__ uint32_t pop_closest_unexpanded_dups() {
    int slot;
    const uint64_t m = col_min_un(slot);
    const int o = warp_argmin_key(m);
    if (o < 0) return kInvalid;
    const uint64_t g = __shfl_sync(FULL, m, o);
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) k[s] = (k[s] == g) ? (k[s] | (uint64_t)FLAG) : k[s];
    return (uint32_t)g;
  }
  // node id of the closest unexpanded entry without popping it (kInvalid if none)
  __device__ __forceinline__ uint32_t peek_closest_unexpanded() const {
    int slot;
    const uint64_t m = col_min_un(slot);
    const int o = warp_argmin_key(m);
    if (o < 0) return kInvalid;
    return (uint32_t)__shfl_sync(FULL, (uint32_t)m, o);
  }
  // slimq.h:741-745: a scored neighbour enters unless the pool is full and it is worse than
  // the worst entry, or it was expanded already (== a flagged copy of its key is in the pool:
  // an expanded entry that left the pool is worse than the worst from then on)
  // maybe: lanes whose candidate MAY have an expanded copy in the pool (a filter without false negatives, e.g. the
  // kernel's Bloom word); the duplicate scan is skipped for the others
  __device__ __forceinline__ unsigned admit_q(bool valid, uint64_t key, unsigned maybe = FULL) {
    unsigned entered = 0;
    unsigned todo = __ballot_sync(FULL, valid);
    if (todo == 0) return 0;
    int slot = 0, owner = 0;
    uint64_t worst = NONE;
    if (size >= ef) {
      const uint64_t cm = col_max(slot);
      owner = warp_argmax_key(cm);
      worst = __shfl_sync(FULL, cm, owner);
      todo &= __ballot_sync(FULL, valid && key < worst);
    }
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t ck = __shfl_sync(FULL, key, src);
      if ((maybe >> src) & 1u) {
        const uint64_t fk = ck | (uint64_t)FLAG;
        bool dup = false;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) dup |= (k[s] == fk);
        if (__any_sync(FULL, dup)) continue;
      }
      if (size < ef) {
        if ((int)(size & 31) == lane) put(size, ck);
        ++size;
        entered |= 1u << src;
        if (size == ef && todo) {
          const uint64_t cm = col_max(slot);
          owner = warp_argmax_key(cm);
          worst = __shfl_sync(FULL, cm, owner);
        }
      } else if (ck < worst) {
        if (lane == owner) {
#pragma unroll
          for (int s = 0; s < SLOTS; ++s) k[s] = (s == slot) ? ck : k[s];
        }
        entered |= 1u << src;
        if (todo) {
          const uint64_t cm = col_max(slot);
          owner = warp_argmax_key(cm);
          worst = __shfl_sync(FULL, cm, owner);
        }
      }
    }
    return entered;
  }
  template <typename F>
  __device__ __forceinline__ void for_each_id(F &&f) const {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s)
      if ((uint32_t)(s * 32 + lane) < size) f((uint32_t)k[s] & ~FLAG);
  }
  // smallest key strictly above `last` in this lane's column (NONE if none)
  __device__ __forceinline__ uint64_t col_next_above(uint64_t last) const {
    uint64_t m = NONE;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const uint64_t km = k[s] & KEYMASK;
      if ((uint32_t)(s * 32 + lane) < size && km > last && km < m) m = km;
    }
    return m;
  }
};

// RegPool with 32-bit comparisons — the pool of the fp32 traversal kernel.  Distances and ids sit
// in separate registers; every comparison on the hot path (closest unexpanded, worst, admission
// test) is on the 32-bit distance word alone: a 3-instruction min/max per lane, ONE REDUX per warp
// and a ballot.  Entries of equal distance are taken in (lane, slot) order; the admission test is
// the reference's strict `lowerBound > dist` (slim.h:403-404) on the distance alone.
//   kd[s]  ord(distance) of a used slot, 0 for an empty one          (worst = max kd)
//   ku[s]  ord(distance) while the entry is unexpanded, else ~0       (closest unexpanded = min ku)
//   id[s]  node id
template <int SLOTS>
struct RegPool32 {
  uint32_t kd[SLOTS], ku[SLOTS], id[SLOTS];
  uint32_t size, ef;
  int lane;

  __device__ __forceinline__ void init(uint64_t *, uint32_t ef_, int lane_) {
    ef = ef_;
    lane = lane_;
    size = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      kd[s] = 0u;
      ku[s] = 0xffffffffu;
      id[s] = 0xffffffffu;
    }
  }
  __device__ __forceinline__ void put(uint32_t e, uint32_t d, uint32_t i) {   // owner lane only
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const bool h = (int)(e >> 5) == s;
      kd[s] = h ? d : kd[s];
      ku[s] = h ? d : ku[s];
      id[s] = h ? i : id[s];
    }
  }
  __device__ __forceinline__ void seed(uint64_t key) {
    if (lane == 0) put(0, (uint32_t)(key >> 32), (uint32_t)key);
    size = 1;
  }
  __device__ __forceinline__ uint32_t col_min_un() const {
    uint32_t m = ku[0];
#pragma unroll
    for (int s = 1; s < SLOTS; ++s) m = min(m, ku[s]);
    return m;
  }
  __device__ __forceinline__ uint32_t col_max() const {
    uint32_t m = kd[0];
#pragma unroll
    for (int s = 1; s < SLOTS; ++s) m = max(m, kd[s]);
    return m;
  }
  __device__ __forceinline__ uint32_t pop_closest_unexpanded() {
    const uint32_t m = col_min_un();
    const uint32_t g = __reduce_min_sync(FULL, m);
    if (g == 0xffffffffu) return kInvalid;
    const int o = __ffs(__ballot_sync(FULL, m == g)) - 1;
    uint32_t node = 0;
    bool open = lane == o;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const bool h = open && ku[s] == g;
      node = h ? id[s] : node;
      ku[s] = h ? 0xffffffffu : ku[s];
      open = open && !h;
    }
    return __shfl_sync(FULL, node, o);
  }
  // node id of the closest unexpanded entry without popping it (kInvalid if none)
  __device__ __forceinline__ uint32_t peek_closest_unexpanded() const {
    const uint32_t m = col_min_un();
    const uint32_t g = __reduce_min_sync(FULL, m);
    if (g == 0xffffffffu) return kInvalid;
    const int o = __ffs(__ballot_sync(FULL, m == g)) - 1;
    uint32_t node = id[SLOTS - 1];
#pragma unroll
    for (int s = SLOTS - 2; s >= 0; --s) node = ku[s] == g ? id[s] : node;     // first matching slot wins
    return __shfl_sync(FULL, node, o);
  }
  __device__ __forceinline__ unsigned admit(bool valid, uint64_t key, uint32_t *ghosts = nullptr) {
    const uint32_t d = (uint32_t)(key >> 32), cid = (uint32_t)key;
    unsigned entered = 0;
    const unsigned vmask = __ballot_sync(FULL, valid);
    if (vmask == 0) return 0;
    unsigned todo = vmask;
    if (size < ef) {   // room left: the first (ef - size) candidates are appended unconditionally
      const uint32_t room = ef - size;
      const uint32_t n_app = min(room, (uint32_t)__popc(vmask));
      for (uint32_t j = 0; j < n_app; ++j) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t cd = __shfl_sync(FULL, d, src), ci = __shfl_sync(FULL, cid, src);
        const uint32_t e = size + j;
        if ((int)(e & 31) == lane) put(e, cd, ci);
        entered |= 1u << src;
      }
      size += n_app;
      if (todo == 0) return entered;
    }
    uint32_t cm = col_max();
    uint32_t worst = __reduce_max_sync(FULL, cm);
    todo &= __ballot_sync(FULL, valid && d < worst);   // the worst only gets smaller
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t cd = __shfl_sync(FULL, d, src);
      if (cd < worst) {
        const uint32_t ci = __shfl_sync(FULL, cid, src);
        const unsigned wmask = __ballot_sync(FULL, cm == worst);
        const int owner = __ffs(wmask) - 1;
        if ((wmask & (wmask - 1)) && ghosts) {     // exact tie at the boundary (see ghost_append): rare
          if (lane == owner) {
            uint32_t gu = 0xffffffffu, gi = 0;
            bool first = true;
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
              const bool h = first && kd[s] == worst;
              gu = h ? ku[s] : gu;
              gi = h ? id[s] : gi;
              first = first && !h;
            }
            if (gu != 0xffffffffu) ghost_append(ghosts, worst, gi);     // still unexpanded: the reference keeps it
          }
          __syncwarp();
        }
        bool open = lane == owner;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
          const bool h = open && kd[s] == worst;
          kd[s] = h ? cd : kd[s];
          ku[s] = h ? cd : ku[s];
          id[s] = h ? ci : id[s];
          open = open && !h;
        }
        entered |= 1u << src;
        if (todo) {
          cm = col_max();
          worst = __reduce_max_sync(FULL, cm);
        }
      }
    }
    return entered;
  }
  __device__ __forceinline__ uint32_t take_ghost(uint32_t *ghosts) {
    if (ghosts[0] == 0) return kInvalid;
    return ghost_take(ghosts, __reduce_max_sync(FULL, col_max()), size >= ef, lane);
  }
  // every entry becomes unexpanded again (a new layer of the layered beam, slim.h:228-233)
  __device__ __forceinline__ void clear_flags() {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) ku[s] = kd[s] ? kd[s] : 0xffffffffu;
  }
  // ---- hnsw_slimq pool semantics (SearchBuffer, slimq.h:80-151): the same (estimate, id) may sit
  //      in the pool several times; "visited" == some copy of the node is marked expanded ----
  // closest unexpanded entry; marks EVERY copy of that node (the reference pops the later copies
  // and skips them as visited, slimq.h:700-702 — a no-op).  A node's estimate is a function of
  // the node, so copies share the distance word.
  __device__ __forceinline__ uint32_t pop_closest_unexpanded_dups() {
    const uint32_t m = col_min_un();
    const uint32_t g = __reduce_min_sync(FULL, m);
    if (g == 0xffffffffu) return kInvalid;
    const int o = __ffs(__ballot_sync(FULL, m == g)) - 1;
    uint32_t node = id[SLOTS - 1];
#pragma unroll
    for (int s = SLOTS - 2; s >= 0; --s) node = ku[s] == g ? id[s] : node;
    node = __shfl_sync(FULL, node, o);
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) ku[s] = (ku[s] == g && id[s] == node) ? 0xffffffffu : ku[s];
    return node;
  }
  // slimq.h:741-745: a scored neighbour enters unless the pool is full and it is worse than the
  // worst entry, or it was expanded already (== an expanded copy of the node is in the pool: an
  // expanded entry that left the pool is worse than the worst from then on)
  __device__ __forceinline__ unsigned admit_q(bool valid, uint64_t key, unsigned maybe = FULL) {
    const uint32_t d = (uint32_t)(key >> 32), cid = (uint32_t)key;
    unsigned entered = 0;
    unsigned todo = __ballot_sync(FULL, valid);
    if (todo == 0) return 0;
    uint32_t cm = 0, worst = 0xffffffffu;
    if (size >= ef) {
      cm = col_max();
      worst = __reduce_max_sync(FULL, cm);
      todo &= __ballot_sync(FULL, valid && d < worst);
    }
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t cd = __shfl_sync(FULL, d, src), ci = __shfl_sync(FULL, cid, src);
      if ((maybe >> src) & 1u) {
        bool dup = false;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) dup |= (id[s] == ci && ku[s] == 0xffffffffu && kd[s] != 0u);
        if (__any_sync(FULL, dup)) continue;
      }
      if (size < ef) {
        if ((int)(size & 31) == lane) put(size, cd, ci);
        ++size;
        entered |= 1u << src;
        if (size == ef && todo) {
          cm = col_max();
          worst = __reduce_max_sync(FULL, cm);
        }
      } else if (cd < worst) {
        const int owner = __ffs(__ballot_sync(FULL, cm == worst)) - 1;
        bool open = lane == owner;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
          const bool h = open && kd[s] == worst;
          kd[s] = h ? cd : kd[s];
          ku[s] = h ? cd : ku[s];
          id[s] = h ? ci : id[s];
          open = open && !h;
        }
        entered |= 1u << src;
        if (todo) {
          cm = col_max();
          worst = __reduce_max_sync(FULL, cm);
        }
      }
    }
    return entered;
  }
  template <typename F>
  __device__ __forceinline__ void for_each_id(F &&f) const {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s)
      if (kd[s]) f(id[s]);
  }
  // smallest (distance,id) key strictly above `last` in this lane's column (NONE if none)
  __device__ __forceinline__ uint64_t col_next_above(uint64_t last) const {
    uint64_t m = NONE;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const uint64_t km = ((uint64_t)kd[s] << 32) | id[s];
      if (kd[s] && km > last && km < m) m = km;
    }
    return m;
  }
};

// RegPool32 without the `ku` column: the "expanded" mark is the top bit of the id word (node ids are < 2^31),
// so a slot costs two registers instead of three.  For ef 129..256 (5..8 slots per lane) that is the difference
// between a pool that fits the 80-register budget of 24 warps per SM and one that spills.  The closest-unexpanded
// scan pays one select per slot for it (once per hop); the worst-entry scan and the admission loop (several times
// per hop) are unchanged.  Same interface and the same tie rules as RegPool32 (fp32 kernel only).
//   kd[s]  ord(distance) of a used slot, 0 for an empty one
//   id[s]  node id, top bit set once expanded; 0xffffffff for an empty slot
template <int SLOTS>
struct RegPool32C {
  uint32_t kd[SLOTS], id[SLOTS];
  uint32_t size, ef;
  int lane;

  __device__ __forceinline__ void init(uint64_t *, uint32_t ef_, int lane_) {
    ef = ef_;
    lane = lane_;
    size = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      kd[s] = 0u;
      id[s] = 0xffffffffu;
    }
  }
  __device__ __forceinline__ void put(uint32_t e, uint32_t d, uint32_t i) {   // owner lane only
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const bool h = (int)(e >> 5) == s;
      kd[s] = h ? d : kd[s];
      id[s] = h ? i : id[s];
    }
  }
  __device__ __forceinline__ void seed(uint64_t key) {
    if (lane == 0) put(0, (uint32_t)(key >> 32), (uint32_t)key);
    size = 1;
  }
  __device__ __forceinline__ uint32_t un(int s) const { return (int32_t)id[s] < 0 ? 0xffffffffu : kd[s]; }
  __device__ __forceinline__ uint32_t col_min_un() const {
    uint32_t m = un(0);
#pragma unroll
    for (int s = 1; s < SLOTS; ++s) m = min(m, un(s));
    return m;
  }
  __device__ __forceinline__ uint32_t col_max() const {
    uint32_t m = kd[0];
#pragma unroll
    for (int s = 1; s < SLOTS; ++s) m = max(m, kd[s]);
    return m;
  }
  __device__ __forceinline__ uint32_t pop_closest_unexpanded() {
    const uint32_t m = col_min_un();
    const uint32_t g = __reduce_min_sync(FULL, m);
    if (g == 0xffffffffu) return kInvalid;
    const int o = __ffs(__ballot_sync(FULL, m == g)) - 1;
    uint32_t node = 0;
    bool open = lane == o;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const bool h = open && un(s) == g;
      node = h ? id[s] : node;
      id[s] = h ? (id[s] | FLAG) : id[s];
      open = open && !h;
    }
    return __shfl_sync(FULL, node, o);
  }
  __device__ __forceinline__ uint32_t peek_closest_unexpanded() const {
    const uint32_t m = col_min_un();
    const uint32_t g = __reduce_min_sync(FULL, m);
    if (g == 0xffffffffu) return kInvalid;
    const int o = __ffs(__ballot_sync(FULL, m == g)) - 1;
    uint32_t node = id[SLOTS - 1];
#pragma unroll
    for (int s = SLOTS - 2; s >= 0; --s) node = un(s) == g ? id[s] : node;     // first matching slot wins
    return __shfl_sync(FULL, node, o);
  }
  __device__ __forceinline__ unsigned admit(bool valid, uint64_t key, uint32_t *ghosts = nullptr) {
    const uint32_t d = (uint32_t)(key >> 32), cid = (uint32_t)key;
    unsigned entered = 0;
    const unsigned vmask = __ballot_sync(FULL, valid);
    if (vmask == 0) return 0;
    unsigned todo = vmask;
    if (size < ef) {   // room left: the first (ef - size) candidates are appended unconditionally
      const uint32_t room = ef - size;
      const uint32_t n_app = min(room, (uint32_t)__popc(vmask));
      for (uint32_t j = 0; j < n_app; ++j) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t cd = __shfl_sync(FULL, d, src), ci = __shfl_sync(FULL, cid, src);
        const uint32_t e = size + j;
        if ((int)(e & 31) == lane) put(e, cd, ci);
        entered |= 1u << src;
      }
      size += n_app;
      if (todo == 0) return entered;
    }
    uint32_t cm = col_max();
    uint32_t worst = __reduce_max_sync(FULL, cm);
    todo &= __ballot_sync(FULL, valid && d < worst);   // the worst only gets smaller
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t cd = __shfl_sync(FULL, d, src);
      if (cd < worst) {
        const uint32_t ci = __shfl_sync(FULL, cid, src);
        const unsigned wmask = __ballot_sync(FULL, cm == worst);
        const int owner = __ffs(wmask) - 1;
        if ((wmask & (wmask - 1)) && ghosts) {     // exact tie at the boundary (see ghost_append): rare
          if (lane == owner) {
            uint32_t gi = 0xffffffffu;
            bool first = true;
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
              const bool h = first && kd[s] == worst;
              gi = h ? id[s] : gi;
              first = first && !h;
            }
            if ((int32_t)gi >= 0) ghost_append(ghosts, worst, gi);     // still unexpanded: the reference keeps it
          }
          __syncwarp();
        }
        bool open = lane == owner;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
          const bool h = open && kd[s] == worst;
          kd[s] = h ? cd : kd[s];
          id[s] = h ? ci : id[s];
          open = open && !h;
        }
        entered |= 1u << src;
        if (todo) {
          cm = col_max();
          worst = __reduce_max_sync(FULL, cm);
        }
      }
    }
    return entered;
  }
  __device__ __forceinline__ uint32_t take_ghost(uint32_t *ghosts) {
    if (ghosts[0] == 0) return kInvalid;
    return ghost_take(ghosts, __reduce_max_sync(FULL, col_max()), size >= ef, lane);
  }
  // every entry becomes unexpanded again (a new layer of the layered beam, slim.h:228-233)
  __device__ __forceinline__ void clear_flags() {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) id[s] = kd[s] ? (id[s] & ~FLAG) : id[s];
  }
  template <typename F>
  __device__ __forceinline__ void for_each_id(F &&f) const {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s)
      if (kd[s]) f(id[s] & ~FLAG);
  }
  // smallest (distance,id) key strictly above `last` in this lane's column (NONE if none)
  __device__ __forceinline__ uint64_t col_next_above(uint64_t last) const {
    uint64_t m = NONE;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const uint64_t km = ((uint64_t)kd[s] << 32) | (id[s] & ~FLAG);
      if (kd[s] && km > last && km < m) m = km;
    }
    return m;
  }
};

struct SmemPool {
  uint64_t *pool;
  uint32_t size, ef;
  int lane;
  uint64_t min_un, max_all;    // cached column statistics
  uint32_t min_e, max_e;

  __device__ __forceinline__ void init(uint64_t *mem, uint32_t ef_, int lane_) {
    pool = mem;
    ef = ef_;
    lane = lane_;
    size = 0;
  }
  __device__ __forceinline__ void rescan_min() {
    min_un = NONE;
    min_e = 0;
    for (uint32_t e = lane; e < size; e += 32) {
      const uint64_t k = pool[e];
      if (!((uint32_t)k & FLAG) && k < min_un) {
        min_un = k;
        min_e = e;
      }
    }
  }
  __device__ __forceinline__ void rescan_max() {
    max_all = 0;
    max_e = 0;
    for (uint32_t e = lane; e < size; e += 32) {
      const uint64_t km = pool[e] & KEYMASK;
      if (km >= max_all) {
        max_all = km;
        max_e = e;
      }
    }
  }
  __device__ __forceinline__ void seed(uint64_t key) {
    if (lane == 0) pool[0] = key;
    size = 1;
    __syncwarp();
    rescan_min();
    rescan_max();
  }
  __device__ __forceinline__ uint32_t pop_closest_unexpanded() {
    const int o = warp_argmin_key(min_un);
    if (o < 0) return kInvalid;
    const uint32_t node = (uint32_t)__shfl_sync(FULL, (uint32_t)min_un, o);
    if (lane == o) {
      pool[min_e] |= (uint64_t)FLAG;
      rescan_min();
    }
    return node;
  }
  __device__ __forceinline__ unsigned admit(bool valid, uint64_t key, uint32_t *ghosts = nullptr) {
    unsigned entered = 0;
    const unsigned vmask = __ballot_sync(FULL, valid);
    if (vmask == 0) return 0;
    unsigned todo = vmask;
    if (size < ef) {
      const uint32_t room = ef - size;
      const uint32_t rank = (uint32_t)__popc(vmask & ((1u << lane) - 1));
      const bool app = valid && rank < room;
      if (app) pool[size + rank] = key;
      const unsigned am = __ballot_sync(FULL, app);
      entered |= am;
      todo &= ~am;
      size += min(room, (uint32_t)__popc(vmask));
      __syncwarp();
      rescan_min();
      rescan_max();
      if (todo == 0) return entered;
    }
    int owner = warp_argmax_key(max_all);
    uint64_t worst = __shfl_sync(FULL, max_all, owner);
    // the reference's test is on the distance alone and strict (`lowerBound > dist`, slim.h:403-404)
    todo &= __ballot_sync(FULL, valid && (uint32_t)(key >> 32) < (uint32_t)(worst >> 32));
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t ck = __shfl_sync(FULL, key, src);
      if ((uint32_t)(ck >> 32) < (uint32_t)(worst >> 32)) {
        // exact tie at the boundary (see ghost_append): another column's worst carries the same distance
        const unsigned tmask = __ballot_sync(FULL, (uint32_t)(max_all >> 32) == (uint32_t)(worst >> 32) && size > (uint32_t)lane);
        if ((tmask & (tmask - 1)) && ghosts) {
          if (lane == owner && !((uint32_t)pool[max_e] & FLAG)) ghost_append(ghosts, (uint32_t)(worst >> 32), (uint32_t)worst & ~FLAG);
          __syncwarp();
        }
        if (lane == owner) {
          const bool was_min = max_e == min_e && min_un != NONE;
          pool[max_e] = ck;
          if (was_min) {
            rescan_min();            // the displaced entry was this column's closest unexpanded
          } else if (ck < min_un) {
            min_un = ck;
            min_e = max_e;
          }
          rescan_max();
        }
        entered |= 1u << src;
        if (todo) {
          owner = warp_argmax_key(max_all);
          worst = __shfl_sync(FULL, max_all, owner);
        }
      }
    }
    return entered;
  }
  __device__ __forceinline__ uint32_t take_ghost(uint32_t *ghosts) {
    if (ghosts[0] == 0) return kInvalid;
    const int o = warp_argmax_key(max_all);
    const uint64_t worst = __shfl_sync(FULL, max_all, o);
    return ghost_take(ghosts, (uint32_t)(worst >> 32), size >= ef, lane);
  }
  __device__ __forceinline__ uint64_t worst_key() const {
    return __shfl_sync(FULL, max_all, warp_argmax_key(max_all));
  }
  __device__ __forceinline__ void clear_flags() {
    __syncwarp();
    for (uint32_t e = lane; e < size; e += 32) pool[e] &= KEYMASK;
    __syncwarp();
    rescan_min();
  }
  // ---- hnsw_slimq pool semantics, see RegPool ----
  __device__ __forceinline__ uint32_t pop_closest_unexpanded_dups() {
    const int o = warp_argmin_key(min_un);
    if (o < 0) return kInvalid;
    const uint64_t g = __shfl_sync(FULL, min_un, o);
    bool hit = false;
    for (uint32_t e = lane; e < size; e += 32)
      if (pool[e] == g) {
        pool[e] = g | (uint64_t)FLAG;
        hit = true;
      }
    if (hit) rescan_min();
    return (uint32_t)g;
  }
  __device__ __forceinline__ uint32_t peek_closest_unexpanded() const {
    const int o = warp_argmin_key(min_un);
    if (o < 0) return kInvalid;
    return (uint32_t)__shfl_sync(FULL, (uint32_t)min_un, o);
  }
  __device__ __forceinline__ unsigned admit_q(bool valid, uint64_t key, unsigned maybe = FULL) {
    unsigned entered = 0;
    unsigned todo = __ballot_sync(FULL, valid);
    if (todo == 0) return 0;
    int owner = 0;
    uint64_t worst = NONE;
    if (size >= ef) {
      owner = warp_argmax_key(max_all);
      worst = __shfl_sync(FULL, max_all, owner);
      todo &= __ballot_sync(FULL, valid && key < worst);
    }
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t ck = __shfl_sync(FULL, key, src);
      if ((maybe >> src) & 1u) {
        const uint64_t fk = ck | (uint64_t)FLAG;
        bool dup = false;
        for (uint32_t e = lane; e < size; e += 32) dup |= (pool[e] == fk);
        if (__any_sync(FULL, dup)) continue;
      }
      if (size < ef) {
        if ((int)(size & 31) == lane) {
          pool[size] = ck;
          if (ck < min_un) {
            min_un = ck;
            min_e = size;
          }
          if (ck >= max_all) {
            max_all = ck;
            max_e = size;
          }
        }
        ++size;
        entered |= 1u << src;
        if (size == ef && todo) {
          owner = warp_argmax_key(max_all);
          worst = __shfl_sync(FULL, max_all, owner);
        }
      } else if (ck < worst) {
        if (lane == owner) {
          const bool was_min = max_e == min_e && min_un != NONE;
          pool[max_e] = ck;
          if (was_min) {
            rescan_min();
          } else if (ck < min_un) {
            min_un = ck;
            min_e = max_e;
          }
          rescan_max();
        }
        entered |= 1u << src;
        if (todo) {
          owner = warp_argmax_key(max_all);
          worst = __shfl_sync(FULL, max_all, owner);
        }
      }
      __syncwarp();
    }
    return entered;
  }
  template <typename F>
  __device__ __forceinline__ void for_each_id(F &&f) const {
    for (uint32_t e = lane; e < size; e += 32) f((uint32_t)pool[e] & ~FLAG);
  }
  __device__ __forceinline__ uint64_t col_next_above(uint64_t last) const {
    uint64_t m = NONE;
    for (uint32_t e = lane; e < size; e += 32) {
      const uint64_t km = pool[e] & KEYMASK;
      if (km > last && km < m) m = km;
    }
    return m;
  }
};

}  // namespace
}  // namespace hs
