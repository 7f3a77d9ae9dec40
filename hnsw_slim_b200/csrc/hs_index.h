// The index handle behind the C ABI (hs_index) and the internal entry points other translation
// units of the library use (shard_group.cu, graph_gpu.cu).
#pragma once
#include <cuda_runtime.h>

#include <memory>
#include <mutex>
#include <vector>

#include "hs_internal.h"
#include "traverse_fp32.cuh"
#include "traverse_slimq.cuh"

// Launches in flight at once are bounded by what fits on the GPU (a dozen small grids); a slot is
// reused only kWorkRing launches later.
constexpr unsigned int kWorkRing = 1024;

struct hs_index {
  hs_index_info info{};
  int device = 0;
  int sm_count = 148;
  // HBM-resident index
  float *d_vec = nullptr;
  uint32_t *d_adj0 = nullptr;
  int32_t *d_upper_slot = nullptr;
  uint32_t *d_upper_adj[hs::kMaxLevels] = {};
  uint32_t *d_labels = nullptr;
  uint8_t *d_deleted = nullptr;
  // hnsw_slimq payload
  uint2 *d_qrec = nullptr;          // n x (words + 2) uint2: code words, (f_add, f_rescale), (cluster, 0)
  float *d_centroids = nullptr;     // num_cluster x padded_dim (rotated)
  uint8_t *d_flip = nullptr;        // 4 * padded_dim / 8
  uint32_t words = 0, trunc_dim = 0;
  // hnsw_slimq fields the file holds but the search does not read, kept on the host for hs_save_index
  std::vector<float> f_error;       // n
  uint64_t ex_bits = 0, size_ex = 0;
  uint32_t level_count[hs::kMaxLevels] = {};
  // delta patches (patch.cu): an index loaded with hs_load_reserve has rows for `capacity` nodes and keeps the
  // small host-side arrays (levels, upper-level slots and rows, labels) as a mirror; null / n otherwise
  size_t capacity = 0;
  size_t cap_upper_words[hs::kMaxLevels] = {};
  std::unique_ptr<hs::HostGraph> mirror;
  double t_const = 0.0;
  // per-call scratch
  unsigned long long *d_work = nullptr;    // ring of kWorkRing tagged work counters (traverse_common.cuh)
  unsigned int launch_seq = 1;             // tags start at 1 (slots are initialised to 0xff..ff)
  int overlap = 0;                         // hs_set_overlap
  unsigned long long *d_stats = nullptr;   // [0] n_dist [1] n_hops [2] n_rerank
  // staging for the host-buffer entry points
  cudaStream_t stream = nullptr;
  float *d_q = nullptr;
  uint32_t *d_lab = nullptr;
  float *d_dist = nullptr;
  uint32_t *d_perq = nullptr;
  size_t cap_q = 0, cap_out = 0, cap_perq = 0;
  int hash_bits_override = 0;
  int ghash_mode = -1;                     // HS_GHASH: -1 auto, 0 shared-memory visited tables, 1 global-memory
  uint32_t *d_ghash = nullptr;             // two halves, alternated by consecutive (possibly overlapping) launches
  size_t cap_ghash = 0;
  uint32_t traverse_flags = 9;             // bit0: L2 row prefetch; bit1: speculative next-pop adjacency load (measured: a loss); bit3: evict_last adjacency prefetch
  uint32_t slimq_flags = 0;
  // the launch plan of the last fp32 traversal (occupancy queries are not free on the host)
  bool plan_ok = false;
  uint32_t plan_ef = 0;
  size_t plan_nq = 0;
  hs::TraverseLaunch plan_l{};
  hs::TraverseParams plan_p{};
  bool planq_ok = false;
  uint32_t planq_ef = 0;
  size_t planq_nq = 0, planq_k = 0;
  hs::TraverseQLaunch planq_l{};
  hs::TraverseQParams planq_p{};
  // completion events of the batches handed to hs_search_batch_submit and not yet waited for (FIFO)
  static constexpr int kEventRing = 64;
  cudaEvent_t ev_ring[kEventRing] = {};
  unsigned long long ev_head = 0, ev_tail = 0;      // [head, tail) are outstanding
  bool zero_copy = true;                   // hs_search_batch reads/writes pinned+mapped host buffers in place
  std::mutex mu;
};

namespace hs {

// cudaSetDevice(device) with the error text the C ABI promises (no device => HS_ERR_CUDA, no fallback)
int select_device(int device);

// Device-visible alias of a host buffer when the whole range [p, p + bytes) is page-locked and mapped
// into the current device's address space; nullptr otherwise.
void *mapped_alias(const void *p, size_t bytes);

// One traversal launch of `ix` over a device-visible query batch (the body of hs_search_batch_device).
// plan_warps != nullptr: do not launch, only plan the launch shape (cached in the handle) and return
// the number of warps the launch will have (grid x warps per CTA) — the shard group needs the total over
// its local launches before the first one starts (ScatterDst::done_target).
int search_device(hs_index *ix, const float *d_queries, size_t nq, size_t k, uint32_t *d_labels, float *d_dists,
                  uint32_t *d_perq, cudaStream_t stream, const ScatterDst *scatter = nullptr,
                  uint32_t *plan_warps = nullptr);

// A finished index whose arrays already live on the device (graph_gpu.cu); adopt_device_graph wraps it
// into an hs_index that owns them (on failure the arrays are freed).
struct DeviceGraph {
  size_t n = 0, dim = 0, dim_padded = 0;
  int metric = 0, kind = HS_KIND_SLIM;
  uint64_t M = 0, maxM = 0, maxM0 = 0, ef_construction = 0;
  int maxlevel = 0, threshold_level = 0;
  uint32_t enterpoint = 0, deg0_stride = 32, max_deg0 = 0, upper_stride = 8, n_upper = 0;
  uint64_t sum_deg0 = 0;
  uint32_t level_count[kMaxLevels] = {};
  float *d_vec = nullptr;
  uint32_t *d_adj0 = nullptr;
  int32_t *d_upper_slot = nullptr;
  uint32_t *d_upper_adj[kMaxLevels] = {};
  const uint32_t *h_labels = nullptr;      // host, n entries
  // hnsw_slimq payload (kind == HS_KIND_SLIMQ)
  uint2 *d_qrec = nullptr;
  float *d_centroids = nullptr;            // rotated, num_cluster x padded_dim_q
  uint8_t *d_flip = nullptr;
  uint64_t padded_dim_q = 0, num_cluster = 0;
  uint32_t trunc_dim = 0;
  std::vector<float> h_f_error;            // host, n entries; moved into the handle
};
int adopt_device_graph(DeviceGraph &dg, int device, hs_index **out);

// patch.cu: the device side of patchFromStream (slim.h:2206-2388); the caller holds ix->mu
int apply_patch_device(hs_index *ix, const PatchSet &ps, const PatchRows &rows, hs_patch_info *info);

// graph_gpu.cu
int gpu_build_slim_index(const float *base, size_t n, size_t dim, int metric, const hs_build_params *bp,
                         double branching, const uint64_t *labels, int device, hs_index **out);
int gpu_build_slimq_index(const float *base, size_t n, size_t dim, const hs_build_params *bp, double branching,
                          const float *centroids, size_t num_cluster, const uint64_t *labels, int device,
                          hs_index **out);
int gpu_debug_convert(const char *hnsw_graph_path, size_t dim, int metric, const hs_build_params *bp, int device,
                      hs_index **out);

}  // namespace hs
