// Internal declarations shared by the host loader, the C ABI and the kernels.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/hnswslim_b200.h"

namespace hs {

constexpr uint32_t kInvalid = 0xFFFFFFFFu;
constexpr int kMaxLevels = 32;   // upper levels addressable by the kernels
constexpr int kTeam = 8;         // lanes cooperating on one vector row
constexpr int kRowAlignFloats = 32;   // 128-byte rows: dim padded to a multiple of 32 floats

void set_error(const std::string &msg);

// Fused exchange of the sharded path (hs_search_batch_device_scatter): besides (or instead of) its
// own output tables a traversal kernel stores every result row into the gather buffers of up to
// kMaxScatter ranks — local memory, or peer memory mapped over NVLink (CUDA IPC) — at row
// row0 + query, so the "all-gather" of the per-shard top-k lists costs no collective call at all.
constexpr int kMaxScatter = 16;
struct ScatterDst {
  uint32_t n = 0;                          // 0: plain out_labels / out_dists
  unsigned long long row0 = 0;             // first row of this shard's slot in every destination table
  uint32_t *labels[kMaxScatter] = {};
  float *dists[kMaxScatter] = {};
  // Completion protocol of a shard group (shard_group.cu), all optional (null / 0 = off).  The
  // traversal launches of one batch count their finished warps in done_ctr; the warp that brings it to
  // done_target resets it and writes `seq` into word [this rank] of every rank's flag array (release,
  // system scope) — the "my rows of batch seq have landed" signal that used to be a stream memory
  // operation between two launches and thereby cut the programmatic-launch chain.  Before its first
  // row store a warp checks that every rank has merged batch seq - depth (acks[r] >= ack_need): the
  // table slot it is about to overwrite is free.
  unsigned int *done_ctr = nullptr;
  uint32_t done_target = 0;
  uint32_t seq = 0;
  uint32_t n_flags = 0;
  uint32_t *flags[kMaxScatter] = {};
  const uint32_t *acks = nullptr;          // local array, one word per rank
  uint32_t n_acks = 0, ack_need = 0;
  unsigned long long ack_timeout_ns = 0;   // give up on a peer's acknowledgement after this long ...
  unsigned int *status = nullptr;          // ... and record it here (local word; 0 = healthy)
};

// A .graph file flattened on the host, ready to upload (see DESIGN.md "HBM layout").
struct HostGraph {
  // header, as stored by saveIndex (slim.h:717-739 / slimq.h:1161-1190)
  uint64_t n = 0, size_data_per_element = 0, label_offset = 0, offset_total = 0, offset_data = 0,
           offset_nbr = 0, maxM = 0, maxM0 = 0, M = 0, ef_construction = 0;
  int32_t maxlevel = 0, threshold_level = 0;
  uint32_t enterpoint = 0;
  bool has_deleted = false;
  int kind = HS_KIND_SLIM;
  size_t dim = 0, dim_padded = 0;

  // flattened graph.  reserve_strides: rows wide enough for ANY list the header allows (maxM0 / maxM ids) instead
  // of the longest list found — an index that will receive delta patches (patch.cu) must not need re-striding
  bool reserve_strides = false;
  bool mirror_only = false;     // adj0 / vec / payload arrays were dropped after the upload: the small arrays mirror a device index
  uint32_t deg0_stride = 32, max_deg0 = 0, upper_stride = 16, max_deg_upper = 0, n_upper = 0;
  uint64_t sum_deg0 = 0;
  std::vector<float> vec;             // n x dim_padded (hnsw_slim); empty for slimq
  std::vector<uint32_t> adj0;         // n x deg0_stride, kInvalid-padded
  std::vector<int32_t> upper_slot;    // n; -1 for level-0-only nodes; slots sorted by level desc
  std::vector<uint32_t> level_count;  // [maxlevel+1]: nodes with level >= l
  std::vector<std::vector<uint32_t>> upper_adj;  // [l] : level_count[l] x upper_stride (l >= 1)
  std::vector<uint32_t> labels;       // n, external labels truncated to 32 bit (slim.h:2129)
  std::vector<int8_t> levels;         // n
  std::vector<uint8_t> deleted;       // n, bit 0 of record byte 6 (slim.h:1776-1781); all 0 in practice

  // hnsw_slimq payload (slimq.h:1187-1206, data_layout.hpp:171-194)
  uint64_t num_cluster = 0, padded_dim_q = 0, ex_bits = 0;
  uint8_t metric_type_q = 0;
  std::vector<float> centroids;       // num_cluster x padded_dim_q (already rotated)
  std::vector<uint8_t> rotator_flip;  // 4 * padded_dim_q / 8 bytes (rotator.hpp:263-275)
  std::vector<uint32_t> cluster_id;   // n
  std::vector<uint64_t> bin_code;     // n x padded_dim_q/64 (MSB-first bit order)
  std::vector<float> f_add, f_rescale, f_error;   // n each
};

// Parses a reference .graph image.  Returns HS_OK or a negative hs_status (message via set_error).
int parse_graph(const uint8_t *bytes, size_t size, int kind, size_t dim, HostGraph *out);

// ---- delta patches: the stream HierarchicalNSWSlim::patchFromStream consumes (slim.h:2206-2388), patch.cu ----
struct PatchNode {
  uint32_t id = 0;
  int32_t level = 0;
  uint32_t total = 0;
  bool is_new = false;                 // "changed_new" record: carries the label and brings a vector
  uint64_t label = 0;
  const uint8_t *blob = nullptr;       // [uint16 offsets[level]][uint32 ids[total]] inside the stream (unaligned), or null
  const uint8_t *row = nullptr;        // inline vector (dim floats, unaligned) or null
  // level-l slice (slim.h:245-260): ids[(l ? offsets[l-1] : 0) .. (l == level ? total : offsets[l]))
  uint32_t slice(int l, const uint8_t **ids) const;
};
struct PatchSet {
  uint64_t n_after = 0, n_old = 0, n_new = 0;
  size_t consumed = 0;
  std::vector<PatchNode> nodes;        // stream order; a later record of the same id supersedes an earlier one
};
// Parses and validates a patch stream against an index of `n_before` nodes and room for `capacity`.
int parse_patch(const uint8_t *bytes, size_t size, size_t dim, bool inline_rows, uint64_t n_before, uint64_t capacity,
                PatchSet *out);
// The vector a "changed_new" record brings: inline, or looked up by label in the caller's rows
// (rows[label] when row_labels == nullptr — patchFromStream(in, data_set), slim.h:2225 — else the row whose
// row_labels entry equals the label — patchFromStream(in, new_data), slim.h:2360).  nullptr if absent.
struct PatchRows {
  const float *rows = nullptr;
  const uint64_t *row_labels = nullptr;
  size_t n_rows = 0, dim = 0;
  std::vector<std::pair<uint64_t, size_t>> sorted;   // (label, row) when row_labels is given
  void prepare();
  const uint8_t *find(const PatchNode &nd) const;
};
// Applies a parsed patch to the host image: levels, labels, upper-level slots and rows are always maintained;
// adj0 / vec only when they are present (host-only inspection, hs_debug_patch) — a device-resident index keeps
// just the small arrays as its mirror.  *upper_changed: the upper-level arrays were rebuilt.
int apply_patch_host(HostGraph *g, const PatchSet &ps, const PatchRows &rows, bool *upper_changed);
int read_file(const char *path, std::vector<uint8_t> *out);
double slimq_default_tconst(size_t padded_dim, size_t ex_bits);

// graph_build.cpp — HNSW construction + HNSW-Slim pruning + saveIndex file format
int build_slim_graph(const float *base, size_t n, size_t dim, int metric, size_t M, size_t ef_construction,
                     double branching, int threshold_level, float top_pct0, float top_pct, size_t top_M0,
                     size_t low_m0, size_t top_M, size_t low_m, int threads, uint64_t seed,
                     const uint64_t *labels, const char *out_path);

int build_hnsw_graph(const float *base, size_t n, size_t dim, int metric, size_t M, size_t ef_construction,
                     double branching, int threads, uint64_t seed, const uint64_t *labels, const char *out_path);

int build_slimq_graph(const float *base, size_t n, size_t dim, size_t M, size_t ef_construction, double branching,
                      int threshold_level, float top_pct0, float top_pct, size_t top_M0, size_t low_m0,
                      size_t top_M, size_t low_m, int threads, uint64_t seed, const float *centroids,
                      size_t num_cluster, const uint32_t *cluster_ids, const uint64_t *labels,
                      const char *out_path);

// HierarchicalNSWSlimQ::saveIndex's file (slimq.h:1161-1216), written by build_slimq_graph and hs_save_index.
// Each element record is [int32 level][uint32 total][uint64 label][8 pointer bytes = 0][uint32 cluster @24]
// [uint64 code[padded_dim / 64] @28, MSB-first][float f_add, f_rescale, f_error][ex block, size_ex bytes = 0].
// The 3-bit ex-codes are not computed and the ex block is written as zeros: no search path reads it (SURVEY.md
// App. A, only get_bin_est is called, slimq.h:737-738).
struct SlimqHead {
  uint64_t n = 0, maxM = 0, maxM0 = 0, M = 0, ef_construction = 0;
  int32_t maxlevel = 0, threshold_level = 0;
  uint32_t enterpoint = 0;
  uint64_t num_cluster = 0, dim = 0, padded_dim = 0, ex_bits = 0, size_ex = 0;
  const float *centroids = nullptr;    // num_cluster x padded_dim, rotated
  const uint8_t *flip = nullptr;       // rotator sign bytes, 4 * padded_dim / 8
};
struct SlimqNode {
  int32_t level = 0;
  uint32_t total = 0;                  // neighbour ids over all of the node's levels
  uint64_t label = 0;
  uint32_t cluster = 0;
  const uint64_t *code = nullptr;      // padded_dim / 64 words
  float f_add = 0.f, f_rescale = 0.f, f_error = 0.f;
};
// Writes the header, the RaBitQ metadata, centroids, flip bytes and the n records to `path`, then the per-node
// neighbour blobs through blobs(f).  nodes(i0, cnt, out) fills out[0, cnt) with nodes i0 .. i0 + cnt - 1, in slabs
// of increasing i0; it returns HS_OK or an error code it has reported.  -> HS_OK, HS_ERR_IO or the nodes() code.
int write_slimq_file(const char *path, const SlimqHead &h,
                     const std::function<int(size_t i0, size_t cnt, SlimqNode *out)> &nodes,
                     const std::function<bool(FILE *f)> &blobs);

// pieces of the hnsw_slimq builder shared with the device builder (graph_gpu.cu)
void host_rotate(const float *x, size_t dim, size_t pd, size_t td, const uint8_t *flip, float *out);
void host_kmeans(const float *base, size_t n, size_t dim, size_t k, int iters, uint64_t seed, int threads,
                 std::vector<float> &cent, std::vector<uint32_t> &ids);

}  // namespace hs
