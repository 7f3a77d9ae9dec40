/* hnswslim_b200 — C ABI of the B200-native batched query engine for the HNSW-Slim
 * search hot path.  Built into hnsw_slim_b200/_build/libhnswslim_b200.so.
 *
 * Every entry point names the reference interface it replaces
 * (reference = InfiniteNightmare/HNSW-Slim; slim.h = third_party/hnswlib/hnswalg_slim.h,
 * slimq.h = third_party/hnswlib/hnswalg_slimq.h).  Plain pointers and sizes only:
 * the reference side binds it with a 20-line C++ shim (INTEGRATION.md).
 *
 * All functions return HS_OK (0) or a negative hs_status; hs_last_error() returns
 * the message of the calling thread's last failure (the reference throws
 * std::runtime_error at the same places: slim.h:757-758,785-788,804-806).
 * There is NO CPU fallback: without a CUDA device every compute entry point fails
 * with HS_ERR_CUDA.
 */
#ifndef HNSWSLIM_B200_H
#define HNSWSLIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HS_ABI_VERSION 1

typedef enum {
  HS_OK = 0,
  HS_ERR_ARG = -1,     /* bad argument */
  HS_ERR_IO = -2,      /* cannot open / truncated / inconsistent .graph file */
  HS_ERR_CUDA = -3,    /* CUDA runtime error (incl. no device) */
  HS_ERR_NOMEM = -4,   /* host or device allocation failed */
  HS_ERR_UNSUPPORTED = -5
} hs_status;

/* --solve_strategy values of main.cc:111-139 that have a GPU engine */
typedef enum {
  HS_KIND_SLIM = 0,   /* hnsw_slim and hnsw_slimzero (same file format, same searchKnn: hnswalg_slimzero.h:701-735,1675-1771) */
  HS_KIND_SLIMQ = 1,  /* hnsw_slimq */
  HS_KIND_HNSW = 2    /* hnsw: the un-pruned hnswlib index (hnsw_strategy.h:15-61, hnswalg.h:748-893,1378-1440) */
} hs_kind;

/* hnswlib::L2Space (space_l2.h:214-251) / hnswlib::InnerProductSpace (space_ip.h:342-398) */
typedef enum { HS_METRIC_L2 = 0, HS_METRIC_IP = 1 } hs_metric;

typedef struct hs_index hs_index;   /* owns the HBM-resident copy of one .graph */

typedef struct {
  uint64_t n;                /* cur_element_count_                      slim.h:34  */
  uint64_t dim;
  uint64_t dim_padded;       /* floats per HBM row (128-byte multiple)             */
  uint64_t M, maxM, maxM0, ef_construction;      /*                      slim.h:38-41 */
  int32_t maxlevel;          /*                                         slim.h:44  */
  int32_t threshold_level;   /*                                         slim.h:45  */
  uint32_t enterpoint;       /* enterpoint_node_                        slim.h:49  */
  int32_t has_deleted;       /* has_deleted_elements_                   slim.h:36  */
  int32_t kind, metric;
  uint32_t deg0_stride;      /* ids per level-0 adjacency row in HBM (multiple of 32) */
  uint32_t max_deg0;         /* largest level-0 degree found in the file            */
  uint32_t upper_stride;     /* ids per upper-level adjacency row                   */
  uint32_t n_upper;          /* nodes with level > 0                                */
  uint64_t sum_deg0;         /* total level-0 edges (avg degree = sum_deg0 / n)     */
  uint64_t device_bytes;     /* HBM held by this handle                             */
  uint64_t ef;               /* current ef_ (hs_set_ef)                             */
  /* hnsw_slimq only (slimq.h:1187-1200), 0 otherwise */
  uint64_t padded_dim_q;     /* RaBitQ padded_dim (multiple of 64)                  */
  uint64_t num_cluster;
} hs_index_info;

/* Replaces HierarchicalNSWSlim::loadIndex (slim.h:753-815) and
 * HierarchicalNSWSlimQ::loadIndex + setDataset (slimq.h:1218-1313, :303-305):
 * parses the reference's .graph byte for byte, flattens it (fixed-stride,
 * 128-byte-aligned adjacency + vector store) and uploads it to `device`.
 *   dim       vector dimension (the reference takes it from the SpaceInterface)
 *   raw_base  hnsw_slimq only: the n_raw x dim float rows used for the exact
 *             rerank (slimq.h:747-749), indexed by internal id; copied to HBM.
 *             NULL for hnsw_slim (vectors live in the .graph). */
int hs_load(const char *graph_path, int kind, int metric, size_t dim, const float *raw_base,
            size_t n_raw, int device, hs_index **out);

/* Same, from a .graph image already in host memory (what a server holds after
 * patchFromStream; also used by tests).  */
int hs_load_memory(const void *graph_bytes, size_t graph_size, int kind, int metric, size_t dim,
                   const float *raw_base, size_t n_raw, int device, hs_index **out);

/* ---- Delta patches (SURVEY.md §8(f) rank 4) ---------------------------------------------------------
 * The reference's serving pair keeps a client index current without re-sending it: the server re-prunes its
 * full HNSW after every /updateIndex (convertFromHNSWWithDiff, slim.h:1110-1424; genPatch, slim.h:1427-1476;
 * hnsw_slim_server_patch.cc:186-279) and answers with the records that changed; the client applies the stream
 * with HierarchicalNSWSlim::patchFromStream (slim.h:2206-2388; hnsw_slim_client_update_patch.cc:41,73,179) and
 * goes on searching.
 *
 * hs_load_reserve = loadIndex(path, space, max_elements) with room to grow (slim.h:753-761,784; the client opens
 * its partial index with the final row count, hnsw_slim_client_update_patch.cc:113): hs_load for an hnsw_slim
 * .graph whose HBM arrays hold max_elements (>= n) nodes and whose adjacency rows are wide enough for any list
 * the header's maxM0 / maxM allow.  Only such an index accepts patches.
 *
 * hs_patch_apply = patchFromStream on the HBM-resident index: the changed level-0 rows (and the vectors and labels
 * of new nodes) are staged once and scattered into place by one kernel each; the upper-level rows (a small
 * fraction of the index) are re-derived on the host mirror and re-uploaded when a patched node has level > 0.
 * Like the reference it leaves the entry point and maxlevel alone.  Vectors of "changed_new" records:
 *   flags & HS_PATCH_INLINE_ROWS   they travel inside the stream        patchFromStream(in, true), slim.h:2292-2340
 *   rows, row_labels == NULL       rows[label * dim], label < n_rows    patchFromStream(in, data_set), slim.h:2206-2253
 *   rows, row_labels               the row i with row_labels[i] == label   patchFromStream(in, new_data), slim.h:2343-2388
 * Synchronous.  The call waits for the batches submitted through this handle (hs_search_batch_submit); launches
 * the caller made on its own streams (hs_search_batch_device) must have completed — patchFromStream is not
 * synchronised with searchKnn in the reference either.  A stream that fails validation leaves the index
 * unchanged; a CUDA failure in the middle of an update (HS_ERR_CUDA / HS_ERR_NOMEM) does not — free the handle
 * then.  hnsw_slim only. */
#define HS_PATCH_INLINE_ROWS 1u
typedef struct {
  uint64_t n_before, n_after;        /* cur_element_count_ before / after                         */
  uint64_t changed_old, changed_new; /* record counts of the stream                               */
  uint64_t bytes_consumed;           /* stream bytes read (a caller may concatenate patches)      */
  uint64_t rows_written;             /* level-0 rows scattered on the device                      */
  uint64_t upper_rebuilt;            /* 1: the upper-level arrays were re-derived and re-uploaded */
} hs_patch_info;
int hs_load_reserve(const char *graph_path, int kind, int metric, size_t dim, size_t max_elements, int device,
                    hs_index **out);
int hs_patch_apply(hs_index *, const void *patch, size_t patch_bytes, unsigned flags, const float *rows,
                   const uint64_t *row_labels, size_t n_rows, hs_patch_info *info_out);

/* ---- hs_service: single-query serving in front of the batched search -------------------------------------
 * The reference's server answers ONE query per request: each /query handler thread calls
 * hnsw_slim.searchKnn(vec, k, out) itself (hnsw_slim_server.cc:69-98, hnsw_slim_server_patch.cc:133-160), /setEf
 * calls setEf (:100-115).  hs_service_query is that handler body for the GPU engine: thread-safe and blocking, it
 * puts the query into the batch that is currently collecting and returns when the batch has been searched.  A
 * dispatcher thread submits a batch (hs_search_batch_submit, batch overlap on: small batches run side by side on
 * the GPU) as soon as it holds a query — or, if max_wait_us > 0, once it is full or its first query has waited that
 * long — and a completion thread wakes the callers batch by batch.  Up to 32 batches are between "collecting" and
 * "answered" (batches of fewer than 8 queries only while fewer than 8 are); when all are, arrivals share the next
 * buffer that frees up, so the batch size follows the load: a
 * lone query is answered at once, a busy server fills its batches (max_batch queries at most).  Batches live in
 * page-locked mapped memory and are searched in place.  A batch holds requests of ONE k (ef = max(ef_, k),
 * slim.h:2080); a request with another k goes to the next batch.  labels_out: k labels, nearest first; dists_out
 * may be NULL.  The service owns the handle's submit queue (no hs_search_batch_submit / _wait* by others meanwhile)
 * and switches hs_set_overlap on.
 *   set_ef   setEf for the batches launched from now on
 *   patch    hs_patch_apply between two batches: requests that have joined a batch are answered on the old
 *            index, later ones wait and see the patched one (the reference's patchFromStream is not synchronised
 *            with its searches at all)
 * The index is borrowed: free the service first, and only when no hs_service_query call is in progress (requests
 * that have joined a batch are still answered; later ones fail). */
typedef struct hs_service hs_service;
typedef struct {
  uint64_t batches, queries;       /* launches, and the queries they carried */
  uint64_t max_batch;              /* largest batch launched                 */
  uint64_t patches;
  double busy_seconds;             /* time the completion thread spent waiting for batches */
} hs_service_stats;
int hs_service_create(hs_index *, size_t max_batch, unsigned max_wait_us, size_t k_max, hs_service **out);
int hs_service_query(hs_service *, const float *vec, size_t k, uint32_t *labels_out, float *dists_out);
int hs_service_set_ef(hs_service *, size_t ef);
int hs_service_patch(hs_service *, const void *patch, size_t patch_bytes, unsigned flags, const float *rows,
                     const uint64_t *row_labels, size_t n_rows, hs_patch_info *info_out);
int hs_service_get_stats(hs_service *, hs_service_stats *out);
void hs_service_free(hs_service *);
/* The same batching front over a caller-supplied search function with hs_search_batch's meaning (host buffers,
 * synchronous, 0 = ok).  No CUDA needed: the CPU test-suite drives the batching logic through it. */
typedef int (*hs_service_backend_fn)(void *ctx, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                                     float *dists_out);
int hs_debug_service_create(hs_service_backend_fn fn, void *ctx, size_t dim, size_t max_batch, unsigned max_wait_us,
                            size_t k_max, hs_service **out);

/* ~HierarchicalNSWSlim / clear() (slim.h:147-167) */
void hs_free(hs_index *);

/* setEf (slim.h:193, slimq.h:346-349) */
int hs_set_ef(hs_index *, size_t ef);

int hs_get_info(const hs_index *, hs_index_info *out);

/* Batch overlap (off by default).  When on, the traversal kernel of one hs_search_batch_device
 * call is launched with programmatic stream serialization, so on ONE stream the next call's grid
 * starts filling SMs while the previous call's last queries are still draining (a batch otherwise
 * ends with a tail of about one query latency during which most of the GPU idles).  The caller
 * promises that the query buffer of a call is complete when the call is enqueued unless it was
 * produced by a non-kernel operation (copy, memset) on the same stream: a kernel of the caller
 * that writes the queries must have finished (event / stream sync) first.  Results are
 * unchanged. */
int hs_set_overlap(hs_index *, int on);

/* Tuning knobs of a handle (no reference analogue; results never depend on them, only speed — except that a
 * visited table that is reset mid-query re-evaluates nodes, so per-query counters may grow).  Every knob has an
 * environment variable that sets its initial value when the index is created:
 *   "visited_table"   HS_GHASH            where the per-warp visited set of the fp32 traversal lives: -1 automatic
 *                                         (default), 0 32-bit table in shared memory, 1 in global memory (L2),
 *                                         2 compact 16-bit table in shared memory where it applies (ef 129..256,
 *                                         96/128-dim rows, n <= 2^24), 3 automatic without the compact table
 *   "hash_bits"       HS_HASH_BITS        log2 of the 32-bit table's slots, 0 = from ef (default)
 *   "traverse_flags"  HS_TRAVERSE_FLAGS   bit 0 L2 row prefetch, bit 1 speculative next-pop adjacency load,
 *                                         bit 2 stop after the descent (profiling), bit 3 evict_last adjacency
 *                                         prefetch, bits 4 / 5 make the compact visited table reset early /
 *                                         overflow (tests), bit 6 forces the shared-memory candidate pool; default 9
 *   "slimq_flags"     HS_SLIMQ_FLAGS      hnsw_slimq kernel experiments, default 0
 *   "zero_copy"       HS_ZERO_COPY        1 (default): pinned + mapped host buffers are used in place
 * Further environment-only knobs, read where noted: HS_WPC (warps per CTA of the traversal launch, 1/2/4),
 * HS_BF_TC (0 / 1 forces the fp32-scan / tcgen05 exact-kNN path), HS_BF_QRES, HS_BF_TC_STATS (see
 * hs_debug_bf_tc_fallback), HS_SLIMQ_CARVEOUT (shared-memory carve-out of the hnsw_slimq kernel, percent),
 * HS_LIB_PATH (Python binding: an alternative build of this library). */
int hs_set_tuning(hs_index *, const char *name, long long value);

/* hnsw_slimq only.  The reference draws its query-quantiser constant at random when it loads an
 * index (slimq.h:1274-1276 -> faster_config, rabitqlib/quantization/rabitq.hpp:27-34 ->
 * rabitq_impl.hpp:363-377: std::random_device), so its estimates differ in the low bits from
 * load to load.  The engine derives the constant the same way from a FIXED seed at hs_load;
 * these read / override it (the parity tests copy the reference's value in). */
double hs_slimq_default_tconst(size_t padded_dim);   /* host only: the value hs_load picks */
int hs_get_query_tconst(const hs_index *, double *t_const);
int hs_set_query_tconst(hs_index *, double t_const);

/* hnsw_slimq only, inspection: the per-query preparation of searchKnn (slimq.h:1816-1847) as the
 * traversal kernel computes it — FhtKacRotator::rotate (rabitqlib/utils/rotator.hpp:370-423),
 * SplitSingleQuery (rabitqlib/index/query.hpp:127-156) and the centroid distances.  Host buffers:
 * rotated nq x padded_dim, planes nq x padded_dim/64*4 (plane j of word w at [w*4+j], MSB-first),
 * scal nq x 3 = (delta, vl, k1xsumq), q2c nq x num_cluster. */
int hs_slimq_prepare(hs_index *, const float *queries, size_t nq, float *rotated_out,
                     uint64_t *planes_out, float *scal_out, float *q2c_out);

/* Replaces the query loop of HnswSlimStrategy::solve / HnswSlimQStrategy::solve
 * (hnsw_slim_strategy.h:112-114, hnsw_slimq_strategy.h:157-159), i.e. nq calls of
 * searchKnn(const void*, size_t k, tableint*) (slim.h:2030-2131, slimq.h:1810-1924),
 * with HOST buffers: queries nq x dim row-major in, labels_out nq x k out
 * (external labels truncated to 32 bit as slim.h:2129).  Unlike the reference
 * (unordered k-subset, no distances) each row is sorted by (distance, id)
 * ascending and dists_out (nq x k, may be NULL) receives the distances.  Rows
 * with fewer than k reachable results are padded with 0xFFFFFFFF / +inf (the
 * reference reads uninitialised memory there).  Synchronous.  Pageable buffers are
 * copied host->device, searched, copied back.  Buffers that are page-locked and mapped
 * (cudaHostAlloc / cudaHostRegister) are used IN PLACE: the traversal kernel reads each
 * query from host memory when the warp that owns it starts (4*dim bytes) and stores each
 * result row with one coalesced write, so the PCIe/C2C transfers overlap the traversal
 * instead of bracketing it (HS_ZERO_COPY=0 in the environment forces the staged path). */
int hs_search_batch(hs_index *, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                    float *dists_out);

/* Page-lock and map a host range the caller owns (cudaHostRegister, portable + mapped) so that
 * hs_search_batch / hs_search_batch_submit use it in place; hs_unpin_host undoes it before the
 * memory is freed.  For callers that do not link the CUDA runtime themselves (the reference's
 * strategies keep queries and results in std::vector).  Registering costs about a millisecond per
 * few MB: do it once per buffer, not per call. */
int hs_pin_host(void *ptr, size_t bytes);
int hs_unpin_host(void *ptr);

/* hs_search_batch split in two so that a caller with a stream of batches (the reference's
 * server answers /query requests back to back, hnsw_slim_server.cc:69-142) keeps more than one
 * batch in flight: submit enqueues the batch on the handle's own stream and returns, wait blocks
 * until every submitted batch is complete.  Batches run in submission order; with hs_set_overlap
 * the tail of one batch overlaps the head of the next.  Buffers must stay valid and untouched
 * until hs_search_batch_wait returns.  Pinned + mapped host buffers (cudaHostAlloc /
 * cudaHostRegister) are read and written in place by the kernel; pageable buffers are staged
 * through device memory like hs_search_batch does. */
int hs_search_batch_submit(hs_index *, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                           float *dists_out);
int hs_search_batch_wait(hs_index *);
/* Blocks until the OLDEST batch that was submitted and not yet waited for is complete (batches
 * complete in submission order), so a caller can keep a fixed number of batches in flight:
 * submit, submit, { wait_oldest, consume, submit } ...  Returns at once when nothing is outstanding.  The wait
 * does not hold the handle's lock: one thread may submit while another waits (one waiting thread at a time). */
int hs_search_batch_wait_oldest(hs_index *);

/* hs_search_batch that also returns per-query counters: per_query_counts[2*i] = distances
 * evaluated for query i, [2*i+1] = nodes expanded (the per-query split of hs_stats). */
int hs_search_batch_counts(hs_index *, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                           float *dists_out, uint32_t *per_query_counts);

/* Same with DEVICE buffers (d_queries nq x dim, d_labels nq x k, d_dists nq x k or
 * NULL) on CUDA stream `stream` (a cudaStream_t, 0 = legacy default stream);
 * asynchronous, no host<->device copies.  This is what the device-resident
 * benchmark number and multi-GPU sharding use.  Thread-safe (the enqueue is serialised per handle; the call
 * selects the index's device).  One restriction: launches of ONE handle must be in flight on one stream at a
 * time — for large ef / dim the per-warp visited tables live in a global scratch area of two halves that
 * consecutive launches alternate between, which only orders correctly within a stream.  Use one handle per
 * stream (hs_load twice) to search the same index from several streams at once. */
int hs_search_batch_device(hs_index *, const float *d_queries, size_t nq, size_t k,
                           uint32_t *d_labels, float *d_dists, void *stream);

/* ---- Sharded corpora: the exchange fused into the traversal kernel ------------------------------
 * (no reference analogue; SURVEY.md §8(e).)  Instead of searching, all-gathering and merging, every
 * rank lets its traversal kernel store each result row of shard `slot` DIRECTLY into the gather
 * tables of all ranks of the box — its own memory and peer memory mapped over NVLink (CUDA IPC) —
 * so the exchange costs no collective call and no extra kernel.  A stream-ordered flag write /
 * flag wait per rank (cuStreamWriteValue32 / cuStreamWaitValue32: no SM, no copy engine) tells
 * when every rank's rows of a batch have arrived; hs_topk_merge_device then reads the local table.
 *
 * hs_search_batch_device_scatter is the kernel-level piece: hs_search_batch_device whose rows go to
 * n_dsts (<= 16) destination tables of shape [slots x nq x k] at slot `slot` (device pointers
 * valid in this process).
 *
 * hs_exchange owns the tables (double-buffered by batch parity) and the flags of one rank:
 *   create    allocates them on `device`; slots = total number of shards over all ranks
 *   handle    64-byte CUDA IPC handle of the allocation, to be all-gathered by the caller
 *   connect   maps the other ranks' allocations (handles = world x 64 bytes, rank-major)
 *   search    this rank's shard `slot` for batch `seq` (1, 2, ...), scattered to every rank
 *   signal_and_wait   after the rank's last shard of batch `seq`: announce, then hold the stream
 *             until every rank has announced `seq`
 *   tables    this rank's gathered [slots x nq x k] tables of batch `seq` for hs_topk_merge_device
 * All ranks must use the same nq and k for a given seq, and merge batch seq before searching seq+2. */
int hs_search_batch_device_scatter(hs_index *, const float *d_queries, size_t nq, size_t k,
                                   uint32_t *const *d_labels_dsts, float *const *d_dists_dsts, size_t n_dsts,
                                   size_t slot, void *stream);
typedef struct hs_exchange hs_exchange;
int hs_exchange_create(int device, int world, int rank, size_t slots, size_t nq_max, size_t k, hs_exchange **out);
int hs_exchange_handle(hs_exchange *, void *handle64);
int hs_exchange_connect(hs_exchange *, const void *handles);
int hs_exchange_search(hs_exchange *, hs_index *, const float *d_queries, size_t nq, size_t k, size_t slot,
                       unsigned int seq, void *stream);
int hs_exchange_signal_and_wait(hs_exchange *, unsigned int seq, void *stream);
int hs_exchange_tables(hs_exchange *, unsigned int seq, uint32_t **d_labels, float **d_dists);
void hs_exchange_free(hs_exchange *);

/* ---- hs_shardgroup: one rank's part of a sharded corpus, pipelined ----------------------------------
 * (no reference analogue; SURVEY.md §8(e): the reference builds ONE graph; here the base set is split into
 * per-GPU sub-graphs with global labels and every shard answers every query with the searchKnn of
 * slim.h:2030-2131 / slimq.h:1810-1924.)  A group owns the gather tables, flags and the two streams of ONE
 * rank; its local shards are hs_index handles on one device, borrowed (free the group first).  With
 * `world` ranks and n_local shards per rank the corpus has world * n_local shards; shard i of rank r is
 * slot r * n_local + i.
 *
 * hs_shardgroup_submit enqueues one batch and returns: one traversal launch per local shard (chained by
 * programmatic stream serialization — also across batches), whose kernels store every result row into
 * the tables of ALL ranks (peer memory over NVLink) and whose last finishing warp raises this rank's flag
 * on every rank; on a second, higher-priority stream a merge kernel waits for all ranks' flags of the
 * batch (cuStreamWaitValue32), writes the global top-k (by (distance, label)) of every query to
 * labels_out / dists_out and acknowledges the table slot to every rank.  No collective call, nothing
 * between two traversal launches: in a stream of batches the exchange + merge of batch s overlap the
 * searches of batch s + 1.  Up to `depth` batches may be in flight between ranks; all ranks must submit
 * the same sequence of (nq, k) shapes.  queries / labels_out / dists_out are device pointers or
 * page-locked + mapped host pointers (read / written in place); the query buffer must be complete when
 * submit is called; outputs are valid after hs_shardgroup_wait (all batches) or the matching
 * hs_shardgroup_wait_oldest.
 *   create         n_local shards of this rank, `world` ranks, this rank's index, table shape nq_max x k
 *   handle/connect one process per GPU: all-gather the 64-byte CUDA IPC handles (rank-major), then connect
 *   connect_local  one process driving all GPUs: groups[r] = rank r; enables peer access
 *   streams        the search / merge CUDA streams (to bracket a run with events) */
typedef struct hs_shardgroup hs_shardgroup;
int hs_shardgroup_create(hs_index *const *shards, size_t n_local, int world, int rank, size_t nq_max, size_t k,
                         int depth, hs_shardgroup **out);
int hs_shardgroup_handle(hs_shardgroup *, void *handle64);
int hs_shardgroup_connect(hs_shardgroup *, const void *handles);
int hs_shardgroup_connect_local(hs_shardgroup *const *groups, size_t world);
int hs_shardgroup_submit(hs_shardgroup *, const float *queries, size_t nq, uint32_t *labels_out, float *dists_out);
int hs_shardgroup_wait_oldest(hs_shardgroup *);
int hs_shardgroup_wait(hs_shardgroup *);
int hs_shardgroup_streams(hs_shardgroup *, void **search_stream, void **merge_stream);
void hs_shardgroup_free(hs_shardgroup *);

/* Counters accumulated since the last hs_reset_stats, with the meaning of
 * metric_distance_computations / metric_hops (slim.h:70-71,371-374,2064-2065):
 * n_dist = distances evaluated, n_hops = nodes expanded (upper + base layer).
 * hnsw_slimq: n_dist counts 1-bit estimates, *n_rerank exact reranks. */
int hs_stats(hs_index *, uint64_t *n_dist, uint64_t *n_hops, uint64_t *n_rerank);
int hs_reset_stats(hs_index *);

/* Replaces BruteForce::solve (brute_force_strategy.h:15-45) =
 * BruteforceSearch<float>::searchKnn per query (bruteforce.h:106-135): exact kNN of
 * nq queries over n base rows (label of row i = i).  Row order: NEAREST first,
 * ties -> smaller label (the reference writes farthest-first; reverse to compare).
 * Host buffers; dists_out may be NULL.  k > n is HS_ERR_ARG whenever nq > 0 (also for n == 0). */
int hs_bruteforce_knn(const float *base, size_t n, size_t dim, const float *queries, size_t nq,
                      size_t k, int metric, int device, uint32_t *labels_out, float *dists_out);

/* Same with device buffers, asynchronous on `stream`. */
int hs_bruteforce_knn_device(const float *d_base, size_t n, size_t dim, const float *d_queries,
                             size_t nq, size_t k, int metric, uint32_t *d_labels, float *d_dists,
                             void *stream);

/* Inspection (set HS_BF_TC_STATS=1): after hs_bruteforce_knn*, -1 if the call ran the fp32 scan
 * kernel only, else the number of queries the tcgen05 path could not certify and handed to the
 * scan kernel.  Both paths return identical results; HS_BF_TC=0 / 1 forces one or the other. */
long long hs_debug_bf_tc_fallback(void);

/* Cross-shard top-k merge for sharded corpora (no reference analogue: the
 * reference builds one graph; SURVEY.md §8(e)).  d_labels_in / d_dists_in hold
 * n_parts consecutive [nq x k] tables (e.g. the output of an NCCL all-gather);
 * writes the global top-k per query sorted by (dist, label).  Asynchronous. */
int hs_topk_merge_device(const uint32_t *d_labels_in, const float *d_dists_in, size_t n_parts,
                         size_t nq, size_t k, uint32_t *d_labels_out, float *d_dists_out,
                         void *stream);

/* SolveStrategy::recall (solve_strategy.h:67-103) on the device: recall@K of knn
 * (nq x K labels, any order) against gt (nq x gt_k ids, any order, gt_k >= K),
 * GT re-ranked by exact distance to `base` rows (ties -> smaller id). Host buffers. */
int hs_recall(const float *base, size_t n, size_t dim, const float *queries, size_t nq,
              const uint32_t *knn, size_t K, const uint32_t *gt, size_t gt_k, int metric, int device,
              double *recall_out);

/* Index construction parameters = the flags of main.cc:10-38 and the values derived
 * from them at main.cc:58-70. */
typedef struct {
  uint64_t M;                  /* --m               (HierarchicalNSW M, hnsw.h:84)            */
  uint64_t ef_construction;    /* --ef_construction                                           */
  const char *branching_factor;/* --branching_factor: "4", "16", "e", "sqrt" (hnsw.h:143-158) */
  int32_t threshold_level;     /* --threshold_level                                           */
  float top_degree_percent0;   /* --top_degree_percent0 (alpha_0)                             */
  float top_degree_percent;    /* alpha (main.cc:62 copies alpha_0)                           */
  uint64_t top_M0, low_m0, top_M, low_m;   /* M_h0, M_l0, M_h, M_l (main.cc:63-66)             */
  int32_t threads;             /* <= 0: all hardware threads                                  */
  uint64_t seed;
} hs_build_params;

/* Fills `p` with the defaults of main.cc:10-38 (M=32 there; pass your own). */
void hs_build_params_default(hs_build_params *p);

/* Host-side builder of the engine's input: HNSW construction (the omp addPoint loop of
 * hnsw_slim_strategy.h:66-69), HNSW-Slim pruning (convertFromHNSW, slim.h:867-1108) and
 * saveIndex (slim.h:717-751).  Writes a .graph that both hs_load and the reference's
 * loadIndex read.  labels may be NULL (label of row i = i).  CPU only, multi-threaded. */
int hs_build_slim_graph(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                        const uint64_t *labels, const char *out_graph_path);

/* Host-side builder of the un-pruned index of the `hnsw` strategy: the omp addPoint loop of
 * hnsw_strategy.h:24-33 and HierarchicalNSW::saveIndex (hnsw.h:748-779).  Writes a .graph that both
 * hs_load(kind = HS_KIND_HNSW) and the reference's HierarchicalNSW::loadIndex read.  Only M,
 * ef_construction, branching_factor, threads and seed of `p` are used.  CPU only, multi-threaded. */
int hs_build_hnsw_graph(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                        const uint64_t *labels, const char *out_graph_path);

/* Host-side builder of an hnsw_slimq index: the same HNSW + HNSW-Slim pruning over the raw floats
 * (the reference builds the graph with rabitqlib's HNSW, hnsw_slimq_strategy.h:100-142, then
 * convertFromHNSW, slimq.h:1471-1762), node payload = 1-bit RaBitQ code + (f_add, f_rescale,
 * f_error) against the node's cluster centroid (one_bit_code_with_factor,
 * rabitqlib/quantization/rabitq_impl.hpp:76-135) after the FHT-Kac rotation, written in
 * HierarchicalNSWSlimQ::saveIndex's format (slimq.h:1161-1216).  centroids (num_cluster x dim)
 * and cluster_ids (n) are the reference's *_centroids_16.fvecs / *_clusterids_16.ivecs inputs
 * (hnsw_slimq_strategy.h:42-45); pass NULL for both to have the builder run k-means with
 * num_cluster clusters.  The 3-bit ex-code block of each record is zero-filled: no search path
 * reads it.  L2 metric.  CPU only, multi-threaded. */
int hs_build_slimq_graph(const float *base, size_t n, size_t dim, const hs_build_params *p,
                         const float *centroids, size_t num_cluster, const uint32_t *cluster_ids,
                         const uint64_t *labels, const char *out_graph_path);

/* GPU-side index construction (SURVEY.md §8(f) rank 3): the same two steps as hs_build_slim_graph — the
 * HNSW build of hnsw_slim_strategy.h:60-82 (HierarchicalNSW::addPoint, hnsw.h:1248-1376) and
 * convertFromHNSW (slim.h:867-1108: PruneByHeuristic per node and level, reverse-edge merge, re-prune,
 * hierarchical pruning) — executed on `device` with the index staying in HBM: `base` (n x dim floats, host
 * OR device memory) is copied once into the engine's 128-byte-aligned row store and the finished index is
 * returned as an hs_index, ready for hs_search_batch*.  Points enter a layer in batches (one warp per
 * point: ef_construction beam search + neighbour selection; reverse edges through one radix sort per
 * batch), so the graph is not the one a sequential build gives; its recall/cost is measured against the
 * host builder's in tests/test_gpu_build.py.  Needs 2 <= M <= 32, ef_construction <= 256.
 * hs_save_index writes any HBM-resident hnsw_slim index in saveIndex's format (slim.h:717-751): the
 * reference's loadIndex (and hs_load) read it. */
int hs_build_slim_index_gpu(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                            const uint64_t *labels, int device, hs_index **out);
int hs_save_index(hs_index *, const char *out_graph_path);

/* The same for hnsw_slimq (HnswSlimQStrategy's build branch, hnsw_slimq_strategy.h:100-142 + convertFromHNSW,
 * slimq.h:1471-1762): the hnsw_slim graph over the raw rows is built on the device as above, then one kernel
 * gives every node its cluster id, FHT-Kac rotation (rotator.hpp:370-423), 1-bit RaBitQ code and factors
 * (one_bit_code_with_factor, rabitq_impl.hpp:76-135) — the payload of hs_build_slimq_graph, computed where the
 * rows already are.  centroids (num_cluster x dim, host) may be NULL: Lloyd iterations over a host-side sample
 * of at most 200k rows then pick them.  The raw rows stay in the index for the exact rerank (setDataset). */
int hs_build_slimq_index_gpu(const float *base, size_t n, size_t dim, const hs_build_params *p, const float *centroids,
                             size_t num_cluster, const uint64_t *labels, int device, hs_index **out);

/* Host-only inspection of the flattened form of a .graph (no CUDA needed): what
 * hs_load uploads.  Used by the CPU test-suite to check the loader against the
 * reference's accessors (slim.h:620-661). */
typedef struct hs_host_graph hs_host_graph;
int hs_debug_flatten(const char *graph_path, int kind, size_t dim, hs_host_graph **out);
void hs_debug_free(hs_host_graph *);
int hs_debug_info(const hs_host_graph *, hs_index_info *out);
int hs_debug_row(const hs_host_graph *, uint32_t node, int level, uint32_t *out, int cap);
int hs_debug_node(const hs_host_graph *, uint32_t node, int *level, uint32_t *label, float *vec_out);
/* hs_patch_apply on the host image (no CUDA needed): the parser, the validation and the upper-level re-slotting
 * are the code the device path runs; the level-0 rows and vectors are written to the host arrays instead. */
int hs_debug_patch(hs_host_graph *, const void *patch, size_t patch_bytes, unsigned flags, const float *rows,
                   const uint64_t *row_labels, size_t n_rows, hs_patch_info *info_out);
/* Phase 2 of hs_build_slim_index_gpu alone: the same device code (convertFromHNSW, slim.h:867-1108) run on the
 * un-pruned lists of an hs_build_hnsw_graph file instead of a device-built HNSW graph, so that its lists can be
 * compared one by one with hs_build_slim_graph's conversion of the same file.  Vectors, levels, labels, entry point
 * and M / maxM / maxM0 come from the file; threshold_level, top_degree_percent, top_M0, low_m0, top_M and low_m
 * from `p`.  The result is an hnsw_slim index (hs_save_index writes it).  Needs maxM0 <= 64 and pruning
 * parameters <= 64 (HS_ERR_UNSUPPORTED otherwise, as for the builder). */
int hs_debug_convert_gpu(const char *hnsw_graph_path, size_t dim, int metric, const hs_build_params *p, int device,
                         hs_index **out);
/* hnsw_slimq only, inspection: the per-node payload as the traversal kernel reads it, for an index built on the
 * device or loaded with hs_load.  records: n x (padded_dim/64 + 2) 8-byte words, per node the code words (bit
 * 63 - j of word w = sign of dimension 64w + j, the file's MSB-first order), then (f_add, f_rescale) as two floats,
 * then (cluster id, 0) as two uint32; rotated_centroids: num_cluster x padded_dim; flip: 4 * padded_dim / 8
 * rotator sign bytes.  Any output may be NULL. */
int hs_debug_slimq_payload(const hs_index *, uint64_t *records, float *rotated_centroids, uint8_t *flip);

const char *hs_last_error(void);
int hs_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HNSWSLIM_B200_H */
