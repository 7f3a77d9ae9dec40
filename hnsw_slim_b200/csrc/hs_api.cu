// C ABI of libhnswslim_b200.so (include/hnswslim_b200.h): index lifetime, batched search.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "bruteforce.cuh"
#include "hs_index.h"

namespace hs {
static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
}  // namespace hs

using namespace hs;

#define HS_CUDA(call)                                                                 \
  do {                                                                                \
    cudaError_t e__ = (call);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      set_error(std::string(#call) + ": " + cudaGetErrorString(e__));                 \
      return HS_ERR_CUDA;                                                             \
    }                                                                                 \
  } while (0)

namespace {
// C++ exceptions must not unwind through the C ABI: file-derived sizes feed std::vector allocations
// (a corrupt header, or a 100M-row shard on a small host, ends in bad_alloc / length_error)
template <typename F>
int guarded(const char *what, F &&body) {
  try {
    return body();
  } catch (const std::bad_alloc &) {
    set_error(std::string(what) + ": out of host memory");
    return HS_ERR_NOMEM;
  } catch (const std::length_error &) {
    set_error(std::string(what) + ": size field out of range (corrupt header?)");
    return HS_ERR_IO;
  } catch (const std::exception &e) {
    set_error(std::string(what) + ": " + e.what());
    return HS_ERR_IO;
  }
}
}  // namespace

namespace hs {
int select_device(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
              "); hnswslim_b200 has no CPU fallback");
    return HS_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    set_error("device ordinal out of range");
    return HS_ERR_ARG;
  }
  HS_CUDA(cudaSetDevice(device));
  return HS_OK;
}

// Device-visible alias of a host buffer when the whole range [p, p + bytes) is page-locked
// (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory) and mapped into this device's address
// space; nullptr otherwise (pageable memory, or pinned without mapping).
void *mapped_alias(const void *p, size_t bytes) {
  if (!p || bytes == 0) return nullptr;
  cudaPointerAttributes a0{}, a1{};
  if (cudaPointerGetAttributes(&a0, p) != cudaSuccess ||
      cudaPointerGetAttributes(&a1, static_cast<const char *>(p) + bytes - 1) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (a0.type != cudaMemoryTypeHost || a1.type != cudaMemoryTypeHost || !a0.devicePointer || !a1.devicePointer)
    return nullptr;
  if (static_cast<char *>(a1.devicePointer) - static_cast<char *>(a0.devicePointer) != (ptrdiff_t)(bytes - 1))
    return nullptr;
  return a0.devicePointer;
}

}  // namespace hs

namespace {

template <typename T>
int upload(T **dst, const T *src, size_t count, size_t *bytes_total) {
  *dst = nullptr;
  if (count == 0) return HS_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void **>(dst), count * sizeof(T));
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc(") + std::to_string(count * sizeof(T)) + "): " + cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? HS_ERR_NOMEM : HS_ERR_CUDA;
  }
  e = cudaMemcpy(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error(std::string("cudaMemcpy H2D: ") + cudaGetErrorString(e));
    return HS_ERR_CUDA;
  }
  *bytes_total += count * sizeof(T);
  return HS_OK;
}

// upload into an allocation of cap_count (>= count) elements whose tail is filled with `fill` bytes
template <typename T>
int upload_cap(T **dst, const T *src, size_t count, size_t cap_count, int fill, size_t *bytes_total) {
  *dst = nullptr;
  if (cap_count < count) cap_count = count;
  if (cap_count == 0) return HS_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void **>(dst), cap_count * sizeof(T));
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc(") + std::to_string(cap_count * sizeof(T)) + "): " + cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? HS_ERR_NOMEM : HS_ERR_CUDA;
  }
  if (count) e = cudaMemcpy(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && cap_count > count) e = cudaMemset(*dst + count, fill, (cap_count - count) * sizeof(T));
  if (e != cudaSuccess) {
    set_error(std::string("cudaMemcpy H2D: ") + cudaGetErrorString(e));
    return HS_ERR_CUDA;
  }
  *bytes_total += cap_count * sizeof(T);
  return HS_OK;
}

// per-handle scratch, knobs and the handle's own stream (both construction paths end here)
int init_scratch(hs_index *ix) {
  cudaDeviceProp prop;
  HS_CUDA(cudaGetDeviceProperties(&prop, ix->device));
  ix->sm_count = prop.multiProcessorCount;
  if (const char *hb = std::getenv("HS_HASH_BITS")) ix->hash_bits_override = std::atoi(hb);
  if (const char *gh = std::getenv("HS_GHASH")) ix->ghash_mode = std::atoi(gh);
  if (const char *tf = std::getenv("HS_TRAVERSE_FLAGS")) ix->traverse_flags = (uint32_t)std::atoi(tf);
  if (const char *qf = std::getenv("HS_SLIMQ_FLAGS")) ix->slimq_flags = (uint32_t)std::atoi(qf);
  if (const char *zc = std::getenv("HS_ZERO_COPY")) ix->zero_copy = std::atoi(zc) != 0;
  if (cudaMalloc(&ix->d_work, kWorkRing * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(ix->d_work, 0xff, kWorkRing * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMalloc(&ix->d_stats, 4 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(ix->d_stats, 0, 4 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_error(std::string("scratch allocation: ") + cudaGetErrorString(cudaGetLastError()));
    return HS_ERR_CUDA;
  }
  return HS_OK;
}

// capacity > 0: room for `capacity` nodes (hs_load_reserve); rows past n read as "no neighbours" / zero vectors
int build_index(const HostGraph &g, int metric, int device, const float *raw_base, hs_index **out, size_t capacity = 0) {
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  std::unique_ptr<hs_index> ix(new hs_index);
  ix->device = device;
  const size_t cap = std::max<size_t>(capacity, g.n);
  ix->capacity = cap;
  size_t bytes = 0;
  auto fail = [&](int code) {
    hs_free(ix.release());
    return code;
  };
  if (g.kind == HS_KIND_SLIMQ) {
    // raw rows for the exact rerank (slimq.h:747-749), padded like the hnsw_slim vector store
    std::vector<float> vec(g.n * g.dim_padded, 0.f);
    for (size_t i = 0; i < g.n; ++i) std::memcpy(&vec[i * g.dim_padded], raw_base + i * g.dim, 4 * g.dim);
    if ((rc = upload(&ix->d_vec, vec.data(), vec.size(), &bytes)) != HS_OK) return fail(rc);
    // one record per node: [u64 code[words]][f_add, f_rescale][cluster, 0]; 32 bytes for padded_dim 128
    const size_t words = g.padded_dim_q / 64, rw = words + 2;
    std::vector<uint2> rec(g.n * rw);
    for (size_t i = 0; i < g.n; ++i) {
      uint2 *r = &rec[i * rw];
      for (size_t w = 0; w < words; ++w) {
        const uint64_t c = g.bin_code[i * words + w];
        r[w] = make_uint2((uint32_t)c, (uint32_t)(c >> 32));
      }
      uint32_t fa, fr;
      std::memcpy(&fa, &g.f_add[i], 4);
      std::memcpy(&fr, &g.f_rescale[i], 4);
      r[words] = make_uint2(fa, fr);
      r[words + 1] = make_uint2(g.cluster_id[i], 0u);
    }
    if ((rc = upload(&ix->d_qrec, rec.data(), rec.size(), &bytes)) != HS_OK) return fail(rc);
    if ((rc = upload(&ix->d_centroids, g.centroids.data(), g.centroids.size(), &bytes)) != HS_OK) return fail(rc);
    if ((rc = upload(&ix->d_flip, g.rotator_flip.data(), g.rotator_flip.size(), &bytes)) != HS_OK) return fail(rc);
    ix->words = (uint32_t)words;
    uint32_t td = 1;                                    // rotator.hpp:233-235
    while ((size_t)td * 2 <= g.dim) td *= 2;
    ix->trunc_dim = td;
    ix->t_const = slimq_default_tconst(g.padded_dim_q, 3);   // kNumBits = 4 (query.hpp:126)
  } else {
    if ((rc = upload_cap(&ix->d_vec, g.vec.data(), g.vec.size(), cap * g.dim_padded, 0, &bytes)) != HS_OK) return fail(rc);
  }
  if ((rc = upload_cap(&ix->d_adj0, g.adj0.data(), g.adj0.size(), cap * g.deg0_stride, 0xff, &bytes)) != HS_OK) return fail(rc);
  if ((rc = upload_cap(&ix->d_upper_slot, g.upper_slot.data(), g.upper_slot.size(), cap, 0xff, &bytes)) != HS_OK) return fail(rc);
  if ((rc = upload_cap(&ix->d_labels, g.labels.data(), g.labels.size(), cap, 0, &bytes)) != HS_OK) return fail(rc);
  if ((rc = upload_cap(&ix->d_deleted, g.deleted.data(), g.deleted.size(), cap, 0, &bytes)) != HS_OK) return fail(rc);
  for (int l = 1; l < (int)g.upper_adj.size() && l < kMaxLevels; ++l) {
    if ((rc = upload(&ix->d_upper_adj[l], g.upper_adj[l].data(), g.upper_adj[l].size(), &bytes)) != HS_OK)
      return fail(rc);
    ix->cap_upper_words[l] = g.upper_adj[l].size();
  }
  if ((rc = init_scratch(ix.get())) != HS_OK) return fail(rc);

  for (int l = 0; l < (int)g.level_count.size() && l < kMaxLevels; ++l) ix->level_count[l] = g.level_count[l];
  hs_index_info &I = ix->info;
  I.n = g.n;
  I.dim = g.dim;
  I.dim_padded = g.dim_padded;
  I.M = g.M;
  I.maxM = g.maxM;
  I.maxM0 = g.maxM0;
  I.ef_construction = g.ef_construction;
  I.maxlevel = g.maxlevel;
  I.threshold_level = g.threshold_level;
  I.enterpoint = g.enterpoint;
  I.has_deleted = g.has_deleted ? 1 : 0;
  I.kind = g.kind;
  I.metric = metric;
  I.deg0_stride = g.deg0_stride;
  I.max_deg0 = g.max_deg0;
  I.upper_stride = g.upper_stride;
  I.n_upper = g.n_upper;
  I.sum_deg0 = g.sum_deg0;
  I.device_bytes = bytes;
  I.ef = 10;   // ef_ = 10 after loadIndex (slim.h:794)
  I.padded_dim_q = g.padded_dim_q;
  I.num_cluster = g.num_cluster;
  *out = ix.release();
  return HS_OK;
}

int load_common(const uint8_t *bytes, size_t size, int kind, int metric, size_t dim, const float *raw_base,
                size_t n_raw, int device, hs_index **out, size_t capacity = 0) {
  if (!out || !bytes) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  if (metric != HS_METRIC_L2 && metric != HS_METRIC_IP) {
    set_error("unknown metric");
    return HS_ERR_ARG;
  }
  if (dim == 0) {
    set_error("dim must be > 0");
    return HS_ERR_ARG;
  }
  if (kind == HS_KIND_SLIMQ && metric != HS_METRIC_L2) {
    // every strategy of the reference builds hnsw_slimq with METRIC_L2 (hnsw_slimq_strategy.h:68)
    set_error("hnsw_slimq: only the L2 metric is supported");
    return HS_ERR_UNSUPPORTED;
  }
  HostGraph g;
  g.reserve_strides = capacity > 0;
  int rc = parse_graph(bytes, size, kind, dim, &g);
  if (rc != HS_OK) return rc;
  if (capacity > 0) {
    if (capacity < g.n) {
      set_error("max_elements is below the element count of the .graph");     // loadIndex, slim.h:759-761
      return HS_ERR_ARG;
    }
    if (capacity >= (1ull << 31)) {
      set_error("max_elements >= 2^31");
      return HS_ERR_UNSUPPORTED;
    }
  }
  if (kind == HS_KIND_SLIMQ) {
    if (!raw_base || n_raw < g.n) {
      set_error("hnsw_slimq needs raw_base with at least n rows for the exact rerank (setDataset, slimq.h:303-305)");
      return HS_ERR_ARG;
    }
    if (g.metric_type_q != 0 /* rabitqlib::METRIC_L2 */) {
      set_error("hnsw_slimq index was built with a non-L2 metric: not supported");
      return HS_ERR_UNSUPPORTED;
    }
    if (g.padded_dim_q > 2048 || g.num_cluster == 0 || g.num_cluster > 4096) {
      set_error("hnsw_slimq: padded_dim > 2048 or cluster count out of range");
      return HS_ERR_UNSUPPORTED;
    }
  }
  if (g.threshold_level < 0) {
    set_error("negative threshold_level in .graph header");
    return HS_ERR_IO;
  }
  if (g.has_deleted) {
    // has_deleted_elements_ switches the reference to searchBaseLayerST<false> (slim.h:2114-2123),
    // whose stop rule adds `&& top_size == ef` (:346-347) and which keeps delete-marked nodes out
    // of the result heap (:418).  While the pool is not full every scored neighbour is admitted, so
    // the closest candidate is never beyond lowerBound and the extra clause changes nothing: an
    // index that only carries the flag is searched exactly like one without it.  Nodes that are
    // actually marked (convertFromHNSW never writes the mark, slim.h:1088-1089) are not supported.
    bool any_marked = false;
    for (uint8_t d : g.deleted) any_marked |= d != 0;
    if (any_marked || kind == HS_KIND_HNSW) {
      set_error("index contains delete-marked elements (slim.h:1776-1781 / hnsw.h:1007-1018): not supported");
      return HS_ERR_UNSUPPORTED;
    }
  }
  rc = build_index(g, metric, device, raw_base, out, capacity);
  if (rc == HS_OK && kind == HS_KIND_SLIMQ) {
    // kept on the host for hs_save_index: the traversal does not read them
    (*out)->f_error = std::move(g.f_error);
    (*out)->ex_bits = g.ex_bits;
    (*out)->size_ex = g.size_data_per_element - 28 - (g.padded_dim_q / 8 + 12);   // checked by parse_graph
  }
  if (rc == HS_OK && capacity > 0) {
    // the mirror of a patchable index: everything but the arrays that only the device needs
    g.mirror_only = true;
    std::vector<float>().swap(g.vec);
    std::vector<uint32_t>().swap(g.adj0);
    (*out)->mirror.reset(new HostGraph(std::move(g)));
  }
  return rc;
}

int ensure(void **p, size_t *cap, size_t need) {
  if (need <= *cap) return HS_OK;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  cudaError_t e = cudaMalloc(p, need);
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc scratch: ") + cudaGetErrorString(e));
    return HS_ERR_NOMEM;
  }
  *cap = need;
  return HS_OK;
}

struct PrepDump {
  float *rotated;
  unsigned long long *planes;
  float *scal, *q2c;
};

int search_device_slimq(hs_index *ix, const float *d_queries, size_t nq, size_t k, uint32_t *d_labels,
                        float *d_dists, uint32_t *d_perq, cudaStream_t stream, const PrepDump *dump,
                        const ScatterDst *scatter = nullptr, uint32_t *plan_warps = nullptr) {
  TraverseQParams p{};
  p.qrec = ix->d_qrec;
  p.vec = reinterpret_cast<const float4 *>(ix->d_vec);
  p.adj0 = ix->d_adj0;
  p.upper_slot = ix->d_upper_slot;
  for (int l = 0; l < kMaxLevels; ++l) p.upper_adj[l] = ix->d_upper_adj[l];
  p.labels = ix->d_labels;
  p.centroids = ix->d_centroids;
  p.flip = ix->d_flip;
  p.n = (uint32_t)ix->info.n;
  p.row_chunks = (uint32_t)(ix->info.dim_padded / 4);
  p.deg0_stride = ix->info.deg0_stride;
  p.upper_stride = ix->info.upper_stride;
  p.enterpoint = ix->info.enterpoint;
  p.maxlevel = ix->info.maxlevel;
  p.threshold_level = ix->info.threshold_level;
  p.padded_dim = (uint32_t)ix->info.padded_dim_q;
  p.trunc_dim = ix->trunc_dim;
  p.num_cluster = (uint32_t)ix->info.num_cluster;
  p.words = ix->words;
  p.rec_words = ix->words + 2;
  p.fht_fac = 1.0f / std::sqrt((float)ix->trunc_dim);   // rotator.hpp:235
  p.t_const = ix->t_const;
  p.queries = d_queries;
  p.nq = (uint32_t)nq;
  p.dim = (uint32_t)ix->info.dim;
  p.k = (uint32_t)k;
  p.ef = (uint32_t)ix->info.ef;       // pool capacity = ef_ (setEf, slimq.h:346-349), not max(ef, k)
  p.out_labels = d_labels;
  p.out_dists = d_dists;
  if (scatter) p.scatter = *scatter;
  if (dump) {
    p.prep_rotated = dump->rotated;
    p.prep_planes = dump->planes;
    p.prep_scal = dump->scal;
    p.prep_q2c = dump->q2c;
  }
  p.overlap = ix->overlap ? 1u : 0u;
  p.stats = ix->d_stats;
  p.per_query = d_perq;
  p.flags = ix->slimq_flags;
  TraverseQLaunch l{};
  if (ix->planq_ok && ix->planq_ef == p.ef && ix->planq_nq == nq && ix->planq_k == k) {
    l = ix->planq_l;
    p.smem_per_warp = ix->planq_p.smem_per_warp;
    p.off_buf = ix->planq_p.off_buf;
    p.off_g2c = ix->planq_p.off_g2c;
    p.off_planes = ix->planq_p.off_planes;
    p.off_topk = ix->planq_p.off_topk;
  } else {
    int rc = plan_traverse_slimq(p, ix->sm_count, (int)nq, &l);
    if (rc != HS_OK) return rc;
    ix->planq_ok = true;
    ix->planq_ef = p.ef;
    ix->planq_nq = nq;
    ix->planq_k = k;
    ix->planq_l = l;
    ix->planq_p = p;
  }
  if (plan_warps) {
    *plan_warps = (uint32_t)(l.grid * l.warps_per_cta);
    return HS_OK;
  }
  const unsigned int seq = ix->launch_seq++;
  p.work_counter = ix->d_work + (seq % kWorkRing);
  p.launch_tag = seq;
  return launch_traverse_slimq(p, l, stream);
}

}  // namespace

int hs::adopt_device_graph(DeviceGraph &dg, int device, hs_index **out) {
  std::unique_ptr<hs_index> ix(new hs_index);
  ix->device = device;
  ix->d_vec = dg.d_vec;
  ix->d_adj0 = dg.d_adj0;
  ix->d_upper_slot = dg.d_upper_slot;
  for (int l = 0; l < kMaxLevels; ++l) ix->d_upper_adj[l] = dg.d_upper_adj[l];
  ix->d_qrec = dg.d_qrec;
  ix->d_centroids = dg.d_centroids;
  ix->d_flip = dg.d_flip;
  dg.d_qrec = nullptr;
  dg.d_centroids = nullptr;
  dg.d_flip = nullptr;
  dg.d_vec = nullptr;                     // owned by the handle from here on (hs_free releases them)
  dg.d_adj0 = nullptr;
  dg.d_upper_slot = nullptr;
  for (auto &p : dg.d_upper_adj) p = nullptr;
  auto fail = [&](int code) {
    hs_free(ix.release());
    return code;
  };
  int rc = select_device(device);
  if (rc != HS_OK) return fail(rc);
  size_t bytes = dg.n * dg.dim_padded * 4 + dg.n * (size_t)dg.deg0_stride * 4 + dg.n * 4;
  for (int l = 1; l <= dg.maxlevel && l < kMaxLevels; ++l) bytes += (size_t)dg.level_count[l] * dg.upper_stride * 4;
  if ((rc = upload(&ix->d_labels, dg.h_labels, dg.n, &bytes)) != HS_OK) return fail(rc);
  if (cudaMalloc(&ix->d_deleted, dg.n) != cudaSuccess || cudaMemset(ix->d_deleted, 0, dg.n) != cudaSuccess) {
    set_error("cudaMalloc (deleted flags) failed");
    cudaGetLastError();
    return fail(HS_ERR_NOMEM);
  }
  bytes += dg.n;
  if ((rc = init_scratch(ix.get())) != HS_OK) return fail(rc);
  for (int l = 0; l <= dg.maxlevel && l < kMaxLevels; ++l) ix->level_count[l] = dg.level_count[l];
  hs_index_info &I = ix->info;
  I.n = dg.n;
  I.dim = dg.dim;
  I.dim_padded = dg.dim_padded;
  I.M = dg.M;
  I.maxM = dg.maxM;
  I.maxM0 = dg.maxM0;
  I.ef_construction = dg.ef_construction;
  I.maxlevel = dg.maxlevel;
  I.threshold_level = dg.threshold_level;
  I.enterpoint = dg.enterpoint;
  I.has_deleted = 0;
  I.kind = dg.kind;
  I.metric = dg.metric;
  I.deg0_stride = dg.deg0_stride;
  I.max_deg0 = dg.max_deg0;
  I.upper_stride = dg.upper_stride;
  I.n_upper = dg.n_upper;
  I.sum_deg0 = dg.sum_deg0;
  if (dg.kind == HS_KIND_SLIMQ) {
    ix->words = (uint32_t)(dg.padded_dim_q / 64);
    ix->trunc_dim = dg.trunc_dim;
    ix->t_const = slimq_default_tconst(dg.padded_dim_q, 3);
    ix->f_error = std::move(dg.h_f_error);
    ix->ex_bits = 3;                                    // as build_slimq_graph (data_layout.hpp)
    ix->size_ex = dg.padded_dim_q * 3 / 8 + 8;
    I.padded_dim_q = dg.padded_dim_q;
    I.num_cluster = dg.num_cluster;
    bytes += dg.n * (dg.padded_dim_q / 64 + 2) * 8 + dg.num_cluster * dg.padded_dim_q * 4 + 4 * dg.padded_dim_q / 8;
  }
  I.device_bytes = bytes;
  I.ef = 10;
  *out = ix.release();
  return HS_OK;
}

int hs::search_device(hs_index *ix, const float *d_queries, size_t nq, size_t k, uint32_t *d_labels,
                      float *d_dists, uint32_t *d_perq, cudaStream_t stream, const ScatterDst *scatter,
                      uint32_t *plan_warps) {
  if (!ix || (!d_queries && nq) || (!d_labels && nq && !(scatter && scatter->n)) || k == 0) {
    set_error("null argument / k == 0");
    return HS_ERR_ARG;
  }
  if (plan_warps) *plan_warps = 0;
  if (nq == 0 || ix->info.n == 0) return HS_OK;    // slim.h:2031-2032
  if (nq > 0x7fffffffu || k > 4096) {
    set_error("nq or k too large");
    return HS_ERR_ARG;
  }
  if (ix->info.kind == HS_KIND_SLIMQ)
    return search_device_slimq(ix, d_queries, nq, k, d_labels, d_dists, d_perq, stream, nullptr, scatter, plan_warps);
  TraverseParams p{};
  p.vec = reinterpret_cast<const float4 *>(ix->d_vec);
  p.adj0 = ix->d_adj0;
  p.upper_slot = ix->d_upper_slot;
  for (int l = 0; l < kMaxLevels; ++l) p.upper_adj[l] = ix->d_upper_adj[l];
  p.labels = ix->d_labels;
  p.deleted = ix->d_deleted;
  for (int l = 0; l < kMaxLevels; ++l) p.level_count[l] = ix->level_count[l];
  p.n = (uint32_t)ix->info.n;
  p.row_chunks = (uint32_t)(ix->info.dim_padded / 4);
  p.deg0_stride = ix->info.deg0_stride;
  p.upper_stride = ix->info.upper_stride;
  p.enterpoint = ix->info.enterpoint;
  p.maxlevel = ix->info.maxlevel;
  p.threshold_level = ix->info.threshold_level;
  p.has_deleted = ix->info.has_deleted;
  p.queries = d_queries;
  p.nq = (uint32_t)nq;
  p.dim = (uint32_t)ix->info.dim;
  p.k = (uint32_t)k;
  p.ef = (uint32_t)std::max<size_t>(ix->info.ef, k);   // slim.h:2080
  p.out_labels = d_labels;
  p.out_dists = d_dists;
  if (scatter) p.scatter = *scatter;
  p.overlap = ix->overlap ? 1u : 0u;
  p.stats = ix->d_stats;
  p.per_query = d_perq;
  p.flags = ix->traverse_flags;
  TraverseLaunch l{};
  int rc = HS_OK;
  if (ix->plan_ok && ix->plan_ef == p.ef) {   // same index, ef and knobs as the last call: reuse its plan
    l = ix->plan_l;
    p.hash_bits = ix->plan_p.hash_bits;
    p.smem_per_warp = ix->plan_p.smem_per_warp;
    p.off_hash = ix->plan_p.off_hash;
    p.off_stage = ix->plan_p.off_stage;
    p.off_query = ix->plan_p.off_query;
    if (ix->plan_nq != nq) resize_traverse_launch(p, (int)nq, &l);      // only the grid depends on the batch size
  } else {
    rc = plan_traverse(p, ix->info.metric, ix->hash_bits_override, ix->ghash_mode, ix->sm_count, (int)nq, &l);
    if (rc != HS_OK) return rc;
    ix->plan_ok = true;
    ix->plan_ef = p.ef;
    ix->plan_nq = nq;
    ix->plan_l = l;
    ix->plan_p = p;
  }
  if (plan_warps) {
    *plan_warps = (uint32_t)(l.grid * l.warps_per_cta);
    return HS_OK;
  }
  const unsigned int seq = ix->launch_seq++;
  p.work_counter = ix->d_work + (seq % kWorkRing);
  p.launch_tag = seq;
  if (l.ghash) {
    if ((rc = ensure((void **)&ix->d_ghash, &ix->cap_ghash, 2 * l.ghash_bytes)) != HS_OK) return rc;
    p.ghash = ix->d_ghash + (seq & 1u) * (l.ghash_bytes / 4);
  }
  if (!l.may_overlap) p.overlap = 0;
  return launch_traverse(p, ix->info.metric, l, stream);
}

namespace {

int search_host(hs_index *ix, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                float *dists_out, uint32_t *perq_out, bool sync = true) {
  if (!ix || (!queries && nq) || (!labels_out && nq)) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  if (nq == 0 || ix->info.n == 0) return HS_OK;
  std::lock_guard<std::mutex> lock(ix->mu);
  HS_CUDA(cudaSetDevice(ix->device));
  const size_t dim = ix->info.dim;
  int rc;
  // Zero-copy: when the caller's buffers are pinned and mapped, the traversal kernel reads every
  // query straight from host memory (one 4*dim-byte read per query, issued by the warp that owns
  // the query and hidden behind the other warps' work) and writes the k results of a query back in
  // one coalesced store — no staging copies, no copy->kernel->copy serialisation: the host<->device
  // transfers overlap the traversal itself.  HS_ZERO_COPY=0 forces the staged path.
  if (ix->zero_copy) {
    const float *zq = static_cast<const float *>(mapped_alias(queries, nq * dim * sizeof(float)));
    uint32_t *zl = static_cast<uint32_t *>(mapped_alias(labels_out, nq * k * 4));
    float *zd = dists_out ? static_cast<float *>(mapped_alias(dists_out, nq * k * 4)) : nullptr;
    uint32_t *zp = perq_out ? static_cast<uint32_t *>(mapped_alias(perq_out, nq * 8)) : nullptr;
    if (zq && zl && (!dists_out || zd) && (!perq_out || zp)) {
      rc = search_device(ix, zq, nq, k, zl, zd, zp, ix->stream);
      if (rc != HS_OK) return rc;
      if (sync) HS_CUDA(cudaStreamSynchronize(ix->stream));
      return HS_OK;
    }
  }
  if ((rc = ensure((void **)&ix->d_q, &ix->cap_q, nq * dim * sizeof(float))) != HS_OK) return rc;
  size_t cap_lab = ix->cap_out, cap_dist = ix->cap_out;
  if ((rc = ensure((void **)&ix->d_lab, &cap_lab, nq * k * 4)) != HS_OK) return rc;
  if ((rc = ensure((void **)&ix->d_dist, &cap_dist, nq * k * 4)) != HS_OK) return rc;
  ix->cap_out = std::min(cap_lab, cap_dist);
  if (perq_out && (rc = ensure((void **)&ix->d_perq, &ix->cap_perq, nq * 8)) != HS_OK) return rc;
  HS_CUDA(cudaMemcpyAsync(ix->d_q, queries, nq * dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
  // the counters variant is a diagnostic entry point: poison its scratch so that a query the kernel
  // never answered shows up as 0xFFFFFFFF counters instead of whatever an earlier call left there
  if (perq_out) HS_CUDA(cudaMemsetAsync(ix->d_perq, 0xff, nq * 8, ix->stream));
  rc = search_device(ix, ix->d_q, nq, k, ix->d_lab, ix->d_dist, perq_out ? ix->d_perq : nullptr, ix->stream);
  if (rc != HS_OK) return rc;
  HS_CUDA(cudaMemcpyAsync(labels_out, ix->d_lab, nq * k * 4, cudaMemcpyDeviceToHost, ix->stream));
  if (dists_out)
    HS_CUDA(cudaMemcpyAsync(dists_out, ix->d_dist, nq * k * 4, cudaMemcpyDeviceToHost, ix->stream));
  if (perq_out) HS_CUDA(cudaMemcpyAsync(perq_out, ix->d_perq, nq * 8, cudaMemcpyDeviceToHost, ix->stream));
  if (sync) HS_CUDA(cudaStreamSynchronize(ix->stream));
  return HS_OK;
}

}  // namespace

extern "C" {

const char *hs_last_error(void) { return g_error.c_str(); }
int hs_abi_version(void) { return HS_ABI_VERSION; }

int hs_load_memory(const void *graph_bytes, size_t graph_size, int kind, int metric, size_t dim,
                   const float *raw_base, size_t n_raw, int device, hs_index **out) {
  return guarded("hs_load_memory", [&] {
    return load_common(static_cast<const uint8_t *>(graph_bytes), graph_size, kind, metric, dim, raw_base, n_raw,
                       device, out);
  });
}

int hs_load(const char *graph_path, int kind, int metric, size_t dim, const float *raw_base, size_t n_raw,
            int device, hs_index **out) {
  if (!graph_path || !out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  return guarded("hs_load", [&] {
    std::vector<uint8_t> bytes;
    int rc = read_file(graph_path, &bytes);
    if (rc != HS_OK) return rc;
    return load_common(bytes.data(), bytes.size(), kind, metric, dim, raw_base, n_raw, device, out);
  });
}

int hs_load_reserve(const char *graph_path, int kind, int metric, size_t dim, size_t max_elements, int device,
                    hs_index **out) {
  if (!graph_path || !out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  if (kind != HS_KIND_SLIM) {
    set_error("hs_load_reserve: delta patches exist for hnsw_slim indices only (patchFromStream, slim.h:2206-2388)");
    return HS_ERR_UNSUPPORTED;
  }
  if (max_elements == 0) {
    set_error("hs_load_reserve: max_elements must be > 0");
    return HS_ERR_ARG;
  }
  return guarded("hs_load_reserve", [&] {
    std::vector<uint8_t> bytes;
    int rc = read_file(graph_path, &bytes);
    if (rc != HS_OK) return rc;
    return load_common(bytes.data(), bytes.size(), kind, metric, dim, nullptr, 0, device, out, max_elements);
  });
}

int hs_patch_apply(hs_index *ix, const void *patch, size_t patch_bytes, unsigned flags, const float *rows,
                   const uint64_t *row_labels, size_t n_rows, hs_patch_info *info_out) {
  if (!ix || !patch) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  if (!ix->mirror) {
    set_error("hs_patch_apply: the index was not loaded with hs_load_reserve");
    return HS_ERR_UNSUPPORTED;
  }
  return guarded("hs_patch_apply", [&]() -> int {
    std::lock_guard<std::mutex> lock(ix->mu);
    HS_CUDA(cudaSetDevice(ix->device));
    HS_CUDA(cudaStreamSynchronize(ix->stream));        // batches handed to hs_search_batch_submit
    PatchSet ps;
    int rc = parse_patch(static_cast<const uint8_t *>(patch), patch_bytes, ix->info.dim, (flags & HS_PATCH_INLINE_ROWS) != 0,
                         ix->info.n, ix->capacity, &ps);
    if (rc != HS_OK) return rc;
    PatchRows pr;
    pr.rows = rows;
    pr.row_labels = row_labels;
    pr.n_rows = n_rows;
    pr.dim = ix->info.dim;
    pr.prepare();
    return apply_patch_device(ix, ps, pr, info_out);
  });
}

void hs_free(hs_index *ix) {
  if (!ix) return;
  cudaSetDevice(ix->device);
  cudaFree(ix->d_vec);
  cudaFree(ix->d_adj0);
  cudaFree(ix->d_upper_slot);
  for (auto *p : ix->d_upper_adj) cudaFree(p);
  cudaFree(ix->d_labels);
  cudaFree(ix->d_deleted);
  cudaFree(ix->d_qrec);
  cudaFree(ix->d_centroids);
  cudaFree(ix->d_flip);
  cudaFree(ix->d_work);
  cudaFree(ix->d_stats);
  cudaFree(ix->d_q);
  cudaFree(ix->d_lab);
  cudaFree(ix->d_dist);
  cudaFree(ix->d_perq);
  cudaFree(ix->d_ghash);
  for (auto &ev : ix->ev_ring)
    if (ev) cudaEventDestroy(ev);
  if (ix->stream) cudaStreamDestroy(ix->stream);
  delete ix;
}

int hs_set_ef(hs_index *ix, size_t ef) {
  if (!ix || ef == 0 || ef > 4096) {
    set_error("hs_set_ef: ef must be in [1, 4096]");
    return HS_ERR_ARG;
  }
  ix->info.ef = ef;
  return HS_OK;
}

int hs_set_tuning(hs_index *ix, const char *name, long long value) {
  if (!ix || !name) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  const std::string n(name);
  std::lock_guard<std::mutex> lock(ix->mu);
  if (n == "visited_table") {
    if (value < -1 || value > 3) {
      set_error("hs_set_tuning: visited_table takes -1 .. 3");
      return HS_ERR_ARG;
    }
    ix->ghash_mode = (int)value;
  } else if (n == "hash_bits") {
    if (value < 0 || value > 16) {
      set_error("hs_set_tuning: hash_bits takes 0 (automatic) .. 16");
      return HS_ERR_ARG;
    }
    ix->hash_bits_override = (int)value;
  } else if (n == "traverse_flags") {
    ix->traverse_flags = (uint32_t)value;
  } else if (n == "slimq_flags") {
    ix->slimq_flags = (uint32_t)value;
  } else if (n == "zero_copy") {
    ix->zero_copy = value != 0;
  } else {
    set_error("hs_set_tuning: unknown knob '" + n + "'");
    return HS_ERR_ARG;
  }
  ix->plan_ok = false;          // launch plans depend on the knobs
  ix->planq_ok = false;
  return HS_OK;
}

int hs_set_overlap(hs_index *ix, int on) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  ix->overlap = on ? 1 : 0;
  return HS_OK;
}

int hs_set_query_tconst(hs_index *ix, double t_const) {
  if (!ix || ix->info.kind != HS_KIND_SLIMQ || !(t_const > 0.0)) {
    set_error("hs_set_query_tconst: hnsw_slimq index and t_const > 0 required");
    return HS_ERR_ARG;
  }
  ix->t_const = t_const;
  return HS_OK;
}

double hs_slimq_default_tconst(size_t padded_dim) { return slimq_default_tconst(padded_dim, 3); }

int hs_get_query_tconst(const hs_index *ix, double *t_const) {
  if (!ix || !t_const || ix->info.kind != HS_KIND_SLIMQ) {
    set_error("hs_get_query_tconst: hnsw_slimq index required");
    return HS_ERR_ARG;
  }
  *t_const = ix->t_const;
  return HS_OK;
}

int hs_slimq_prepare(hs_index *ix, const float *queries, size_t nq, float *rotated_out, uint64_t *planes_out,
                     float *scal_out, float *q2c_out) {
  if (!ix || ix->info.kind != HS_KIND_SLIMQ || !queries || !rotated_out || !planes_out || !scal_out || !q2c_out) {
    set_error("hs_slimq_prepare: hnsw_slimq index and non-null buffers required");
    return HS_ERR_ARG;
  }
  if (nq == 0) return HS_OK;
  std::lock_guard<std::mutex> lock(ix->mu);
  HS_CUDA(cudaSetDevice(ix->device));
  const size_t dim = ix->info.dim, pd = ix->info.padded_dim_q, pw = ix->words * 4, nc = ix->info.num_cluster;
  float *d_q = nullptr, *d_rot = nullptr, *d_scal = nullptr, *d_q2c = nullptr;
  unsigned long long *d_pl = nullptr;
  auto cleanup = [&]() {
    cudaFree(d_q);
    cudaFree(d_rot);
    cudaFree(d_scal);
    cudaFree(d_q2c);
    cudaFree(d_pl);
  };
  if (cudaMalloc(&d_q, nq * dim * 4) != cudaSuccess || cudaMalloc(&d_rot, nq * pd * 4) != cudaSuccess ||
      cudaMalloc(&d_scal, nq * 12) != cudaSuccess || cudaMalloc(&d_q2c, nq * nc * 4) != cudaSuccess ||
      cudaMalloc(&d_pl, nq * pw * 8) != cudaSuccess) {
    cleanup();
    set_error("hs_slimq_prepare: cudaMalloc failed");
    return HS_ERR_NOMEM;
  }
  PrepDump dump{d_rot, d_pl, d_scal, d_q2c};
  int rc = HS_OK;
  cudaError_t e = cudaMemcpyAsync(d_q, queries, nq * dim * 4, cudaMemcpyHostToDevice, ix->stream);
  if (e == cudaSuccess) rc = search_device_slimq(ix, d_q, nq, 1, nullptr, nullptr, nullptr, ix->stream, &dump);
  if (e == cudaSuccess && rc == HS_OK) e = cudaMemcpyAsync(rotated_out, d_rot, nq * pd * 4, cudaMemcpyDeviceToHost, ix->stream);
  if (e == cudaSuccess && rc == HS_OK) e = cudaMemcpyAsync(planes_out, d_pl, nq * pw * 8, cudaMemcpyDeviceToHost, ix->stream);
  if (e == cudaSuccess && rc == HS_OK) e = cudaMemcpyAsync(scal_out, d_scal, nq * 12, cudaMemcpyDeviceToHost, ix->stream);
  if (e == cudaSuccess && rc == HS_OK) e = cudaMemcpyAsync(q2c_out, d_q2c, nq * nc * 4, cudaMemcpyDeviceToHost, ix->stream);
  if (e == cudaSuccess && rc == HS_OK) e = cudaStreamSynchronize(ix->stream);
  cleanup();
  if (rc != HS_OK) return rc;
  if (e != cudaSuccess) {
    set_error(std::string("hs_slimq_prepare: ") + cudaGetErrorString(e));
    return HS_ERR_CUDA;
  }
  return HS_OK;
}

int hs_get_info(const hs_index *ix, hs_index_info *out) {
  if (!ix || !out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = ix->info;
  return HS_OK;
}

int hs_search_batch(hs_index *ix, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                    float *dists_out) {
  return search_host(ix, queries, nq, k, labels_out, dists_out, nullptr);
}

int hs_search_batch_submit(hs_index *ix, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                           float *dists_out) {
  int rc = search_host(ix, queries, nq, k, labels_out, dists_out, nullptr, false);
  if (rc != HS_OK || !ix) return rc;
  std::lock_guard<std::mutex> lock(ix->mu);
  if (ix->ev_tail - ix->ev_head == hs_index::kEventRing) {       // ring full: retire the oldest batch
    HS_CUDA(cudaEventSynchronize(ix->ev_ring[ix->ev_head % hs_index::kEventRing]));
    ix->ev_head++;
  }
  cudaEvent_t &ev = ix->ev_ring[ix->ev_tail % hs_index::kEventRing];
  if (!ev) HS_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  HS_CUDA(cudaEventRecord(ev, ix->stream));
  ix->ev_tail++;
  return HS_OK;
}

int hs_search_batch_wait(hs_index *ix) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  std::lock_guard<std::mutex> lock(ix->mu);
  HS_CUDA(cudaSetDevice(ix->device));
  HS_CUDA(cudaStreamSynchronize(ix->stream));
  ix->ev_head = ix->ev_tail;
  return HS_OK;
}

int hs_search_batch_wait_oldest(hs_index *ix) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  cudaEvent_t ev;
  unsigned long long head;
  {
    std::lock_guard<std::mutex> lock(ix->mu);
    if (ix->ev_head == ix->ev_tail) return HS_OK;                  // nothing outstanding
    head = ix->ev_head;
    ev = ix->ev_ring[head % hs_index::kEventRing];
  }
  // the wait itself runs WITHOUT the handle's lock: another thread may go on submitting batches meanwhile
  // (hs_service: one thread submits, one waits).  The event cannot be re-used before ev_head moves past it.
  HS_CUDA(cudaSetDevice(ix->device));
  HS_CUDA(cudaEventSynchronize(ev));
  std::lock_guard<std::mutex> lock(ix->mu);
  if (ix->ev_head == head) ix->ev_head++;
  return HS_OK;
}

int hs_pin_host(void *ptr, size_t bytes) {
  if (!ptr || bytes == 0) {
    set_error("hs_pin_host: null / empty range");
    return HS_ERR_ARG;
  }
  cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
  if (e == cudaErrorHostMemoryAlreadyRegistered) {
    cudaGetLastError();
    return HS_OK;
  }
  if (e != cudaSuccess) {
    set_error(std::string("cudaHostRegister: ") + cudaGetErrorString(e));
    cudaGetLastError();
    return HS_ERR_CUDA;
  }
  return HS_OK;
}

int hs_unpin_host(void *ptr) {
  if (!ptr) return HS_OK;
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess && e != cudaErrorHostMemoryNotRegistered) {
    set_error(std::string("cudaHostUnregister: ") + cudaGetErrorString(e));
    cudaGetLastError();
    return HS_ERR_CUDA;
  }
  cudaGetLastError();
  return HS_OK;
}

int hs_search_batch_counts(hs_index *ix, const float *queries, size_t nq, size_t k, uint32_t *labels_out,
                           float *dists_out, uint32_t *per_query_counts) {
  return search_host(ix, queries, nq, k, labels_out, dists_out, per_query_counts);
}

int hs_search_batch_device(hs_index *ix, const float *d_queries, size_t nq, size_t k, uint32_t *d_labels,
                           float *d_dists, void *stream) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  // enqueueing mutates the handle (launch sequence number, plan cache, scratch growth): one caller at a time;
  // the launch itself is asynchronous, so this serialises microseconds of host work, not the searches
  std::lock_guard<std::mutex> lock(ix->mu);
  HS_CUDA(cudaSetDevice(ix->device));
  return search_device(ix, d_queries, nq, k, d_labels, d_dists, nullptr, static_cast<cudaStream_t>(stream));
}

int hs_search_batch_device_scatter(hs_index *ix, const float *d_queries, size_t nq, size_t k,
                                   uint32_t *const *d_labels_dsts, float *const *d_dists_dsts, size_t n_dsts,
                                   size_t slot, void *stream) {
  if (!d_labels_dsts || !d_dists_dsts || n_dsts == 0 || n_dsts > (size_t)kMaxScatter) {
    set_error("hs_search_batch_device_scatter: 1.." + std::to_string(kMaxScatter) + " destinations required");
    return HS_ERR_ARG;
  }
  ScatterDst sc;
  sc.n = (uint32_t)n_dsts;
  sc.row0 = (unsigned long long)slot * nq;
  for (size_t i = 0; i < n_dsts; ++i) {
    if (!d_labels_dsts[i] || !d_dists_dsts[i]) {
      set_error("hs_search_batch_device_scatter: null destination");
      return HS_ERR_ARG;
    }
    sc.labels[i] = d_labels_dsts[i];
    sc.dists[i] = d_dists_dsts[i];
  }
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  std::lock_guard<std::mutex> lock(ix->mu);
  HS_CUDA(cudaSetDevice(ix->device));
  return search_device(ix, d_queries, nq, k, nullptr, nullptr, nullptr, static_cast<cudaStream_t>(stream), &sc);
}

// ---- hs_exchange: the gather buffers of the sharded path, shared between the ranks of one box ----
}  // extern "C"

struct hs_exchange {
  int device = 0, world = 1, rank = 0;
  size_t rows = 0, k = 0;                  // rows = slots * nq_max per table
  uint8_t *base = nullptr;                 // own allocation: [2 x labels][2 x dists][flags]
  size_t bytes = 0;
  std::vector<uint8_t *> peer;             // base address of every rank's allocation in THIS process
  CUresult (*write32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  CUresult (*wait32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  size_t off_labels(int parity) const { return (size_t)parity * rows * k * 4; }
  size_t off_dists(int parity) const { return 2 * rows * k * 4 + (size_t)parity * rows * k * 4; }
  size_t off_flags() const { return 4 * rows * k * 4; }
};

extern "C" {

int hs_exchange_create(int device, int world, int rank, size_t slots, size_t nq_max, size_t k, hs_exchange **out) {
  if (!out || world < 1 || world > kMaxScatter || rank < 0 || rank >= world || slots == 0 || nq_max == 0 || k == 0) {
    set_error("hs_exchange_create: bad argument (world <= " + std::to_string(kMaxScatter) + ")");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  std::unique_ptr<hs_exchange> ex(new hs_exchange);
  ex->device = device;
  ex->world = world;
  ex->rank = rank;
  ex->rows = slots * nq_max;
  ex->k = k;
  ex->bytes = ex->off_flags() + 256;
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
    set_error("cuStreamWriteValue32 is not available from this driver");
    return HS_ERR_CUDA;
  }
  ex->write32 = reinterpret_cast<decltype(ex->write32)>(fn);
  if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
    set_error("cuStreamWaitValue32 is not available from this driver");
    return HS_ERR_CUDA;
  }
  ex->wait32 = reinterpret_cast<decltype(ex->wait32)>(fn);
  cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&ex->base), ex->bytes);
  if (e != cudaSuccess) {
    set_error(std::string("hs_exchange_create: cudaMalloc: ") + cudaGetErrorString(e));
    return HS_ERR_NOMEM;
  }
  if (cudaMemset(ex->base, 0, ex->bytes) != cudaSuccess) {
    set_error(std::string("hs_exchange_create: cudaMemset: ") + cudaGetErrorString(cudaGetLastError()));
    cudaFree(ex->base);
    return HS_ERR_CUDA;
  }
  ex->peer.assign(world, nullptr);
  ex->peer[rank] = ex->base;
  *out = ex.release();
  return HS_OK;
}

int hs_exchange_handle(hs_exchange *ex, void *handle64) {
  if (!ex || !handle64) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  HS_CUDA(cudaSetDevice(ex->device));
  HS_CUDA(cudaIpcGetMemHandle(&h, ex->base));
  std::memcpy(handle64, &h, 64);
  return HS_OK;
}

int hs_exchange_connect(hs_exchange *ex, const void *handles) {
  if (!ex || !handles) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  HS_CUDA(cudaSetDevice(ex->device));
  for (int r = 0; r < ex->world; ++r) {
    if (r == ex->rank) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const uint8_t *>(handles) + 64 * (size_t)r, 64);
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      set_error("cudaIpcOpenMemHandle(rank " + std::to_string(r) + "): " + cudaGetErrorString(e));
      cudaGetLastError();
      return HS_ERR_CUDA;
    }
    ex->peer[r] = static_cast<uint8_t *>(p);
  }
  return HS_OK;
}

int hs_exchange_search(hs_exchange *ex, hs_index *ix, const float *d_queries, size_t nq, size_t k, size_t slot,
                       unsigned int seq, void *stream) {
  if (!ex || nq * (slot + 1) > ex->rows || k != ex->k) {
    set_error("hs_exchange_search: slot / nq / k outside the exchange's shape");
    return HS_ERR_ARG;
  }
  uint32_t *labs[kMaxScatter];
  float *dsts[kMaxScatter];
  for (int r = 0; r < ex->world; ++r) {
    if (!ex->peer[r]) {
      set_error("hs_exchange_search: exchange not connected");
      return HS_ERR_ARG;
    }
    labs[r] = reinterpret_cast<uint32_t *>(ex->peer[r] + ex->off_labels(seq & 1));
    dsts[r] = reinterpret_cast<float *>(ex->peer[r] + ex->off_dists(seq & 1));
  }
  // the tables of one batch are laid out [slot][nq][k] with the CALL's nq (all ranks use the same)
  return hs_search_batch_device_scatter(ix, d_queries, nq, k, labs, dsts, (size_t)ex->world, slot, stream);
}

int hs_exchange_signal_and_wait(hs_exchange *ex, unsigned int seq, void *stream) {
  if (!ex || seq == 0) {
    set_error("hs_exchange_signal_and_wait: sequence numbers start at 1");
    return HS_ERR_ARG;
  }
  for (int r = 0; r < ex->world; ++r) {
    if (!ex->peer[r]) {
      set_error("hs_exchange_signal_and_wait: exchange not connected");
      return HS_ERR_ARG;
    }
  }
  CUstream s = static_cast<CUstream>(stream);
  // stream-ordered: after this rank's shard searches of batch `seq`, tell every rank (flag word
  // [this rank] in ITS allocation, release semantics), then hold the stream until every rank has
  // told us — copy-engine-free and SM-free: the traversal grids keep the SMs
  for (int r = 0; r < ex->world; ++r) {
    const CUdeviceptr a = reinterpret_cast<CUdeviceptr>(ex->peer[r] + ex->off_flags()) + 4u * (unsigned)ex->rank;
    const CUresult cr = ex->write32(s, a, seq, 0 /* CU_STREAM_WRITE_VALUE_DEFAULT */);
    if (cr != CUDA_SUCCESS) {
      set_error("cuStreamWriteValue32 failed (" + std::to_string((int)cr) + ")");
      return HS_ERR_CUDA;
    }
  }
  for (int r = 0; r < ex->world; ++r) {
    const CUdeviceptr a = reinterpret_cast<CUdeviceptr>(ex->base + ex->off_flags()) + 4u * (unsigned)r;
    const CUresult cr = ex->wait32(s, a, seq, 0 /* CU_STREAM_WAIT_VALUE_GEQ */);
    if (cr != CUDA_SUCCESS) {
      set_error("cuStreamWaitValue32 failed (" + std::to_string((int)cr) + ")");
      return HS_ERR_CUDA;
    }
  }
  return HS_OK;
}

int hs_exchange_tables(hs_exchange *ex, unsigned int seq, uint32_t **d_labels, float **d_dists) {
  if (!ex || !d_labels || !d_dists) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *d_labels = reinterpret_cast<uint32_t *>(ex->base + ex->off_labels(seq & 1));
  *d_dists = reinterpret_cast<float *>(ex->base + ex->off_dists(seq & 1));
  return HS_OK;
}

void hs_exchange_free(hs_exchange *ex) {
  if (!ex) return;
  cudaSetDevice(ex->device);
  for (int r = 0; r < ex->world; ++r)
    if (r != ex->rank && ex->peer[r]) cudaIpcCloseMemHandle(ex->peer[r]);
  cudaFree(ex->base);
  delete ex;
}

int hs_bruteforce_knn_device(const float *d_base, size_t n, size_t dim, const float *d_queries, size_t nq,
                             size_t k, int metric, uint32_t *d_labels, float *d_dists, void *stream) {
  if ((!d_base && n) || (!d_queries && nq) || (!d_labels && nq)) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  if (k > n) {
    set_error("bruteforce: k > n (bruteforce.h:107 asserts k <= cur_element_count)");
    return HS_ERR_ARG;
  }
  return bruteforce_device(d_base, n, dim, d_queries, nq, k, metric, d_labels, d_dists,
                           static_cast<cudaStream_t>(stream));
}

int hs_bruteforce_knn(const float *base, size_t n, size_t dim, const float *queries, size_t nq, size_t k,
                      int metric, int device, uint32_t *labels_out, float *dists_out) {
  if ((!base && n) || (!queries && nq) || (!labels_out && nq)) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  if (nq == 0) return HS_OK;
  // checked before the n == 0 return below: with no base rows there is nothing to write k rows from
  if (k > n) {
    set_error("bruteforce: k > n (bruteforce.h:107 asserts k <= cur_element_count)");
    return HS_ERR_ARG;
  }
  if (n == 0) return HS_OK;
  float *d_base = nullptr, *d_q = nullptr, *d_dist = nullptr;
  uint32_t *d_lab = nullptr;
  size_t bytes = 0;
  auto cleanup = [&]() {
    cudaFree(d_base);
    cudaFree(d_q);
    cudaFree(d_dist);
    cudaFree(d_lab);
  };
  if ((rc = upload(&d_base, base, n * dim, &bytes)) != HS_OK || (rc = upload(&d_q, queries, nq * dim, &bytes)) != HS_OK) {
    cleanup();
    return rc;
  }
  if (cudaMalloc(&d_lab, nq * k * 4) != cudaSuccess || cudaMalloc(&d_dist, nq * k * 4) != cudaSuccess) {
    set_error("cudaMalloc (bruteforce outputs) failed");
    cleanup();
    return HS_ERR_NOMEM;
  }
  rc = hs_bruteforce_knn_device(d_base, n, dim, d_q, nq, k, metric, d_lab, d_dist, nullptr);
  if (rc == HS_OK) {
    cudaError_t e = cudaMemcpy(labels_out, d_lab, nq * k * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && dists_out) e = cudaMemcpy(dists_out, d_dist, nq * k * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      set_error(std::string("bruteforce: ") + cudaGetErrorString(e));
      rc = HS_ERR_CUDA;
    }
  }
  cleanup();
  return rc;
}

long long hs_debug_bf_tc_fallback(void) { return bruteforce_last_tc_fallback(); }

int hs_topk_merge_device(const uint32_t *d_labels_in, const float *d_dists_in, size_t n_parts, size_t nq,
                         size_t k, uint32_t *d_labels_out, float *d_dists_out, void *stream) {
  if (!d_labels_in || !d_dists_in || !d_labels_out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  return topk_merge_device(d_labels_in, d_dists_in, n_parts, nq, k, d_labels_out, d_dists_out,
                           static_cast<cudaStream_t>(stream));
}

int hs_recall(const float *base, size_t n, size_t dim, const float *queries, size_t nq, const uint32_t *knn,
              size_t K, const uint32_t *gt, size_t gt_k, int metric, int device, double *recall_out) {
  if (!base || !queries || !knn || !gt || !recall_out || nq == 0 || K == 0) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  int rc = select_device(device);
  if (rc != HS_OK) return rc;
  float *d_base = nullptr, *d_q = nullptr;
  uint32_t *d_knn = nullptr, *d_gt = nullptr;
  unsigned long long *d_hits = nullptr;
  size_t bytes = 0;
  auto cleanup = [&]() {
    cudaFree(d_base);
    cudaFree(d_q);
    cudaFree(d_knn);
    cudaFree(d_gt);
    cudaFree(d_hits);
  };
  if ((rc = upload(&d_base, base, n * dim, &bytes)) != HS_OK || (rc = upload(&d_q, queries, nq * dim, &bytes)) != HS_OK ||
      (rc = upload(&d_knn, knn, nq * K, &bytes)) != HS_OK || (rc = upload(&d_gt, gt, nq * gt_k, &bytes)) != HS_OK) {
    cleanup();
    return rc;
  }
  if (cudaMalloc(&d_hits, 8) != cudaSuccess) {
    set_error("cudaMalloc failed");
    cleanup();
    return HS_ERR_NOMEM;
  }
  rc = recall_device(d_base, n, dim, d_q, nq, d_knn, K, d_gt, gt_k, metric, d_hits, nullptr);
  if (rc == HS_OK) {
    unsigned long long hits = 0;
    if (cudaMemcpy(&hits, d_hits, 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
      set_error("recall: cudaMemcpy failed");
      rc = HS_ERR_CUDA;
    } else {
      *recall_out = (double)hits / ((double)nq * (double)K);    // solve_strategy.h:101
    }
  }
  cleanup();
  return rc;
}

void hs_build_params_default(hs_build_params *p) {
  if (!p) return;
  p->M = 32;                       // core.h:31
  p->ef_construction = 128;        // main.cc:16
  p->branching_factor = "4";       // core.h:36
  p->threshold_level = 0;          // core.h:38
  p->top_degree_percent0 = 0.02f;  // main.cc:27
  p->top_degree_percent = 0.02f;
  p->top_M0 = 32;                  // main.cc:29
  p->low_m0 = 8;                   // top_M0 * Mm_ratio / 100, main.cc:64
  p->top_M = 16;                   // level_ratio% * top_M0, main.cc:65
  p->low_m = 4;                    // main.cc:66
  p->threads = 0;
  p->seed = 100;                   // hnsw.h:85 random_seed
}

static int parse_branching(const hs_build_params *p, double *bf) {
  if (!p || !p->branching_factor) {
    set_error("null build params");
    return HS_ERR_ARG;
  }
  const std::string b = p->branching_factor;     // hnsw.h:143-158
  if (b == "e") *bf = M_E;
  else if (b == "sqrt") *bf = std::sqrt(2.0) / (std::sqrt(2.0) - 1.0);
  else {
    char *end = nullptr;
    *bf = std::strtod(b.c_str(), &end);
    if (end == b.c_str() || *bf <= 1.0) {
      set_error("Invalid branching factor: " + b);
      return HS_ERR_ARG;
    }
  }
  return HS_OK;
}

int hs_build_slimq_graph(const float *base, size_t n, size_t dim, const hs_build_params *p, const float *centroids,
                         size_t num_cluster, const uint32_t *cluster_ids, const uint64_t *labels,
                         const char *out_graph_path) {
  double bf;
  int rc = parse_branching(p, &bf);
  if (rc != HS_OK) return rc;
  return guarded("hs_build_slimq_graph", [&] {
    return build_slimq_graph(base, n, dim, p->M, p->ef_construction, bf, p->threshold_level, p->top_degree_percent0,
                             p->top_degree_percent, p->top_M0, p->low_m0, p->top_M, p->low_m, p->threads, p->seed,
                             centroids, num_cluster, cluster_ids, labels, out_graph_path);
  });
}

int hs_build_slim_graph(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                        const uint64_t *labels, const char *out_graph_path) {
  double bf;
  int rc0 = parse_branching(p, &bf);
  if (rc0 != HS_OK) return rc0;
  return guarded("hs_build_slim_graph", [&] {
    return build_slim_graph(base, n, dim, metric, p->M, p->ef_construction, bf, p->threshold_level,
                            p->top_degree_percent0, p->top_degree_percent, p->top_M0, p->low_m0, p->top_M, p->low_m,
                            p->threads, p->seed, labels, out_graph_path);
  });
}

int hs_build_hnsw_graph(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                        const uint64_t *labels, const char *out_graph_path) {
  double bf;
  int rc0 = parse_branching(p, &bf);
  if (rc0 != HS_OK) return rc0;
  return guarded("hs_build_hnsw_graph", [&] {
    return build_hnsw_graph(base, n, dim, metric, p->M, p->ef_construction, bf, p->threads, p->seed, labels,
                            out_graph_path);
  });
}

int hs_build_slim_index_gpu(const float *base, size_t n, size_t dim, int metric, const hs_build_params *p,
                            const uint64_t *labels, int device, hs_index **out) {
  if (!out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  if (metric != HS_METRIC_L2 && metric != HS_METRIC_IP) {
    set_error("unknown metric");
    return HS_ERR_ARG;
  }
  double bf;
  int rc0 = parse_branching(p, &bf);
  if (rc0 != HS_OK) return rc0;
  try {
    return gpu_build_slim_index(base, n, dim, metric, p, bf, labels, device, out);
  } catch (const std::bad_alloc &) {
    set_error("hs_build_slim_index_gpu: out of host memory");
    return HS_ERR_NOMEM;
  }
}

int hs_build_slimq_index_gpu(const float *base, size_t n, size_t dim, const hs_build_params *p, const float *centroids,
                             size_t num_cluster, const uint64_t *labels, int device, hs_index **out) {
  if (!out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  double bf;
  int rc0 = parse_branching(p, &bf);
  if (rc0 != HS_OK) return rc0;
  return guarded("hs_build_slimq_index_gpu", [&] {
    return gpu_build_slimq_index(base, n, dim, p, bf, centroids, num_cluster, labels, device, out);
  });
}

int hs_debug_convert_gpu(const char *hnsw_graph_path, size_t dim, int metric, const hs_build_params *p, int device,
                         hs_index **out) {
  if (!out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  if (!hnsw_graph_path || !p || dim == 0 || (metric != HS_METRIC_L2 && metric != HS_METRIC_IP)) {
    set_error("hs_debug_convert_gpu: bad argument");
    return HS_ERR_ARG;
  }
  return guarded("hs_debug_convert_gpu", [&] { return gpu_debug_convert(hnsw_graph_path, dim, metric, p, device, out); });
}

int hs_debug_slimq_payload(const hs_index *ix, uint64_t *records, float *rotated_centroids, uint8_t *flip) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  if (ix->info.kind != HS_KIND_SLIMQ) {
    set_error("hs_debug_slimq_payload: not an hnsw_slimq index");
    return HS_ERR_ARG;
  }
  const hs_index_info &I = ix->info;
  HS_CUDA(cudaSetDevice(ix->device));
  if (records) HS_CUDA(cudaMemcpy(records, ix->d_qrec, I.n * (I.padded_dim_q / 64 + 2) * 8, cudaMemcpyDeviceToHost));
  if (rotated_centroids)
    HS_CUDA(cudaMemcpy(rotated_centroids, ix->d_centroids, I.num_cluster * I.padded_dim_q * 4, cudaMemcpyDeviceToHost));
  if (flip) HS_CUDA(cudaMemcpy(flip, ix->d_flip, 4 * I.padded_dim_q / 8, cudaMemcpyDeviceToHost));
  return HS_OK;
}

// saveIndex of an HBM-resident index: hnsw_slim (slim.h:717-751) — header, element records
// [int32 level][uint32 total][uint64 label][8 stale pointer bytes][float vec[dim]] — or hnsw_slimq
// (slimq.h:1161-1216, write_slimq_file in graph_build.cpp); then per node uint32 blob size +
// [uint16 offsets[level]][uint32 ids[total]].  Labels are the device's 32-bit labels, zero-extended; the
// pointer bytes are written as 0.
int hs_save_index(hs_index *ix, const char *path) {
  if (!ix || !path) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  if (ix->info.kind != HS_KIND_SLIM && ix->info.kind != HS_KIND_SLIMQ) {
    set_error("hs_save_index: only hnsw_slim and hnsw_slimq indices can be saved");
    return HS_ERR_UNSUPPORTED;
  }
  try {
    HS_CUDA(cudaSetDevice(ix->device));
    HS_CUDA(cudaDeviceSynchronize());
    const hs_index_info &I = ix->info;
    const size_t n = I.n, dim = I.dim, dp = I.dim_padded;
    std::vector<int32_t> slot(n);
    std::vector<uint32_t> labels(n), adj0(n * (size_t)I.deg0_stride);
    HS_CUDA(cudaMemcpy(slot.data(), ix->d_upper_slot, n * 4, cudaMemcpyDeviceToHost));
    HS_CUDA(cudaMemcpy(labels.data(), ix->d_labels, n * 4, cudaMemcpyDeviceToHost));
    HS_CUDA(cudaMemcpy(adj0.data(), ix->d_adj0, adj0.size() * 4, cudaMemcpyDeviceToHost));
    // a patched index may hold nodes above the header's maxlevel (patchFromStream leaves maxlevel_ alone)
    int top = I.maxlevel;
    while (top + 1 < kMaxLevels && ix->level_count[top + 1] > 0 && ix->d_upper_adj[top + 1]) ++top;
    std::vector<std::vector<uint32_t>> up(top + 1);
    for (int l = 1; l <= top; ++l) {
      up[l].resize((size_t)ix->level_count[l] * I.upper_stride);
      if (!up[l].empty())
        HS_CUDA(cudaMemcpy(up[l].data(), ix->d_upper_adj[l], up[l].size() * 4, cudaMemcpyDeviceToHost));
    }
    auto level_of = [&](size_t i) {
      int lv = 0;
      if (slot[i] >= 0)
        while (lv < top && (uint32_t)slot[i] < ix->level_count[lv + 1]) ++lv;
      return lv;
    };
    auto list = [&](size_t i, int l, const uint32_t **ids) {
      const uint32_t *row = l == 0 ? &adj0[i * I.deg0_stride] : &up[l][(size_t)slot[i] * I.upper_stride];
      const uint32_t stride = l == 0 ? I.deg0_stride : I.upper_stride;
      uint32_t c = 0;
      while (c < stride && row[c] != kInvalid) ++c;
      *ids = row;
      return c;
    };
    auto total_of = [&](size_t i, int lv) {
      uint32_t total = 0;
      const uint32_t *ids;
      for (int l = 0; l <= lv; ++l) total += list(i, l, &ids);
      return total;
    };
    auto write_blobs = [&](FILE *f) {
      std::vector<uint8_t> blob;
      bool ok = true;
      for (size_t i = 0; i < n && ok; ++i) {
        const int lv = level_of(i);
        const uint32_t total = total_of(i, lv);
        const uint32_t bsz = (uint32_t)(2 * lv + 4 * total);
        ok &= std::fwrite(&bsz, 1, 4, f) == 4;
        if (bsz == 0 || total == 0) continue;          // slim.h:741-748
        blob.resize(bsz);
        uint32_t run = 0;
        size_t w = 2 * (size_t)lv;
        const uint32_t *ids;
        for (int l = 0; l <= lv; ++l) {
          const uint32_t c = list(i, l, &ids);
          std::memcpy(&blob[w], ids, 4 * (size_t)c);
          w += 4 * (size_t)c;
          run += c;
          if (l < lv) {
            const uint16_t o = (uint16_t)run;
            std::memcpy(&blob[2 * l], &o, 2);
          }
        }
        ok &= std::fwrite(blob.data(), 1, bsz, f) == bsz;
      }
      return ok;
    };

    if (I.kind == HS_KIND_SLIMQ) {
      const size_t pd = I.padded_dim_q, words = pd / 64, rw = words + 2;
      std::vector<float> cent(I.num_cluster * pd);
      std::vector<uint8_t> flip(4 * pd / 8);
      HS_CUDA(cudaMemcpy(cent.data(), ix->d_centroids, cent.size() * 4, cudaMemcpyDeviceToHost));
      HS_CUDA(cudaMemcpy(flip.data(), ix->d_flip, flip.size(), cudaMemcpyDeviceToHost));
      SlimqHead head;
      head.n = n;
      head.maxlevel = I.maxlevel;
      head.threshold_level = I.threshold_level;
      head.enterpoint = I.enterpoint;
      head.maxM = I.maxM;
      head.maxM0 = I.maxM0;
      head.M = I.M;
      head.ef_construction = I.ef_construction;
      head.num_cluster = I.num_cluster;
      head.dim = dim;
      head.padded_dim = pd;
      head.ex_bits = ix->ex_bits;
      head.size_ex = ix->size_ex;
      head.centroids = cent.data();
      head.flip = flip.data();
      std::vector<uint2> rec;
      std::vector<uint64_t> code;
      // the records streamed from the device in slabs; qrec holds each code word as (low half, high half)
      return write_slimq_file(
          path, head,
          [&](size_t i0, size_t cnt, SlimqNode *out) -> int {
            rec.resize(cnt * rw);
            code.resize(cnt * words);
            HS_CUDA(cudaMemcpy(rec.data(), ix->d_qrec + i0 * rw, rec.size() * 8, cudaMemcpyDeviceToHost));
            for (size_t j = 0; j < cnt; ++j) {
              const size_t i = i0 + j;
              const uint2 *r = &rec[j * rw];
              for (size_t w = 0; w < words; ++w) code[j * words + w] = (uint64_t)r[w].y << 32 | r[w].x;
              SlimqNode &nd = out[j];
              nd.level = level_of(i);
              nd.total = total_of(i, nd.level);
              nd.label = labels[i];
              nd.cluster = r[words + 1].x;
              nd.code = &code[j * words];
              std::memcpy(&nd.f_add, &r[words].x, 4);
              std::memcpy(&nd.f_rescale, &r[words].y, 4);
              nd.f_error = ix->f_error[i];
            }
            return HS_OK;
          },
          write_blobs);
    }

    FILE *f = std::fopen(path, "wb");
    if (!f) {
      set_error(std::string("cannot open ") + path + " for writing");
      return HS_ERR_IO;
    }
    auto put = [&](const void *p, size_t sz) { return std::fwrite(p, 1, sz, f) == sz; };
    bool ok = true;
    const uint64_t rec = 24 + 4 * dim;
    const uint64_t hdr[6] = {n, rec, 8, 4, 24, 16};
    ok &= put(hdr, sizeof hdr);
    const int32_t ml = I.maxlevel, thr = I.threshold_level;
    const uint32_t ep = I.enterpoint;
    ok &= put(&ml, 4) && put(&thr, 4) && put(&ep, 4);
    const uint64_t ms[4] = {I.maxM, I.maxM0, I.M, I.ef_construction};
    ok &= put(ms, sizeof ms);
    const uint8_t has_deleted = 0;
    ok &= put(&has_deleted, 1);
    // element records, the vectors streamed from the device in slabs
    const size_t slab = std::max<size_t>(1, (64u << 20) / (dp * 4));
    std::vector<float> rows(slab * dp);
    std::vector<uint8_t> record(rec);
    for (size_t i0 = 0; i0 < n && ok; i0 += slab) {
      const size_t cnt = std::min(slab, n - i0);
      HS_CUDA(cudaMemcpy(rows.data(), ix->d_vec + i0 * dp, cnt * dp * 4, cudaMemcpyDeviceToHost));
      for (size_t j = 0; j < cnt && ok; ++j) {
        const size_t i = i0 + j;
        const int32_t lv = level_of(i);
        const uint32_t total = total_of(i, lv);
        const uint64_t label = labels[i], stale_ptr = 0;
        std::memcpy(&record[0], &lv, 4);
        std::memcpy(&record[4], &total, 4);
        std::memcpy(&record[8], &label, 8);
        std::memcpy(&record[16], &stale_ptr, 8);
        std::memcpy(&record[24], &rows[j * dp], 4 * dim);
        ok &= put(record.data(), rec);
      }
    }
    ok = ok && write_blobs(f);
    ok &= std::fclose(f) == 0;
    if (!ok) {
      set_error(std::string("write error on ") + path);
      return HS_ERR_IO;
    }
    return HS_OK;
  } catch (const std::bad_alloc &) {
    set_error("hs_save_index: out of host memory");
    return HS_ERR_NOMEM;
  }
}

// ---- host-only inspection of the flattened graph (used by the CPU test-suite; no CUDA) ----
struct hs_host_graph {
  HostGraph g;
};

int hs_debug_flatten(const char *graph_path, int kind, size_t dim, hs_host_graph **out) {
  if (!graph_path || !out) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  *out = nullptr;
  return guarded("hs_debug_flatten", [&] {
    std::vector<uint8_t> bytes;
    int rc = read_file(graph_path, &bytes);
    if (rc != HS_OK) return rc;
    std::unique_ptr<hs_host_graph> h(new hs_host_graph);
    rc = parse_graph(bytes.data(), bytes.size(), kind, dim, &h->g);
    if (rc != HS_OK) return rc;
    *out = h.release();
    return (int)HS_OK;
  });
}

void hs_debug_free(hs_host_graph *h) { delete h; }

int hs_debug_info(const hs_host_graph *h, hs_index_info *I) {
  if (!h || !I) return HS_ERR_ARG;
  const HostGraph &g = h->g;
  std::memset(I, 0, sizeof *I);
  I->n = g.n;
  I->dim = g.dim;
  I->dim_padded = g.dim_padded;
  I->M = g.M;
  I->maxM = g.maxM;
  I->maxM0 = g.maxM0;
  I->ef_construction = g.ef_construction;
  I->maxlevel = g.maxlevel;
  I->threshold_level = g.threshold_level;
  I->enterpoint = g.enterpoint;
  I->has_deleted = g.has_deleted;
  I->kind = g.kind;
  I->deg0_stride = g.deg0_stride;
  I->max_deg0 = g.max_deg0;
  I->upper_stride = g.upper_stride;
  I->n_upper = g.n_upper;
  I->sum_deg0 = g.sum_deg0;
  I->padded_dim_q = g.padded_dim_q;
  I->num_cluster = g.num_cluster;
  return HS_OK;
}

// level-`level` row of `node` as stored for the device (kInvalid-padded); returns the row
// stride, 0 if the node has no row at that level, negative on error.
int hs_debug_row(const hs_host_graph *h, uint32_t node, int level, uint32_t *out, int cap) {
  if (!h || !out || node >= h->g.n || level < 0) return HS_ERR_ARG;
  const HostGraph &g = h->g;
  const uint32_t *row;
  int stride;
  if (level == 0) {
    row = &g.adj0[(size_t)node * g.deg0_stride];
    stride = (int)g.deg0_stride;
  } else {
    if ((size_t)level >= g.upper_adj.size() || (size_t)level >= g.level_count.size() || g.upper_slot[node] < 0 ||
        (uint32_t)g.upper_slot[node] >= g.level_count[level])
      return 0;
    row = &g.upper_adj[level][(size_t)g.upper_slot[node] * g.upper_stride];
    stride = (int)g.upper_stride;
  }
  for (int i = 0; i < stride && i < cap; ++i) out[i] = row[i];
  return stride;
}

int hs_debug_node(const hs_host_graph *h, uint32_t node, int *level, uint32_t *label, float *vec_out) {
  if (!h || node >= h->g.n) return HS_ERR_ARG;
  const HostGraph &g = h->g;
  if (level) *level = g.levels[node];
  if (label) *label = g.labels[node];
  if (vec_out && !g.vec.empty()) std::memcpy(vec_out, &g.vec[(size_t)node * g.dim_padded], g.dim_padded * 4);
  return HS_OK;
}

int hs_debug_patch(hs_host_graph *h, const void *patch, size_t patch_bytes, unsigned flags, const float *rows,
                   const uint64_t *row_labels, size_t n_rows, hs_patch_info *info_out) {
  if (!h || !patch) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  return guarded("hs_debug_patch", [&]() -> int {
    HostGraph &g = h->g;
    PatchSet ps;
    // the host image grows as needed, within reason: a corrupt element count must not turn into a 100 GB resize
    const uint64_t cap = std::min<uint64_t>((1ull << 31) - 1, g.n + (1ull << 22));
    int rc = parse_patch(static_cast<const uint8_t *>(patch), patch_bytes, g.dim, (flags & HS_PATCH_INLINE_ROWS) != 0, g.n,
                         cap, &ps);
    if (rc != HS_OK) return rc;
    PatchRows pr;
    pr.rows = rows;
    pr.row_labels = row_labels;
    pr.n_rows = n_rows;
    pr.dim = g.dim;
    pr.prepare();
    const uint64_t n_before = g.n;
    bool upper = false;
    rc = apply_patch_host(&g, ps, pr, &upper);
    if (rc != HS_OK) return rc;
    if (info_out) {
      info_out->n_before = n_before;
      info_out->n_after = g.n;
      info_out->changed_old = ps.n_old;
      info_out->changed_new = ps.n_new;
      info_out->bytes_consumed = ps.consumed;
      info_out->rows_written = 0;
      info_out->upper_rebuilt = upper ? 1 : 0;
    }
    return (int)HS_OK;
  });
}

int hs_stats(hs_index *ix, uint64_t *n_dist, uint64_t *n_hops, uint64_t *n_rerank) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  unsigned long long h[4] = {0, 0, 0, 0};
  HS_CUDA(cudaSetDevice(ix->device));
  HS_CUDA(cudaDeviceSynchronize());
  HS_CUDA(cudaMemcpy(h, ix->d_stats, sizeof h, cudaMemcpyDeviceToHost));
  if (n_dist) *n_dist = h[0];
  if (n_hops) *n_hops = h[1];
  if (n_rerank) *n_rerank = h[2];
  return HS_OK;
}

int hs_reset_stats(hs_index *ix) {
  if (!ix) {
    set_error("null argument");
    return HS_ERR_ARG;
  }
  HS_CUDA(cudaSetDevice(ix->device));
  HS_CUDA(cudaDeviceSynchronize());
  HS_CUDA(cudaMemset(ix->d_stats, 0, 4 * sizeof(unsigned long long)));
  return HS_OK;
}

}  // extern "C"
