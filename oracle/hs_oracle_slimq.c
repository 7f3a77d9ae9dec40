/* TEST INFRASTRUCTURE — NOT PRODUCT CODE.  See hs_oracle.h.
 *
 * Plain-C restatement of the reference's hnsw_slimq search path
 * (slimq.h = third_party/hnswlib/hnswalg_slimq.h, rq/ = third_party/rabitqlib/):
 * index load, FHT-Kac query rotation, 4-bit scalar query quantiser, bit-plane
 * transpose, 1-bit popcount distance estimator, sorted-buffer beam search and exact
 * rerank.  Written from the algorithm; every function names the file:line it follows.
 *
 * Floating point: every operation is a single correctly-rounded fp32 (or, where the
 * reference computes in double, fp64) operation, no contraction (-ffp-contract=off).
 * Reductions (sums of squares, dot products, the query sum) use ONE fixed association
 * — "warp order": 32 partial sums, partial l takes elements l, l+32, ... in index
 * order, then an xor butterfly 16,8,4,2,1 — which the CUDA kernel reproduces bit for
 * bit.  The reference reduces with Eigen / std::accumulate under -Ofast (association
 * unspecified), so the pin against the live reference is: rotation bit-exact,
 * quantised query codes identical, scalar factors and estimates within 1e-5 relative,
 * search results identical when the reference's own per-query preparation is injected
 * (tests/test_oracle_slimq.py).
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "hs_oracle.h"

#ifdef _OPENMP
#include <omp.h>
#endif

static _Thread_local char gq_err[256];
const char *hsoq_last_error(void) { return gq_err; }

/* slimq.h:1498-1505 record: [int32 level @0][uint32 total @4][uint64 label @8][ptr @16]
 * [uint32 cluster @24][bin @28: uint64 code[pd/64], float f_add, f_rescale, f_error][ex ...] */
struct hsoq_index {
  uint64_t n, size_data_per_element, label_offset, offset_total, offset_data, offset_nbr;
  uint64_t maxM, maxM0, M, ef_construction;
  int32_t maxlevel, threshold_level;
  uint32_t enterpoint;
  uint8_t has_deleted;
  uint64_t num_cluster, dim, padded_dim, offset_cluster_id, offset_bin_data, offset_ex_data, size_bin_data,
      size_ex_data, ex_bits;
  uint8_t metric_type;
  float *centroids;    /* num_cluster x padded_dim, already rotated */
  uint8_t *flip;       /* 4 * padded_dim / 8 bytes */
  char *elements;
  char **blobs;
  double t_const;
  size_t trunc_dim;
};

static int rdq(FILE *f, void *p, size_t n) { return fread(p, 1, n, f) == n ? 0 : -1; }

/* slimq.h:1218-1313 (written by :1161-1216) */
hsoq_index *hsoq_load(const char *path, size_t dim) {
  FILE *f = fopen(path, "rb");
  if (!f) {
    snprintf(gq_err, sizeof gq_err, "Cannot open file %s", path);
    return NULL;
  }
  hsoq_index *ix = (hsoq_index *)calloc(1, sizeof *ix);
  int bad = 0;
  bad |= rdq(f, &ix->n, 8);
  bad |= rdq(f, &ix->size_data_per_element, 8);
  bad |= rdq(f, &ix->label_offset, 8);
  bad |= rdq(f, &ix->offset_total, 8);
  bad |= rdq(f, &ix->offset_data, 8);
  bad |= rdq(f, &ix->offset_nbr, 8);
  bad |= rdq(f, &ix->maxlevel, 4);
  bad |= rdq(f, &ix->threshold_level, 4);
  bad |= rdq(f, &ix->enterpoint, 4);
  bad |= rdq(f, &ix->maxM, 8);
  bad |= rdq(f, &ix->maxM0, 8);
  bad |= rdq(f, &ix->M, 8);
  bad |= rdq(f, &ix->ef_construction, 8);
  bad |= rdq(f, &ix->has_deleted, 1);
  bad |= rdq(f, &ix->num_cluster, 8);
  bad |= rdq(f, &ix->dim, 8);
  bad |= rdq(f, &ix->padded_dim, 8);
  bad |= rdq(f, &ix->offset_cluster_id, 8);
  bad |= rdq(f, &ix->offset_bin_data, 8);
  bad |= rdq(f, &ix->offset_ex_data, 8);
  bad |= rdq(f, &ix->size_bin_data, 8);
  bad |= rdq(f, &ix->size_ex_data, 8);
  bad |= rdq(f, &ix->ex_bits, 8);
  bad |= rdq(f, &ix->metric_type, 1);
  if (bad || ix->dim != dim || ix->padded_dim % 64 || ix->padded_dim < dim) {
    snprintf(gq_err, sizeof gq_err, "bad hnsw_slimq header in %s", path);
    fclose(f);
    free(ix);
    return NULL;
  }
  ix->centroids = (float *)malloc(ix->num_cluster * ix->padded_dim * sizeof(float) + 4);
  ix->flip = (uint8_t *)malloc(4 * ix->padded_dim / 8);
  bad |= rdq(f, ix->centroids, ix->num_cluster * ix->padded_dim * sizeof(float));
  bad |= rdq(f, ix->flip, 4 * ix->padded_dim / 8);          /* rotator.hpp:256-261 */
  ix->elements = (char *)malloc(ix->n * ix->size_data_per_element + 1);
  ix->blobs = (char **)calloc(ix->n + 1, sizeof(char *));
  bad |= rdq(f, ix->elements, ix->n * ix->size_data_per_element);
  for (uint64_t i = 0; i < ix->n && !bad; i++) {
    uint32_t sz;
    if (rdq(f, &sz, 4)) { bad = 1; break; }
    uint32_t total = *(uint32_t *)(ix->elements + i * ix->size_data_per_element + ix->offset_total);
    if (sz == 0 || total == 0) continue;                    /* slimq.h:1295-1298 */
    ix->blobs[i] = (char *)malloc(sz);
    if (rdq(f, ix->blobs[i], sz)) bad = 1;
  }
  fclose(f);
  if (bad) {
    snprintf(gq_err, sizeof gq_err, "truncated graph file %s", path);
    hsoq_free(ix);
    return NULL;
  }
  /* rotator.hpp:233-235: trunc_dim = 2^floor(log2(dim)) of the UNPADDED dim */
  size_t t = 1;
  while (t * 2 <= dim) t *= 2;
  ix->trunc_dim = t;
  ix->t_const = -1.0;
  return ix;
}

void hsoq_free(hsoq_index *ix) {
  if (!ix) return;
  if (ix->blobs) {
    for (uint64_t i = 0; i < ix->n; i++) free(ix->blobs[i]);
    free(ix->blobs);
  }
  free(ix->elements);
  free(ix->centroids);
  free(ix->flip);
  free(ix);
}

void hsoq_get_info(const hsoq_index *ix, hsoq_info *o) {
  o->n = ix->n;
  o->size_data_per_element = ix->size_data_per_element;
  o->maxM = ix->maxM;
  o->maxM0 = ix->maxM0;
  o->M = ix->M;
  o->ef_construction = ix->ef_construction;
  o->dim = ix->dim;
  o->padded_dim = ix->padded_dim;
  o->num_cluster = ix->num_cluster;
  o->ex_bits = ix->ex_bits;
  o->maxlevel = ix->maxlevel;
  o->threshold_level = ix->threshold_level;
  o->enterpoint = ix->enterpoint;
  o->metric_type = ix->metric_type;
}

/* the query-quantiser constant (slimq.h:1274-1276): the reference draws it at random at
 * load time; the caller supplies the value to use */
void hsoq_set_tconst(hsoq_index *ix, double t) { ix->t_const = t; }

static inline const char *qelem(const hsoq_index *ix, uint32_t i) {
  return ix->elements + (size_t)i * ix->size_data_per_element;
}
static inline int q_level(const hsoq_index *ix, uint32_t i) { return *(const int32_t *)qelem(ix, i); }
static inline uint32_t q_total(const hsoq_index *ix, uint32_t i) {
  return *(const uint32_t *)(qelem(ix, i) + ix->offset_total);
}
static inline uint64_t q_label(const hsoq_index *ix, uint32_t i) {
  uint64_t l;
  memcpy(&l, qelem(ix, i) + ix->label_offset, 8);
  return l;
}

/* level slice of the blob: slimq.h:1873-1886 (upper levels), :706-715 (level 0) */
static int q_neighbors(const hsoq_index *ix, uint32_t i, int level, const uint32_t **ids) {
  const char *blob = ix->blobs[i];
  *ids = NULL;
  if (!blob) return 0;
  int el = q_level(ix, i);
  if (level > el) return 0;
  const uint16_t *offs = (const uint16_t *)blob;
  uint32_t begin = level == 0 ? 0 : offs[level - 1];
  uint32_t end = level == el ? q_total(ix, i) : offs[level];
  *ids = (const uint32_t *)(blob + 2 * (size_t)el) + begin;
  return (int)(end - begin);
}

int hsoq_node(const hsoq_index *ix, uint32_t node, uint32_t *cluster, uint64_t *code, float *factors,
              uint32_t *nbr_out, int cap) {
  const char *e = qelem(ix, node);
  memcpy(cluster, e + ix->offset_cluster_id, 4);
  memcpy(code, e + ix->offset_bin_data, ix->padded_dim / 8);
  memcpy(factors, e + ix->offset_bin_data + ix->padded_dim / 8, 12);
  const uint32_t *ids;
  int cnt = q_neighbors(ix, node, 0, &ids);
  for (int j = 0; j < cnt && j < cap; j++) nbr_out[j] = ids[j];
  return cnt;
}

/* ------------------------------------------------------------ reductions -- */
/* "warp order" sum of term(i), i < len (see the file comment) */
static float warp_sum(const float *terms, size_t len) {
  float lane[32];
  for (int l = 0; l < 32; l++) {
    float acc = 0.f;
    for (size_t i = (size_t)l; i < len; i += 32) acc = acc + terms[i];
    lane[l] = acc;
  }
  for (int off = 16; off >= 1; off >>= 1) {
    float nxt[32];
    for (int l = 0; l < 32; l++) nxt[l] = lane[l] + lane[l ^ off];
    memcpy(lane, nxt, sizeof lane);
  }
  return lane[0];
}
/* same association with term(i) = a[i]*b[i] accumulated by fma */
static float warp_dot(const float *a, const float *b, size_t len) {
  float lane[32];
  for (int l = 0; l < 32; l++) {
    float acc = 0.f;
    for (size_t i = (size_t)l; i < len; i += 32) acc = fmaf(a[i], b[i], acc);
    lane[l] = acc;
  }
  for (int off = 16; off >= 1; off >>= 1) {
    float nxt[32];
    for (int l = 0; l < 32; l++) nxt[l] = lane[l] + lane[l ^ off];
    memcpy(lane, nxt, sizeof lane);
  }
  return lane[0];
}
/* sum (a-b)^2, fma accumulation, warp order */
static float warp_l2(const float *a, const float *b, size_t len) {
  float lane[32];
  for (int l = 0; l < 32; l++) {
    float acc = 0.f;
    for (size_t i = (size_t)l; i < len; i += 32) {
      float d = a[i] - b[i];
      acc = fmaf(d, d, acc);
    }
    lane[l] = acc;
  }
  for (int off = 16; off >= 1; off >>= 1) {
    float nxt[32];
    for (int l = 0; l < 32; l++) nxt[l] = lane[l] + lane[l ^ off];
    memcpy(lane, nxt, sizeof lane);
  }
  return lane[0];
}

/* --------------------------------------------------------------- rotation -- */
/* rotator.hpp:100-205: bit (i % 8) of byte i / 8 set => negate element i */
static void flip_sign(const uint8_t *flip, float *data, size_t dim) {
  for (size_t i = 0; i < dim; i++)
    if ((flip[i / 8] >> (i % 8)) & 1u) data[i] = -data[i];
}
/* fht_avx.hpp:29-38 ...: unnormalised in-place Walsh-Hadamard transform, natural order,
 * butterfly distance 1, 2, 4, ... (u, v) -> (u + v, u - v) */
static void fwht(float *buf, size_t len) {
  for (size_t h = 1; h < len; h *= 2)
    for (size_t j = 0; j < len; j += 2 * h)
      for (size_t k = 0; k < h; k++) {
        float u = buf[j + k], v = buf[j + k + h];
        buf[j + k] = u + v;
        buf[j + k + h] = u - v;
      }
}
/* rotator.hpp:299-368 */
static void kacs_walk(float *data, size_t len) {
  for (size_t i = 0; i < len / 2; i++) {
    float x = data[i], y = data[i + len / 2];
    data[i] = x + y;
    data[i + len / 2] = x - y;
  }
}
static void rescale(float *data, size_t len, float f) {
  for (size_t i = 0; i < len; i++) data[i] = data[i] * f;
}

/* FhtKacRotator::rotate, rotator.hpp:370-423 */
void hsoq_rotate(const hsoq_index *ix, const float *q, float *out) {
  const size_t pd = ix->padded_dim, td = ix->trunc_dim;
  const float fac = 1.0f / sqrtf((float)td);                 /* rotator.hpp:235 */
  memcpy(out, q, sizeof(float) * ix->dim);
  for (size_t i = ix->dim; i < pd; i++) out[i] = 0.f;
  if (td == pd) {                                             /* :374-396 */
    for (int r = 0; r < 4; r++) {
      flip_sign(ix->flip + r * pd / 8, out, pd);
      fwht(out, td);
      rescale(out, td, fac);
    }
    return;
  }
  const size_t start = pd - td;                               /* :398-422 */
  for (int r = 0; r < 4; r++) {
    float *seg = (r & 1) ? out + start : out;
    flip_sign(ix->flip + r * pd / 8, out, pd);
    fwht(seg, td);
    rescale(seg, td, fac);
    kacs_walk(out, pd);
  }
  rescale(out, pd, 0.25f);
}

/* -------------------------------------------------------- query quantiser -- */
/* SplitSingleQuery ctor (rq/index/query.hpp:127-156) -> quantize_scalar (rabitq.hpp:322-337)
 * -> rabitq_scalar_impl (rabitq_impl.hpp:534-581) with centroid 0 -> one_bit_code (:39-54),
 * ex_bits_code (:405-432), faster_quantize_ex (:379-403); then new_transpose_bin
 * (rq/utils/space.hpp:1405-1516).
 *   planes[w*4 + j]: bit (63 - l) = bit j of the 4-bit code of dimension 64 w + l
 *   scal[0] = delta, scal[1] = vl, scal[2] = k1xsumq = -0.5 * sum(q')            */
void hsoq_quantize_query(const hsoq_index *ix, const float *rq, uint64_t *planes, float *scal,
                         uint16_t *codes_out) {
  const size_t pd = ix->padded_dim;
  const int ex_bits = 3;                                      /* kNumBits = 4 total (query.hpp:126) */
  float *tmp = (float *)malloc(sizeof(float) * pd * 2);
  float *ucb = tmp + pd;
  const float sumq = warp_sum(rq, pd);                        /* query.hpp:135-136 */
  const float norm_data = sqrtf(warp_dot(rq, rq, pd));        /* rabitq_impl.hpp:561 */
  for (size_t i = 0; i < pd; i++) {
    const float r = rq[i];
    /* rabitq_impl.hpp:414: rowwise().normalized().abs() */
    const float o = norm_data > 0.f ? fabsf(r) / norm_data : fabsf(r);
    /* rabitq_impl.hpp:386-390: double arithmetic */
    int c = (int)((ix->t_const * (double)o) + 1e-5);
    if (c >= (1 << ex_bits)) c = (1 << ex_bits) - 1;
    if (r < 0.f) c = (~c) & ((1 << ex_bits) - 1);             /* :424-429 */
    const int b = r > 0.f ? 1 : 0;                            /* :51 */
    const int u = c + (b << ex_bits);                         /* :553-555 */
    if (codes_out) codes_out[i] = (uint16_t)u;
    ucb[i] = (float)u + -7.5f;                                /* :557-559, cb = -(2^3 - 0.5) */
    tmp[i] = (float)u;
  }
  const float norm_quan = sqrtf(warp_dot(ucb, ucb, pd));      /* :562 */
  /* :563-564.  norm_data == 0 (zero query, or squares that underflow): the reference divides 0 by 0 and every
   * estimate is NaN, which qb_is_full never rejects, so its search walks the whole reachable graph.  We depart
   * from it on purpose: cosv = 0, so delta = vl = 0 and the estimate is f_add + |c|^2, the RaBitQ estimate of
   * |x|^2 (traverse_slimq.cu does the same). */
  const float cosv = norm_data > 0.f ? warp_dot(rq, ucb, pd) / (norm_data * norm_quan) : 0.f;
  const float delta = norm_data / norm_quan * cosv;           /* :567 (RECONSTRUCTION) */
  scal[0] = delta;
  scal[1] = delta * -7.5f;                                    /* :574 */
  scal[2] = sumq * -0.5f;                                     /* query.hpp:133,138 */
  for (size_t w = 0; w < pd / 64; w++)
    for (int j = 0; j < 4; j++) {
      uint64_t v = 0;
      for (int l = 0; l < 64; l++)
        if (((int)tmp[64 * w + l] >> j) & 1) v |= 1ull << (63 - l);
      planes[w * 4 + j] = v;
    }
  free(tmp);
}

/* the whole per-query preparation of searchKnn, slimq.h:1816-1847 (L2 metric) */
void hsoq_prep(const hsoq_index *ix, const float *q, float *rotated, uint64_t *planes, float *scal,
               float *q2c) {
  hsoq_rotate(ix, q, rotated);
  hsoq_quantize_query(ix, rotated, planes, scal, NULL);
  for (size_t c = 0; c < ix->num_cluster; c++)               /* slimq.h:1825-1832 */
    q2c[c] = sqrtf(warp_l2(rotated, ix->centroids + c * ix->padded_dim, ix->padded_dim));
}

/* -------------------------------------------------------------- estimator -- */
/* get_bin_est (slimq.h:408-440, L2 branch) -> split_single_estdist (rq/index/estimator.hpp:164-188)
 * -> warmup_ip_x0_q<4> (rq/utils/warmup_space.hpp:8-102) */
float hsoq_est(const hsoq_index *ix, uint32_t node, const uint64_t *planes, const float *scal,
               const float *q2c) {
  const char *e = qelem(ix, node);
  uint32_t cluster;
  memcpy(&cluster, e + ix->offset_cluster_id, 4);
  const char *bin = e + ix->offset_bin_data;
  const size_t words = ix->padded_dim / 64;
  uint64_t ip = 0, ppc = 0;
  for (size_t w = 0; w < words; w++) {
    uint64_t x;
    memcpy(&x, bin + 8 * w, 8);
    ppc += (uint64_t)__builtin_popcountll(x);
    for (int j = 0; j < 4; j++) ip += (uint64_t)__builtin_popcountll(x & planes[w * 4 + j]) << j;
  }
  float f_add, f_rescale;
  memcpy(&f_add, bin + 8 * words, 4);
  memcpy(&f_rescale, bin + 8 * words + 4, 4);
  const float ipf = (scal[0] * (float)ip) + (scal[1] * (float)ppc);   /* warmup_space.hpp:101 */
  const float norm = q2c[cluster];
  const float g_add = norm * norm;                                     /* slimq.h:428-437 */
  return (f_add + g_add) + (f_rescale * (ipf + scal[2]));              /* estimator.hpp:185 */
}

/* ------------------------------------------------------------ search pool -- */
/* SearchBuffer, slimq.h:80-151: linear buffer sorted by distance, capacity ef, ids carry a
 * "checked" flag in bit 31 */
typedef struct {
  float d;
  uint32_t id;
} qpair;
typedef struct {
  qpair *data;   /* capacity + 1 */
  size_t size, cur, capacity;
} qbuffer;

static size_t qb_search(const qbuffer *b, float dist) {      /* :86-96 */
  size_t lo = 0, len = b->size, half;
  while (len > 1) {
    half = len >> 1;
    len -= half;
    lo += (size_t)(b->data[lo + half - 1].d < dist) * half;
  }
  return (lo < b->size && b->data[lo].d < dist) ? lo + 1 : lo;
}
static void qb_insert(qbuffer *b, uint32_t id, float dist) { /* :112-119 */
  size_t lo = qb_search(b, dist);
  memmove(&b->data[lo + 1], &b->data[lo], (b->size - lo) * sizeof(qpair));
  b->data[lo].d = dist;
  b->data[lo].id = id;
  b->size += (size_t)(b->size < b->capacity);
  b->cur = lo < b->cur ? lo : b->cur;
}
static int qb_is_full(const qbuffer *b, float dist) {        /* :121-123 */
  return b->size == b->capacity && dist > b->data[b->size - 1].d;
}
static uint32_t qb_pop(qbuffer *b) {                         /* :126-134 */
  uint32_t id = b->data[b->cur].id;
  b->data[b->cur].id |= 1u << 31;
  ++b->cur;
  while (b->cur < b->size && (b->data[b->cur].id >> 31)) ++b->cur;
  return id;
}

/* bounded set of the k smallest (dist, id) pairs; the reference keeps a max-heap ordered by
 * distance only (slimq.h:750-757) — identical content except among exactly tied distances */
typedef struct {
  qpair *v;
  size_t size, k;
} topk;
static int pair_less(qpair a, qpair b) { return a.d < b.d || (a.d == b.d && a.id < b.id); }
static void topk_push(topk *t, qpair p) {
  if (t->k == 0) return;
  if (t->size < t->k) {
    t->v[t->size++] = p;
    return;
  }
  size_t worst = 0;
  for (size_t i = 1; i < t->size; i++)
    if (pair_less(t->v[worst], t->v[i])) worst = i;
  if (pair_less(p, t->v[worst])) t->v[worst] = p;
}
static int qpair_cmp(const void *a, const void *b) {
  const qpair *x = (const qpair *)a, *y = (const qpair *)b;
  if (x->d < y->d) return -1;
  if (x->d > y->d) return 1;
  return x->id < y->id ? -1 : (x->id > y->id ? 1 : 0);
}

/* searchKnn(q, k, result), slimq.h:1810-1924, for one query whose preparation
 * (planes, scal, q2c) is given */
static void search_one(const hsoq_index *ix, const float *raw_base, const float *q, const uint64_t *planes,
                       const float *scal, const float *q2c, size_t k, size_t ef, int order, int team,
                       uint16_t *visited, uint16_t tag, qbuffer *pool, topk *top, uint32_t *n_est,
                       uint32_t *n_hops, uint32_t *n_rerank) {
  pool->size = pool->cur = 0;                                /* :1814 */
  pool->capacity = ef;                                       /* setEf, :346-349 */
  top->size = 0;
  top->k = k;
  uint32_t ne = 0, nh = 0, nr = 0;

  uint32_t cur = ix->enterpoint;                             /* :1849-1856 */
  float curdist = hsoq_est(ix, cur, planes, scal, q2c);
  ne++;
  for (int level = ix->maxlevel; level > ix->threshold_level; level--) {   /* :1862-1901 */
    int changed = 1;
    while (changed) {
      changed = 0;
      const uint32_t *ids;
      int cnt = q_neighbors(ix, cur, level, &ids);
      if (cnt == 0) continue;
      nh++;
      ne += (uint32_t)cnt;
      for (int i = 0; i < cnt; i++) {
        float d = hsoq_est(ix, ids[i], planes, scal, q2c);
        if (d < curdist) {
          curdist = d;
          cur = ids[i];
          changed = 1;
        }
      }
    }
  }

  qb_insert(pool, cur, curdist);                             /* :1914 */
  while (pool->cur < pool->size) {                           /* searchBaseLayerST, :688-759 */
    uint32_t node = qb_pop(pool);
    if (visited[node] == tag) continue;                      /* :700-704 */
    visited[node] = tag;
    const uint32_t *ids;
    int cnt = q_neighbors(ix, node, 0, &ids);
    if (cnt == 0) continue;                                  /* :708-715: no rerank either */
    nh++;
    ne += (uint32_t)cnt;
    for (int j = 0; j < cnt; j++) {                          /* :728-746 */
      uint32_t c = ids[j];
      float d = hsoq_est(ix, c, planes, scal, q2c);
      if (qb_is_full(pool, d) || visited[c] == tag) continue;
      qb_insert(pool, c, d);
    }
    qpair p;                                                 /* :747-757 */
    p.d = hso_dist(q, raw_base + (size_t)node * ix->dim, ix->dim, HSO_L2, order, team);
    p.id = node;
    nr++;
    topk_push(top, p);
  }
  if (n_est) *n_est = ne;
  if (n_hops) *n_hops = nh;
  if (n_rerank) *n_rerank = nr;
}

int hsoq_search(const hsoq_index *ix, const float *raw_base, const float *queries, size_t nq, size_t k,
                size_t ef, int order, int team, int threads, const uint64_t *inj_planes,
                const float *inj_scal, const float *inj_q2c, uint32_t *out_labels, float *out_dists,
                uint32_t *n_est, uint32_t *n_hops, uint32_t *n_rerank) {
  if (ix->t_const <= 0 && !inj_planes) {
    snprintf(gq_err, sizeof gq_err, "hsoq_search: t_const not set");
    return -1;
  }
  if (ef == 0 || ix->n == 0) return -1;
  const size_t pw = ix->padded_dim / 64 * 4, nc = ix->num_cluster;
#ifdef _OPENMP
  if (threads <= 0) threads = omp_get_max_threads();
#else
  threads = 1;
#endif
#pragma omp parallel num_threads(threads)
  {
    uint16_t *visited = (uint16_t *)calloc(ix->n, sizeof(uint16_t));
    uint16_t tag = 0;
    qbuffer pool;
    pool.data = (qpair *)malloc((ef + 2) * sizeof(qpair));
    topk top;
    top.v = (qpair *)malloc((k + 1) * sizeof(qpair));
    float *rot = (float *)malloc(ix->padded_dim * sizeof(float));
    uint64_t *planes = (uint64_t *)malloc(pw * 8);
    float scal[3];
    float *q2c = (float *)malloc(nc * sizeof(float));
#pragma omp for schedule(dynamic, 16)
    for (long long qi = 0; qi < (long long)nq; qi++) {
      if (++tag == 0) {                                      /* visited_list_pool.h:22-28 */
        memset(visited, 0, ix->n * sizeof(uint16_t));
        tag = 1;
      }
      const float *q = queries + (size_t)qi * ix->dim;
      const uint64_t *pl = planes;
      const float *sc = scal, *qc = q2c;
      if (inj_planes) {
        pl = inj_planes + (size_t)qi * pw;
        sc = inj_scal + (size_t)qi * 3;
        qc = inj_q2c + (size_t)qi * nc;
      } else {
        hsoq_prep(ix, q, rot, planes, scal, q2c);
      }
      search_one(ix, raw_base, q, pl, sc, qc, k, ef, order, team, visited, tag, &pool, &top,
                 n_est ? n_est + qi : NULL, n_hops ? n_hops + qi : NULL, n_rerank ? n_rerank + qi : NULL);
      qsort(top.v, top.size, sizeof(qpair), qpair_cmp);
      for (size_t i = 0; i < k; i++) {
        if (i < top.size) {
          out_labels[(size_t)qi * k + i] = (uint32_t)q_label(ix, top.v[i].id);   /* :1921-1923 */
          if (out_dists) out_dists[(size_t)qi * k + i] = top.v[i].d;
        } else {
          out_labels[(size_t)qi * k + i] = 0xFFFFFFFFu;
          if (out_dists) out_dists[(size_t)qi * k + i] = INFINITY;
        }
      }
    }
    free(visited);
    free(pool.data);
    free(top.v);
    free(rot);
    free(planes);
    free(q2c);
  }
  return 0;
}
