"""Float64 restatement of the hnsw_slimq query side, to judge traverse_slimq.cu and oracle/hs_oracle_slimq.c by
something neither of them was written next to:

  query_codes      the 4-bit code per dimension of an fp32 rotated query (prepare_query; rabitq_impl.hpp:386-429,
                   553-555) with the quantiser's ratio taken in float64, and a mask of the dimensions whose code an
                   fp32 norm may round either way
  pack_planes      the bit-plane layout: dimension 64 w + l is bit 63 - l of word w, plane j of word w is word 4 w + j
  query_scalars    delta, vl, k1xsumq and the centroid distances q2c in float64, each with the error bound of the
                   fp32 chain that computes it
  estimate         f_add + q2c^2 + f_rescale (delta ip + vl ppc + k1xsumq) in float64 with exact integer ip and ppc,
                   and the bound of its fp32 chain
  true_l2          the float64 distance the estimate estimates

The rotation (rotate_f32, rotate_f64) and the payload reader are build_reference.py's.

An all-zero query (or one whose squares underflow) has norm 0.  The reference's fp32 path then divides 0 by 0;
this module states the project's choice instead: the quantiser uses |r| unnormalised and cosv = 0, so delta = vl = 0.
"""
from __future__ import annotations

import numpy as np

from build_reference import pack_codes, rotate_f32
from exact_regimes import U
from hnsw_slim_b200 import capi
from oracle import refharness as rh

NUM_BITS = 4          # query code width (query.hpp:126): one sign bit and three ex bits
CB = -7.5             # -(2^3 - 0.5): the code's centre (rabitq_impl.hpp:557-559)


def sum_depth(pd: int) -> int:
    """Rounding depth of a sum in the kernels' "warp order": pd / 32 terms per lane, then 5 butterfly levels."""
    return -(-pd // 32) + 5


def fp32_norm_is_zero(rot32) -> np.ndarray:
    """Per row: the fp32 sum of squares is 0, i.e. every r_i^2 rounds to zero (|r_i| <= 2^-75)."""
    r = np.asarray(rot32, np.float32).astype(np.float64)
    return (r.reshape(-1, r.shape[-1]) ** 2 <= 2.0 ** -150).all(1)


def query_codes(rot32, t_const: float):
    """-> codes[nq, pd] int64 (0..15), mask[nq, pd] bool.

    mask marks the dimensions where t_const * |r| / |r| + 1e-5 lies so close to an integer 1..7 that the fp32 norm
    (relative error (depth / 2 + 1) u) and the fp32 division (u) may put the truncation on either side.  Above 8 the
    code saturates at 7 either way."""
    r = np.asarray(rot32, np.float32).astype(np.float64)
    r = r.reshape(-1, r.shape[-1])
    pd = r.shape[1]
    norm = np.where(fp32_norm_is_zero(r)[:, None], 0.0, np.sqrt((r * r).sum(1, keepdims=True)))
    a = np.abs(r)
    with np.errstate(invalid="ignore", divide="ignore"):
        o = np.where(norm > 0, a / norm, a)
    v = t_const * o + 1e-5
    c = np.minimum(np.floor(v).astype(np.int64), 7)
    c = np.where(r < 0, 7 - c, c)
    codes = c + np.where(r > 0, 8, 0)
    rel = 2 * (sum_depth(pd) / 2 + 2) * U
    near = np.rint(v)
    mask = (np.abs(v - near) <= rel * v + 1e-12) & (near >= 1) & (near <= 7) & (norm > 0)
    return codes, mask


def pack_planes(codes) -> np.ndarray:
    """codes[nq, pd] -> planes[nq, pd / 64 * 4] uint64 (new_transpose_bin, space.hpp:1405-1516)."""
    codes = np.asarray(codes, np.int64)
    nq, pd = codes.shape
    w = pd // 64
    pl = np.stack([pack_codes(((codes >> j) & 1).astype(bool)) for j in range(NUM_BITS)], axis=-1)
    return pl.reshape(nq, w * NUM_BITS)


def unpack_planes(planes, pd: int) -> np.ndarray:
    """The inverse of pack_planes: planes[nq, pd / 64 * 4] -> codes[nq, pd]."""
    planes = np.asarray(planes, np.uint64).reshape(-1, pd // 64, NUM_BITS)
    codes = np.zeros((planes.shape[0], pd), np.int64)
    for j in range(NUM_BITS):
        codes |= unpack_codes(planes[:, :, j]).astype(np.int64) << j
    return codes


def unpack_codes(words) -> np.ndarray:
    """[n, pd / 64] uint64 (dimension 64 w + l at bit 63 - l) -> [n, pd] bool."""
    words = np.ascontiguousarray(words, np.uint64)
    by = words.astype(">u8").view(np.uint8).reshape(words.shape[0], -1)
    return np.unpackbits(by, axis=1, bitorder="big").astype(bool)


def query_scalars(rot32, codes, centroids) -> dict:
    """delta, vl, k1xsumq [nq] and q2c [nq, nc] in float64 from the fp32 rotated query, its codes and the rotated
    centroids, with the error bounds (same keys + "_bound") of fp32 chains that compute them in warp order.

    The bounds are first-order sums of u per rounding, doubled for the second-order terms:
      k1xsumq  a depth-d sum of pd terms of either sign: d u sum|r|
      delta    <r, ucb> / |ucb|^2 with every product r_i ucb_i >= 0 (no cancellation) and |ucb|^2 exact in fp32:
               (d + 6) u relative (the norm of r appears twice and cancels to first order)
      q2c      sqrt of a depth-d sum of squared fp32 differences: (d / 2 + 3) u relative"""
    r = np.asarray(rot32, np.float32).astype(np.float64).reshape(len(codes), -1)
    pd = r.shape[1]
    d = sum_depth(pd)
    ucb = np.asarray(codes, np.float64) + CB
    delta = np.where(~fp32_norm_is_zero(r), (r * ucb).sum(1) / (ucb * ucb).sum(1), 0.0)
    vl = delta * CB
    k1 = -0.5 * r.sum(1)
    c = np.asarray(centroids, np.float32).astype(np.float64)
    q2c = np.stack([np.sqrt(((c - row) ** 2).sum(1)) for row in r])
    rd = 2 * (d + 6) * U * np.abs(delta)
    return {"delta": delta, "vl": vl, "k1xsumq": k1, "q2c": q2c,
            "delta_bound": rd, "vl_bound": 7.5 * rd + U * np.abs(vl),
            "k1xsumq_bound": 2 * d * U * 0.5 * np.abs(r).sum(1) + U * np.abs(k1),
            "q2c_bound": 2 * (d / 2 + 3) * U * q2c + 1e-300}


def check_preparation(q, dim: int, payload: dict, t_const: float, rot, planes, scal, q2c) -> int:
    """Asserts that one implementation's per-query preparation (hs_slimq_prepare or OracleQ.prep) is the reference's:
    rotation equal to rotate_f32 bit for bit, plane codes equal outside the mask, scalars and q2c within their
    float64 bounds (computed with the implementation's own codes on the masked dimensions).  -> masked dimensions."""
    pd = payload["centroids"].shape[1]
    want = rotate_f32(q, dim, pd, payload["flip"])
    assert np.array_equal(np.asarray(rot, np.float32).view(np.uint32), want.view(np.uint32)), "rotation"
    codes, mask = query_codes(want, t_const)
    got = unpack_planes(planes, pd)
    bad = (got != codes) & ~mask
    assert not bad.any(), f"plane codes differ at {np.argwhere(bad)[:8].tolist()}"
    s = query_scalars(want, np.where(mask, got, codes), payload["centroids"])
    for i, key in enumerate(("delta", "vl", "k1xsumq")):
        err = np.abs(np.asarray(scal, np.float64)[:, i] - s[key])
        assert (err <= s[key + "_bound"]).all(), (key, (err / np.maximum(s[key + "_bound"], 1e-300)).max())
    err = np.abs(np.asarray(q2c, np.float64) - s["q2c"])
    assert (err <= s["q2c_bound"]).all(), ("q2c", (err / np.maximum(s["q2c_bound"], 1e-300)).max())
    return int(mask.sum())


def ip_ppc(data_codes, qcodes) -> tuple[np.ndarray, np.ndarray]:
    """Exact ip = sum_i bit_i(x) qcode_i and ppc = popcount(x) of node codes [n, pd / 64] against one query's
    codes [pd]."""
    bits = unpack_codes(data_codes).astype(np.int64)
    return bits @ np.asarray(qcodes, np.int64), bits.sum(1)


def estimate(f_add, f_rescale, cluster, ip, ppc, delta, vl, k1xsumq, q2c):
    """-> (est, bound) per node: the estimator (split_single_estdist, estimator.hpp:164-188; the L2 branch of
    get_bin_est, slimq.h:408-440) in float64 for the given per-query scalars and q2c[cluster], and the bound of the
    fp32 chain (q2c * q2c; delta ip + vl ppc; + k1; * f_rescale; f_add + g; + the product) that computes it from
    the same inputs: the terms cancel, so 5 u times the sum of their magnitudes."""
    fa = np.asarray(f_add, np.float64)
    fr = np.asarray(f_rescale, np.float64)
    g = np.asarray(q2c, np.float64)[np.asarray(cluster, np.int64)] ** 2
    ip, ppc = np.asarray(ip, np.float64), np.asarray(ppc, np.float64)
    inner = delta * ip + vl * ppc + k1xsumq
    est = fa + g + fr * inner
    mag = np.abs(fa) + g + np.abs(fr) * (abs(delta) * ip + abs(vl) * ppc + abs(k1xsumq))
    return est, 5 * U * mag


def assign_centroids(base, nc: int, seed: int = 1):
    """-> (centroids[nc, dim], cluster ids[n]).  Up to 64 clusters: Lloyd k-means (refharness.kmeans).  More: nc
    centroids drawn from the rows, so some rows equal their centroid (zero residual, f_rescale = -0), and the
    float64 nearest centroid of every row."""
    base = np.asarray(base, np.float32)
    if nc <= 64:
        return rh.kmeans(base, nc, seed=seed)
    cen = base[np.random.default_rng(seed).choice(len(base), nc, replace=False)].copy()
    x, c = base.astype(np.float64), cen.astype(np.float64)
    d = (x * x).sum(1)[:, None] + (c * c).sum(1)[None] - 2 * x @ c.T
    return cen, np.argmin(d, axis=1).astype(np.uint32)


def host_index(path: str, base, nc: int, *, M: int = 8, ef_construction: int = 64, **kw):
    """Single-threaded host build (hs_build_slimq_graph) with assign_centroids' centroids -> (centroids, cluster)."""
    cen, cid = assign_centroids(base, nc)
    capi.build_slimq_graph(base, path, M=M, ef_construction=ef_construction, centroids=cen, cluster_ids=cid,
                           threads=1, **kw)
    return cen, cid


def true_l2(base, q, ids) -> np.ndarray:
    """float64 |x_id - q|^2."""
    x = np.asarray(base, np.float64)[np.asarray(ids, np.int64)]
    return ((x - np.asarray(q, np.float64)) ** 2).sum(-1)


def relative_error_stats(est, exact) -> tuple[float, float]:
    """(mean, rms) of (est - d) / d over the pairs with d > 0."""
    est, exact = np.asarray(est, np.float64).ravel(), np.asarray(exact, np.float64).ravel()
    keep = exact > 0
    e = (est[keep] - exact[keep]) / exact[keep]
    return float(e.mean()), float(np.sqrt((e * e).mean()))


def statistics_hold(est, exact, pd: int) -> bool:
    """The estimator is unbiased to 1 % and its rms relative error is below 1.2 / sqrt(padded_dim) (measured about
    0.75 / sqrt(padded_dim) on latent data at dims 64 to 2048)."""
    mean, rms = relative_error_stats(est, exact)
    return abs(mean) <= 0.01 and rms <= 1.2 / np.sqrt(pd)
