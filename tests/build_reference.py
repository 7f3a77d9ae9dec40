"""Plain restatements of the index builder's deterministic steps, to compare the GPU builder with list by list
and bit by bit:

  convert_reference   convertFromHNSW (slim.h:867-1108) as graph_build.cpp states it: degree thresholds, first
                      prune, reverse-edge union, re-prune, hierarchical filter.  Exact int64-valued distances on
                      integer rows (float64 holds them exactly), float64 elsewhere, with an `uncertain` mask of the
                      lists whose outcome an fp32 implementation may legitimately decide otherwise.
  rotate_f32          FhtKacRotator::rotate as host_rotate computes it (bit for bit)
  rotate_f64          the same rotation in float64 (orthogonal to rounding)
  payload_reference   the 1-bit RaBitQ code and (f_add, f_rescale) of one_bit_code_with_factor, in the host's order
  read_slimq_payload  the per-node payload of an hnsw_slimq .graph (build_slimq_graph's record layout)

The fp32 error bounds are those of exact_regimes.py: an implementation that sums a distance in any order is
within (dim + 3) u d of the float64 L2 distance d and within (dim + 1) u sum|x_i y_i| + u |d| of the IP one.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from exact_regimes import U
from hnsw_slim_b200 import capi

DEFAULT_PRUNE = dict(threshold_level=0, top_degree_percent=0.02, top_M0=32, low_m0=8, top_M=16, low_m=4)
GRAM_EPS = 2.0 ** -48          # float64 rounding of the reference's own sums, relative to the squared norms


# ---------------------------------------------------------------------------------------------------------
# graphs as per-level lists
# ---------------------------------------------------------------------------------------------------------
def graph_lists(path: str, dim: int, kind: int = capi.HS_KIND_SLIM):
    """(levels[n], lists) of a .graph: lists[l] maps every node with level >= l to its level-l list."""
    g = capi.HostGraph(path, dim, kind=kind)
    n = g.info()["n"]
    levels = np.array([g.node(i)[0] for i in range(n)], dtype=np.int64)
    lists = [{int(v): g.row(int(v), l).astype(np.int64) for v in np.nonzero(levels >= l)[0]}
             for l in range(int(levels.max()) + 1)]
    return levels, lists


def build_host_pair(base, directory, *, metric: int = 0, M: int = 8, ef_construction: int = 60,
                    branching: str = "4", seed: int = 100, **prune):
    """The un-pruned HNSW file and the slim file of the same single-threaded host build (same seed, so the
    same HNSW phase): the slim lists are the host's conversion of the hnsw file's lists."""
    hp, sp = f"{directory}/hnsw.graph", f"{directory}/slim.graph"
    kw = dict(metric=metric, M=M, ef_construction=ef_construction, branching=branching, seed=seed, threads=1)
    capi.build_hnsw_graph(base, hp, **kw)
    capi.build_slim_graph(base, sp, **kw, **prune)
    return hp, sp


def list_mismatches(want, got, uncertain=None) -> list[tuple[int, int]]:
    """(node, level) whose list differs between two per-level list sets (ids and order), skipping the
    (node, level) pairs in `uncertain`."""
    assert len(want) == len(got), (len(want), len(got))
    bad = []
    for l, (a, b) in enumerate(zip(want, got)):
        assert a.keys() == b.keys(), l
        for v, lst in a.items():
            if uncertain is not None and (v, l) in uncertain:
                continue
            if not np.array_equal(lst, b[v]):
                bad.append((v, l))
    return bad


# ---------------------------------------------------------------------------------------------------------
# distances with their fp32 error bounds
# ---------------------------------------------------------------------------------------------------------
class Metric:
    def __init__(self, base: np.ndarray, metric: int):
        self.x = np.ascontiguousarray(base, dtype=np.float64)
        self.metric = metric
        self.dim = base.shape[1]
        integer = bool(np.array_equal(base, np.round(base)))
        span = max(float(base.max()), 0.0) - min(float(base.min()), 0.0)
        # integer rows with every partial sum below 2^24: fp32 distances are exact in any summation order
        self.exact = integer and self.dim * span * span < 2.0 ** 24
        if integer:
            assert self.exact, f"integer rows of span {span} in {self.dim} dims: fp32 distances are not exact"
        # rows with equal content get equal distances in every implementation (exact ties, broken by id)
        _, self.uid = np.unique(base, axis=0, return_inverse=True)
        self.uid = self.uid.reshape(-1)

    def dist(self, a: np.ndarray, b: np.ndarray):
        """float64 distances between row stacks a[..., dim] and b[..., dim] (broadcast) and their bounds."""
        if self.metric == 1:
            p = a * b
            d = 1.0 - p.sum(-1)
            if self.exact:
                return d, np.zeros_like(d)
            s = np.abs(p).sum(-1)
            return d, (self.dim + 1) * U * s + U * np.abs(d) + GRAM_EPS * s
        t = a - b
        d = (t * t).sum(-1)
        if self.exact:
            return d, np.zeros_like(d)
        return d, (self.dim + 3) * U * d + GRAM_EPS * d


def _select(mt: Metric, v: np.ndarray, cands: np.ndarray, keep: np.ndarray):
    """The relative-neighbourhood selection of slim.h:836-865 for b nodes at once: candidates in ascending
    (distance, id) order, a candidate is kept unless a kept one is strictly closer to it than v is, at most
    keep[i] kept.  cands[b, m] is -1 padded.  -> kept ids [b, m] (-1 padded, selection order), uncertain[b]:
    some comparison on the way had a gap within the fp32 bounds."""
    b, m = cands.shape
    valid = cands >= 0
    c = np.where(valid, cands, v[:, None])
    dvc, tvc = mt.dist(mt.x[c], mt.x[v][:, None, :])
    dvc = np.where(valid, dvc, np.inf)
    order = np.lexsort((np.where(valid, cands, np.iinfo(np.int64).max), dvc), axis=-1)
    cs, ds = np.take_along_axis(c, order, 1), np.take_along_axis(dvc, order, 1)
    ts, vs = np.take_along_axis(tvc, order, 1), np.take_along_axis(valid, order, 1)
    kmax = int(keep.max()) if b else 0
    kept = np.full((b, max(kmax, 1)), -1, np.int64)
    cnt = np.zeros(b, np.int64)
    unc = np.zeros(b, bool)
    consumed = np.zeros((b, m), bool)
    for j in range(m):
        act = np.nonzero(vs[:, j] & (cnt < keep))[0]
        if len(act) == 0:
            break
        consumed[act, j] = True
        cj, dj, tj = cs[act, j], ds[act, j], ts[act, j]
        kc = int(cnt[act].max())
        good = np.ones(len(act), bool)
        if kc:
            k = kept[act, :kc]
            live = np.arange(kc)[None, :] < cnt[act][:, None]
            dk, tk = mt.dist(mt.x[np.where(live, k, cj[:, None])], mt.x[cj][:, None, :])
            # a kept row with v's content is exactly as far from the candidate as v is: never strictly closer
            same = mt.uid[np.where(live, k, cj[:, None])] == mt.uid[v[act]][:, None]
            good = ~(live & ~same & (dk < dj[:, None])).any(1)
            if not mt.exact:
                unc[act] |= (live & ~same & (np.abs(dk - dj[:, None]) <= tk + tj[:, None])).any(1)
        g = act[good]
        kept[g, cnt[g]] = cs[g, j]
        cnt[g] += 1
    if not mt.exact and m > 1:
        # the (distance, id) order of the consumed prefix and of the first candidate after it
        pair = consumed[:, :-1] & vs[:, 1:]
        with np.errstate(invalid="ignore"):                     # inf - inf past the valid candidates
            near = ds[:, 1:] - ds[:, :-1] <= ts[:, 1:] + ts[:, :-1]
        same = mt.uid[cs[:, 1:]] == mt.uid[cs[:, :-1]]
        unc |= (pair & near & ~same).any(1)
    return kept, unc


def _select_lists(mt: Metric, nodes, lists, keep, budget: int = 1 << 22):
    """_select over ragged lists, batched by list length (padding stays small)."""
    out: list = [None] * len(nodes)
    unc = np.zeros(len(nodes), bool)
    lens = np.array([len(x) for x in lists], np.int64)
    for lo in sorted({1 << int(np.ceil(np.log2(max(1, k)))) for k in lens}):
        idx = np.nonzero((lens <= lo) & (lens > lo // 2) if lo > 1 else lens <= 1)[0]
        step = max(1, budget // (lo * mt.dim))
        for s in range(0, len(idx), step):
            part = idx[s:s + step]
            cand = np.full((len(part), lo), -1, np.int64)
            for r, i in enumerate(part):
                cand[r, :lens[i]] = lists[i]
            kept, u = _select(mt, np.asarray(nodes, np.int64)[part], cand, np.asarray(keep, np.int64)[part])
            unc[part] = u
            for r, i in enumerate(part):
                out[i] = kept[r][kept[r] >= 0]
    return out, unc


@dataclass
class Converted:
    lists: list          # [l] {node: final list}
    first: list          # [l] {node: list after the first prune}
    merged: list         # [l] {node: size of the reverse-edge union}
    uncertain: set       # {(node, level)}
    thresholds: list     # [l] degree threshold


def convert_reference(levels, lists, base, metric: int, params: dict) -> Converted:
    """convertFromHNSW over HNSW lists[l] {node: ids} of nodes with levels[node] >= l (graph_lists of an
    hs_build_hnsw_graph file).  params: maxM, maxM0 and the pruning parameters (DEFAULT_PRUNE's names).

    A list is uncertain if one of its own comparisons (first prune or re-prune) had a float64 gap within the
    summed fp32 bounds, or if a node that has it among its HNSW candidates had an uncertain first prune (its
    reverse edge may go either way).  On exact (integer) data nothing is uncertain."""
    p = dict(DEFAULT_PRUNE, **params)
    mt = Metric(base, metric)
    levels = np.asarray(levels)
    maxM, maxM0 = int(p["maxM"]), int(p["maxM0"])
    res = Converted([], [], [], set(), [])
    for l, H in enumerate(lists):
        nodes = sorted(H)
        cnt = np.array([len(H[v]) for v in nodes], np.int64)
        # degree threshold (slim.h:905-947): level 0 never counts its population, so topN = 0 and the
        # threshold lands on maxM0 + 1; above, the top `pct` of the level's nodes by out-degree
        if l == 0:
            thr = maxM0 + 1
        else:
            hist = np.bincount(np.minimum(cnt, maxM0 + 1), minlength=maxM0 + 2)
            top_n = int(float(np.float32(len(nodes)) * np.float32(p["top_degree_percent"])) + 0.5)
            thr, acc = 0, 0
            for d in range(maxM0 + 1, 0, -1):
                acc += int(hist[d])
                if acc >= top_n:
                    thr = d
                    break
        res.thresholds.append(thr)
        hi, lo_ = (p["top_M0"], p["low_m0"]) if l == 0 else (p["top_M"], p["low_m"])
        keep = np.where(cnt > thr, hi, lo_)
        first, unc1 = _select_lists(mt, nodes, [H[v] for v in nodes], keep)
        rev: dict = {v: [] for v in nodes}
        for v, f in zip(nodes, first):
            for u in f.tolist():
                rev[u].append(v)
        # the union sorted by id (slim.h:985-1011), re-pruned above maxM0 / maxM (:1036-1058)
        merged = [np.unique(np.concatenate([f, np.asarray(rev[v], np.int64)])) for v, f in zip(nodes, first)]
        res.merged.append({v: len(mg) for v, mg in zip(nodes, merged)})
        limit = maxM0 if l == 0 else maxM
        big = [i for i, mg in enumerate(merged) if len(mg) > limit]
        unc2 = np.zeros(len(nodes), bool)
        if big:
            kept, u2 = _select_lists(mt, [nodes[i] for i in big], [merged[i] for i in big], [limit] * len(big))
            for i, k, u in zip(big, kept, u2):
                merged[i], unc2[i] = k, u
        # hierarchical pruning (:1063-1084): away from threshold_level keep neighbours whose top level is l
        final = {}
        for v, lst in zip(nodes, merged):
            if l != p["threshold_level"]:
                lst = lst[levels[lst] == l]
            final[v] = lst
        res.lists.append(final)
        res.first.append(dict(zip(nodes, first)))
        for i, v in enumerate(nodes):
            if unc1[i] or unc2[i]:
                res.uncertain.add((v, l))
            if unc1[i]:
                res.uncertain.update((int(u), l) for u in H[v])
    return res


# ---------------------------------------------------------------------------------------------------------
# hnsw_slimq payload
# ---------------------------------------------------------------------------------------------------------
def rotation_shape(dim: int):
    """(padded_dim, trunc_dim) of the RaBitQ rotation (hnsw.hpp:424-427, rotator.hpp:233-235)."""
    td = 1
    while td * 2 <= dim:
        td *= 2
    return (dim + 63) // 64 * 64, td


def _rotate(x, dim, pd, flip, dt, fac):
    td = rotation_shape(dim)[1]
    x = np.asarray(x)
    n = x.shape[0]
    out = np.zeros((n, pd), dt)
    out[:, :dim] = x
    bits = np.unpackbits(np.asarray(flip, np.uint8), bitorder="little").reshape(4, pd).astype(bool)
    pow2, start = td == pd, pd - td
    for r in range(4):
        out[:, bits[r]] = -out[:, bits[r]]
        s0 = start if (not pow2 and r & 1) else 0
        seg = out[:, s0:s0 + td].copy()
        h = 1
        while h < td:                      # one IEEE add / sub per butterfly: the order does not matter
            v = seg.reshape(n, td // (2 * h), 2, h)
            a, b = v[:, :, 0, :].copy(), v[:, :, 1, :].copy()
            v[:, :, 0, :] = a + b
            v[:, :, 1, :] = a - b
            h *= 2
        out[:, s0:s0 + td] = seg * fac
        if not pow2:
            a, b = out[:, :pd // 2].copy(), out[:, pd // 2:].copy()
            out[:, :pd // 2] = a + b
            out[:, pd // 2:] = a - b
    if not pow2:
        out *= dt(0.25)
    return out


def rotate_f32(x, dim: int, pd: int, flip) -> np.ndarray:
    """FhtKacRotator::rotate exactly as host_rotate (graph_build.cpp) computes it in fp32."""
    td = rotation_shape(dim)[1]
    return _rotate(np.asarray(x, np.float32), dim, pd, flip, np.float32, np.float32(1.0) / np.sqrt(np.float32(td)))


def rotate_f64(x, dim: int, pd: int, flip) -> np.ndarray:
    """The same rotation in float64 (an orthogonal map: norms and inner products are preserved)."""
    td = rotation_shape(dim)[1]
    return _rotate(np.asarray(x, np.float64), dim, pd, flip, np.float64, 1.0 / np.sqrt(td))


def rotation_bound(x, dim: int) -> np.ndarray:
    """Bound on the 2-norm (so on every coordinate) of rotate_f32(x) - rotate_f64(x), per row: four rounds of
    log2(td) butterfly levels, the scale (with its own rounding) and the half-sum step, u relative each."""
    td = rotation_shape(dim)[1]
    ops = 4 * (int(np.log2(td)) + 3)
    return 2 * ops * U * np.linalg.norm(np.asarray(x, np.float64), axis=1)


def pack_codes(bits: np.ndarray) -> np.ndarray:
    """[n, pd] bool -> [n, pd / 64] uint64, dimension 64w + j at bit 63 - j (pack_binary, space.hpp:272-286)."""
    n, pd = bits.shape
    by = np.packbits(bits.reshape(n, pd // 64, 64), axis=-1, bitorder="big")
    return np.ascontiguousarray(by).view(">u8").reshape(n, pd // 64).astype(np.uint64)


def payload_reference(rot32: np.ndarray, rcent: np.ndarray, cluster) -> dict:
    """one_bit_code_with_factor (rabitq_impl.hpp:76-135, L2) as build_slimq_graph computes it: fp32 residual
    against the rotated centroid, sign bits, and the three sums in double, left to right."""
    cen = np.asarray(rcent, np.float32)[np.asarray(cluster, np.int64)]
    res = (np.asarray(rot32, np.float32) - cen).astype(np.float32)
    bits = res > 0
    xu = np.where(bits, 0.5, -0.5)
    r = res.astype(np.float64)
    l2 = np.cumsum(r * r, axis=1)[:, -1]
    ip_resi = np.cumsum(r * xu, axis=1)[:, -1]
    ip_cent = np.cumsum(cen.astype(np.float64) * xu, axis=1)[:, -1]
    ip_resi = np.where(ip_resi == 0, np.inf, ip_resi)
    with np.errstate(invalid="ignore"):
        f_add = (l2 + 2 * l2 * ip_cent / ip_resi).astype(np.float32)
        f_rescale = (-2 * l2 / ip_resi).astype(np.float32)
    return {"codes": pack_codes(bits), "f_add": f_add, "f_rescale": f_rescale,
            "cluster": np.asarray(cluster, np.uint32), "residual": res}


def nearest_centroid(base, centroids):
    """float64 nearest centroid (first minimum) and, per row, the gap to the nearest centroid of different
    content and the fp32 bound of the two distances: the argmin is only binding where gap > bound."""
    x = np.asarray(base, np.float64)
    uc, inv = np.unique(np.asarray(centroids), axis=0, return_inverse=True)
    c = uc.astype(np.float64)
    nx, nc = (x * x).sum(1), (c * c).sum(1)
    d = np.maximum(nx[:, None] + nc[None, :] - 2 * (x @ c.T), 0)    # exact on integer rows
    full = d[:, inv.reshape(-1)]                                    # duplicated centroids: identical columns
    arg = np.argmin(full, axis=1)
    if d.shape[1] == 1:                                             # one centroid content: nothing to confuse
        return arg.astype(np.uint32), np.full(len(x), np.inf), np.zeros(len(x))
    two = np.sort(d, axis=1)[:, :2]
    mt = Metric(np.concatenate([np.asarray(base), np.asarray(centroids)]), 0)
    if mt.exact:
        bound = np.zeros(len(x))
    else:
        bound = (x.shape[1] + 3) * U * (two[:, 0] + two[:, 1]) + 8 * GRAM_EPS * (nx + nc.max())
    return arg.astype(np.uint32), two[:, 1] - two[:, 0], bound


def read_slimq_payload(path: str) -> dict:
    """The payload build_slimq_graph writes (slimq.h:1161-1216 layout): rotated centroids, rotator flip bytes,
    per node cluster id, code words (MSB-first uint64), f_add, f_rescale, f_error."""
    raw = open(path, "rb").read()
    n, rec = (int(v) for v in np.frombuffer(raw, np.uint64, 2, 0))
    o = 48 + 12 + 32 + 1
    meta = np.frombuffer(raw, np.uint64, 9, o)
    o += 72 + 1
    nc, pd, off_cluster, off_bin = int(meta[0]), int(meta[2]), int(meta[3]), int(meta[4])
    words = pd // 64
    cent = np.frombuffer(raw, np.float32, nc * pd, o).reshape(nc, pd).copy()
    o += nc * pd * 4
    flip = np.frombuffer(raw, np.uint8, 4 * pd // 8, o).copy()
    o += 4 * pd // 8
    el = np.frombuffer(raw, np.uint8, n * rec, o).reshape(n, rec)
    fac = el[:, off_bin + 8 * words:off_bin + 8 * words + 12].copy().view(np.float32)
    return {"codes": el[:, off_bin:off_bin + 8 * words].copy().view(np.uint64),
            "f_add": fac[:, 0].copy(), "f_rescale": fac[:, 1].copy(), "f_error": fac[:, 2].copy(),
            "cluster": el[:, off_cluster:off_cluster + 4].copy().view(np.uint32)[:, 0].copy(),
            "centroids": cent, "flip": flip}


def ulp_distance(a, b) -> np.ndarray:
    """|a - b| in units in the last place of float32 (sign-magnitude order; +0 and -0 are 0 apart)."""
    def key(x):
        i = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))
