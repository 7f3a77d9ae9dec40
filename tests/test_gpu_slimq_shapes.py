"""GPU: traverse_slimq.cu across padded dims, degrees, cluster counts and all 16 dispatch variants, against the C
oracle (bit for bit) and the float64 query-side reference of slimq_reference.py.

Every index is a single-threaded host build (hs_build_slimq_graph).  Per case the search must equal the oracle on
>= 99.5 % of the rows (ids, distance bits and counters; not counters on copies data, whose estimates tie bit for
bit and are ordered differently), its rows must be sorted, each returned distance must be the
exact distance of its row within the fp32 bound, and its recall must be within 0.01 of the oracle's.

The zero query has norm 0.  The reference divides 0 by 0 there; the kernel and the oracle take cosv = 0 instead
(see prepare_query).  Queries that overflow the fp32 norm (coordinates around 1e19 and above) still give NaN
estimates and are out of scope."""
import numpy as np
import pytest

from build_reference import read_slimq_payload, rotate_f32, rotation_shape
from exact_regimes import U, make_regime
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset
from oracle import refharness as rh
from slimq_reference import check_preparation, host_index
from test_gpu_slimq import check_against_oracle

pytestmark = pytest.mark.gpu

HS_ERR_UNSUPPORTED = -5
NQ = 200


# the kernel's dispatch (traverse_slimq.cu), restated: WREG x SLOTS x KREG
def wreg_variant(words):
    return 2 if words == 2 else 0


def slots_variant(ef):
    return 2 if ef <= 64 else (4 if ef <= 128 else (8 if ef <= 256 else 0))


def kreg_variant(k):
    return 1 if k <= 32 else 0


ALL_VARIANTS = [(1, 40), (40, 50), (10, 100), (64, 120), (10, 200), (100, 250), (10, 300), (50, 400)]

# name: (regime, n, dim, clusters, M, build parameters, [(k, ef), ...])
CASES = {
    "w1-d64": ("latent", 3000, 64, 16, 16, {}, ALL_VARIANTS),
    "w2-d96-M8": ("latent", 3000, 96, 16, 8, {}, ALL_VARIANTS),
    "w3-d130-M32": ("latent", 3000, 130, 16, 32, {}, [(10, 40), (10, 200), (100, 250), (10, 300)]),
    "w2-d128-M48": ("latent", 3000, 128, 16, 48, {}, [(10, 100), (40, 300)]),
    "w15-d960": ("latent", 3000, 960, 16, 16, {}, [(10, 100), (40, 64)]),
    "w16-d1000-c1": ("latent", 3000, 1000, 1, 16, {}, [(10, 50), (10, 150)]),
    "w32-d2048-c4096": ("latent", 5000, 2048, 4096, 16, {}, [(10, 100)]),
    "w2-d96-c4096": ("latent", 5000, 96, 4096, 16, {}, [(10, 100)]),
    "threshold1": ("latent", 3000, 96, 16, 16, dict(threshold_level=1), [(10, 60)]),
    "threshold2-e": ("latent", 3000, 200, 16, 16, dict(threshold_level=2, branching="e"), [(10, 60)]),
    "sqrt": ("latent", 3000, 96, 16, 16, dict(branching="sqrt"), [(10, 60)]),
    "labels-perm": ("latent", 3000, 96, 16, 16, dict(labels="perm"), [(10, 60)]),
    "copies": ("copies", 3000, 200, 16, 16, {}, [(10, 100)]),
    "integer": ("integer", 3000, 96, 16, 16, {}, [(10, 100)]),
    # ef = 1, ef < k (padded rows), ef == k, ef > n
    "ef-edges": ("latent", 500, 200, 16, 16, {}, [(1, 1), (10, 3), (20, 20), (10, 600)]),
}


class Built:
    def __init__(self, name, directory):
        regime, n, dim, nc, M, kw, self.pairs = CASES[name]
        kw = dict(kw)
        self.base, self.q = make_regime(regime, n, NQ, dim, seed=5)
        self.labels = np.arange(n, dtype=np.uint64)
        if kw.pop("labels", None) == "perm":
            self.labels = np.random.default_rng(2).permutation(n).astype(np.uint64)
            kw["labels"] = self.labels
        self.path = f"{directory}/q.graph"
        self.cen, self.cid = host_index(self.path, self.base, nc, M=M, **kw)
        self.dim, self.n = dim, n
        self.ix = capi.Index(self.path, dim, kind=capi.HS_KIND_SLIMQ, raw_base=self.base)
        self.o = rh.OracleQ(self.path, self.base, t_const=self.ix.query_tconst)
        self.pay = read_slimq_payload(self.path)


_built = {}


def built(name, tmp_path_factory):
    if name not in _built:
        _built.clear()                                    # one device index at a time
        _built[name] = Built(name, tmp_path_factory.mktemp(name))
    return _built[name]


def test_cases_reach_every_dispatch_variant():
    seen = {(wreg_variant(rotation_shape(c[2])[0] // 64), slots_variant(ef), kreg_variant(k))
            for c in CASES.values() for k, ef in c[6]}
    assert seen == {(w, s, k) for w in (0, 2) for s in (2, 4, 8, 0) for k in (0, 1)}


def exact_knn(base, q, k):
    x, y = base.astype(np.float64), q.astype(np.float64)
    d = (y * y).sum(1)[:, None] + (x * x).sum(1)[None] - 2 * y @ x.T
    return np.argsort(d, axis=1, kind="stable")[:, :k]


def recall(rows, gt):
    return float(np.mean([len(set(a[a >= 0]) & set(b)) / len(b) for a, b in zip(rows, gt)]))


@pytest.mark.parametrize("name", list(CASES))
def test_search_against_oracle_and_exact_distances(name, tmp_path_factory):
    b = built(name, tmp_path_factory)
    inv = np.empty(b.n, np.int64)
    inv[b.labels.astype(np.int64)] = np.arange(b.n)
    for k, ef in b.pairs:
        if name == "copies":
            # equal rows have equal codes and estimates: the kernel orders tied pool entries by id, the oracle's sorted
            # buffer puts the newest first, so the expansion order (and the counters) of a tied row may differ
            b.ix.set_ef(ef)
            lab, dist = b.ix.search(b.q, k)
        else:
            lab, dist = check_against_oracle(b.ix, b.o, b.q, k, ef)
        olab, odist, _, _, onr = b.o.search(b.q, k, ef, order=rh.ORDER_GPU, team=32)
        same = np.all(lab == olab, axis=1)
        assert same.mean() >= 0.995
        assert np.array_equal(dist[same].view(np.uint32), odist[same].view(np.uint32))
        same = same.mean()
        valid = lab != 0xFFFFFFFF
        assert np.array_equal(valid, np.isfinite(dist))
        assert np.array_equal(valid.sum(1), np.minimum(onr, k))        # the k closest of the expanded nodes
        padded = np.where(valid, dist, np.inf)
        assert np.array_equal(np.sort(padded, axis=1), padded)          # sorted, padding last
        rows = np.where(valid, inv[np.where(valid, lab, 0).astype(np.int64)], -1)
        for i in range(len(b.q)):
            r = rows[i][valid[i]]
            assert len(set(r.tolist())) == len(r)
            d64 = ((b.base[r].astype(np.float64) - b.q[i].astype(np.float64)) ** 2).sum(1)
            assert (np.abs(dist[i][valid[i]] - d64) <= (b.dim + 3) * U * d64).all(), (i, k, ef)
        orows = np.where(olab != 0xFFFFFFFF, inv[np.where(olab != 0xFFFFFFFF, olab, 0).astype(np.int64)], -1)
        gt = exact_knn(b.base, b.q, k)
        rg, ro = recall(rows, gt), recall(orows, gt)
        print(f"{name} k={k} ef={ef}: {same:.4f} of rows identical to the oracle, recall {rg:.4f} (oracle {ro:.4f})")
        assert abs(rg - ro) <= 0.01


PREP = ["w1-d64", "w2-d96-M8", "w3-d130-M32", "threshold2-e", "w15-d960", "w16-d1000-c1", "w32-d2048-c4096"]


@pytest.mark.parametrize("name", PREP)
def test_preparation_equals_oracle_and_reference(name, tmp_path_factory):
    b = built(name, tmp_path_factory)
    edge = np.stack([np.zeros(b.dim, np.float32), b.base[3], b.cen[0], np.full(b.dim, 0.5, np.float32)])
    q = np.concatenate([b.q[:32], edge])
    rot, planes, scal, q2c = b.ix.slimq_prepare(q)
    orot, oplanes, oscal, oq2c = b.o.prep(q)
    pd = rotation_shape(b.dim)[0]
    assert np.array_equal(rot.view(np.uint32), rotate_f32(q, b.dim, pd, b.pay["flip"]).view(np.uint32))
    assert np.array_equal(rot.view(np.uint32), orot.view(np.uint32))
    assert np.array_equal(planes, oplanes)
    assert np.array_equal(scal.view(np.uint32), oscal.view(np.uint32))
    assert np.array_equal(q2c.view(np.uint32), oq2c.view(np.uint32))
    masked = check_preparation(q, b.dim, b.pay, b.ix.query_tconst, rot, planes, scal, q2c)
    print(f"{name}: {masked} masked plane dimensions of {q.shape[0] * pd}")
    assert np.isfinite(scal).all() and scal[32, 0] == 0            # the zero query
    assert q2c[34, 0] == 0                                           # the centroid query: g2c = 0


@pytest.mark.parametrize("name", ["w2-d96-M8", "w15-d960", "w32-d2048-c4096"])
def test_query_edge_cases(name, tmp_path_factory):
    """The zero query, a base row (distance 0 first), a centroid and a constant query: each row equals the oracle's
    and holds k valid labels; the zero query's recall against float64 brute force is that of an ordinary query."""
    b = built(name, tmp_path_factory)
    k, ef = 10, 100
    edge = np.stack([np.zeros(b.dim, np.float32), b.base[3], b.cen[0], np.full(b.dim, 0.5, np.float32)])
    b.ix.set_ef(ef)
    lab, dist = b.ix.search(edge, k)
    olab, odist, *_ = b.o.search(edge, k, ef, order=rh.ORDER_GPU, team=32)
    print(f"{name} zero query row: {lab[0].tolist()} {dist[0].tolist()}")
    assert np.array_equal(lab, olab) and np.array_equal(dist.view(np.uint32), odist.view(np.uint32))
    assert (lab != 0xFFFFFFFF).all() and np.isfinite(dist).all()
    assert dist[1, 0] == 0 and (b.base[lab[1, 0]] == b.base[3]).all()
    gt = exact_knn(b.base, np.concatenate([b.q[:50], edge[:1]]), k)
    lq, _ = b.ix.search(b.q[:50], k)
    ordinary = [recall(lq[i:i + 1].astype(np.int64), gt[i:i + 1]) for i in range(50)]
    assert recall(lab[:1].astype(np.int64), gt[50:]) >= np.quantile(ordinary, 0.1), ordinary


def test_gpu_built_index_prepares_like_the_host_one(tmp_path):
    """hs_build_slimq_index_gpu sets its index up separately (adopt_device_graph): same rotator, centroids, t_const
    and therefore the same preparation, bit for bit, as the host build with the same centroids and seed."""
    for dim in (96, 200, 1000):
        base, q = make_dataset(2000, 32, dim, rank=10, seed=dim)
        path = str(tmp_path / f"h{dim}.graph")
        cen, cid = host_index(path, base, 16, M=16, ef_construction=64)
        host = capi.Index(path, dim, kind=capi.HS_KIND_SLIMQ, raw_base=base)
        dev = capi.Index.build_gpu(base, kind=capi.HS_KIND_SLIMQ, centroids=cen, M=16, ef_construction=64)
        assert dev.query_tconst == host.query_tconst
        for a, c in zip(dev.slimq_prepare(q), host.slimq_prepare(q)):
            assert np.array_equal(a.view(np.uint32 if a.dtype == np.float32 else np.uint64),
                                  c.view(np.uint32 if c.dtype == np.float32 else np.uint64))


def test_dim_above_2048_is_refused_at_load(tmp_path):
    for dim in (2049, 2112):
        base, _ = make_dataset(300, 1, dim, rank=10, seed=1)
        path = str(tmp_path / f"q{dim}.graph")
        capi.build_slimq_graph(base, path, M=8, ef_construction=32, threads=1)
        with pytest.raises(capi.HsError) as e:
            capi.Index(path, dim, kind=capi.HS_KIND_SLIMQ, raw_base=base)
        assert e.value.code == HS_ERR_UNSUPPORTED


def test_largest_working_set(tmp_path_factory):
    """ef = k = 4096 (the caps of hs_set_ef and the search) at dim 2048 with 4096 clusters: shared-memory pool and
    top-k, 8 KB query buffer, 16 KB of centroid distances and 1 KB of planes per warp (about 91 KB)."""
    b = built("w32-d2048-c4096", tmp_path_factory)
    check_against_oracle(b.ix, b.o, b.q[:8], 4096, 4096, min_exact=1.0)
    with pytest.raises(capi.HsError):
        b.ix.set_ef(4097)
    b.ix.set_ef(100)
    with pytest.raises(capi.HsError):
        b.ix.search(b.q[:1], 4097)
