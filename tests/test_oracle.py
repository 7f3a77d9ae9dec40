"""CPU suite, part 1: the plain-C oracle (oracle/hs_oracle.c) is pinned to the reference.

* against the committed golden vectors in tests/golden/ (generated from the reference itself by
  tests/golden/make_golden.py) — always runs;
* against the live reference (oracle/_ref, compiled unmodified from /root/reference) on a bigger
  corpus — runs wherever that library exists.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, get_corpus, needs_ref
from oracle import refharness as rh

FIXTURES = [("slim_l2_2k", 0), ("slim_ip_1k", 1)]
EFS = (10, 40, 100)


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return z, os.path.join(GOLDEN, name + ".graph")


@pytest.mark.parametrize("name,metric", FIXTURES)
def test_golden_header_and_accessors(name, metric):
    z, graph = _load(name)
    orc = rh.Oracle(graph, int(z["dim"]), metric)
    info = orc.info()
    n, maxlevel, ep, maxM, maxM0, M = [int(x) for x in z["info"]]
    assert (info["n"], info["maxlevel"], info["enterpoint"], info["maxM"], info["maxM0"], info["M"]) == \
        (n, maxlevel, ep, maxM, maxM0, M)
    offs, nbrs, c = z["node_nbr_offsets"], z["node_nbrs"], 0
    for j, node in enumerate(z["node_ids"]):
        for l in range(maxlevel + 1):
            level, label, ids = orc.node(int(node), l)
            if l == 0:
                assert level == z["node_level"][j] and label == z["node_label"][j]
            want = nbrs[offs[c]:offs[c + 1]]
            assert np.array_equal(ids if l <= level else np.zeros(0, np.uint32), want), (node, l)
            c += 1


@pytest.mark.parametrize("name,metric", FIXTURES)
@pytest.mark.parametrize("order", [rh.ORDER_SEQ, rh.ORDER_REF, rh.ORDER_GPU])
def test_golden_search(name, metric, order):
    """Same k-subset as the reference's searchKnn and the same number of distance evaluations."""
    z, graph = _load(name)
    orc = rh.Oracle(graph, int(z["dim"]), metric)
    k = int(z["k"])
    for ef in EFS:
        lab, dist, nd, nh = orc.search(z["queries"], k, ef, order=order, team=8, threads=1)
        ref = z[f"ref_labels_ef{ef}"]
        same = np.array([set(a) == set(b) for a, b in zip(lab, ref)])
        # the three fp32 associations agree with the reference except at (near-)ties
        assert same.mean() >= 0.97, (ef, same.mean())
        assert (nd[same] == z[f"ref_counts_ef{ef}"][same]).all()
        assert (np.diff(dist, axis=1) >= 0).all()


@pytest.mark.parametrize("name,metric", FIXTURES)
def test_golden_distance_and_bruteforce(name, metric):
    z, graph = _load(name)
    dim, n = int(z["dim"]), int(z["n"])
    orc = rh.Oracle(graph, dim, metric)
    base = np.stack([orc.vector(i) for i in range(n)])
    q = z["queries"]
    for order in (rh.ORDER_SEQ, rh.ORDER_REF, rh.ORDER_GPU, rh.ORDER_SEQFMA):
        d = np.array([rh.oracle_dist(q[i], base[i], metric, order) for i in range(len(q))], np.float32)
        np.testing.assert_allclose(d, z["ref_dist_samples"], rtol=2e-6, atol=1e-6)
    gt, gd = rh.oracle_bruteforce(base, q, 100, metric=metric, order=rh.ORDER_REF)
    ref = z["ref_gt100"]
    # farthest-first rows; identical except where the two fp32 associations reorder a near-tie
    same = (gt == ref).mean()
    assert same >= 0.995, same
    assert all(len(set(a) ^ set(b)) <= 2 for a, b in zip(gt, ref))
    assert (np.diff(gd, axis=1) <= 0).all()


def test_recall_definition():
    """hso_recall == SolveStrategy::recall restated in numpy (solve_strategy.h:67-103)."""
    rng = np.random.default_rng(0)
    n, nq, dim, K, gtk = 500, 40, 8, 10, 100
    base = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    gt = np.stack([rng.permutation(n)[:gtk] for _ in range(nq)]).astype(np.uint32)
    knn = np.stack([rng.permutation(n)[:K] for _ in range(nq)]).astype(np.uint32)
    knn[:, :5] = np.stack([g[np.argsort(((base[g] - x) ** 2).sum(1))[:5]] for g, x in zip(gt, q)])
    hits = 0
    for i in range(nq):
        d = ((base[gt[i]] - q[i]) ** 2).sum(1).astype(np.float32)
        order = np.lexsort((gt[i], d))
        hits += len(set(gt[i][order[:K]].tolist()) & set(knn[i].tolist()))
    want = hits / (nq * K)
    got = rh.oracle_recall(base, q, knn, gt, K)
    assert abs(got - want) < 1e-9 and got >= 0.5


@needs_ref
@pytest.mark.parametrize("K,gtk", [(10, 100), (3, 10), (10, 10)])
def test_recall_pinned_to_the_executed_reference(K, gtk):
    """hso_recall against the reference's OWN SolveStrategy::recall (solve_strategy.h:67-103), executed by
    oracle/_ref on .fvecs/.ivecs files the way `main` runs it — not a restatement.  The reference prints the
    value through operator<<(float) (6 significant digits), which bounds the comparison."""
    rng = np.random.default_rng(K * 7 + gtk)
    n, nq, dim = 4000, 120, 16
    base = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    d = ((base[None] - q[:, None]) ** 2).sum(-1)
    gt = np.argsort(d, axis=1)[:, :gtk][:, ::-1].astype(np.uint32).copy()       # farthest first, as BruteForce writes it
    knn = np.argsort(d, axis=1)[:, :K].astype(np.uint32)
    wrong = rng.random((nq, K)) < 0.3                                            # spoil ~30 % of the answers
    knn[wrong] = rng.integers(0, n, int(wrong.sum()))
    for row in knn:                                                              # answers of a search are distinct
        seen = set()
        for j in range(K):
            while int(row[j]) in seen:
                row[j] = rng.integers(0, n)
            seen.add(int(row[j]))
    want = rh.ref_strategy_recall(base, q, knn, gt, K)
    got = rh.oracle_recall(base, q, knn, gt, K)
    assert 0.4 < want < 0.95
    assert abs(got - want) <= 5e-6 * max(1.0, want) + 1e-6, (got, want)


@needs_ref
@pytest.mark.parametrize("metric,dim", [(0, 32), (1, 48)])
def test_live_reference_search_and_counts(metric, dim):
    c = get_corpus(n=20000, nq=300, dim=dim, metric=metric, rank=8)
    ref = rh.RefSlim(c.graph, c.dim, c.n, metric, counting=True)
    orc = rh.Oracle(c.graph, c.dim, metric)
    assert {k: ref.info()[k] for k in ("n", "maxlevel", "enterpoint", "maxM0")} == \
        {k: orc.info()[k] for k in ("n", "maxlevel", "enterpoint", "maxM0")}
    for ef in (10, 64, 150):
        rlab, rcnt = ref.counts(c.queries, 10, ef)
        for order in (rh.ORDER_REF, rh.ORDER_GPU):
            lab, dist, nd, nh = orc.search(c.queries, 10, ef, order=order, threads=2)
            same = np.array([set(a) == set(b) for a, b in zip(lab, rlab)])
            if order == rh.ORDER_REF and rh.ref_slim_path().endswith("_v4.so"):
                # the reference's own arithmetic, bit for bit (test_ref_order_is_bit_exact): nothing may differ
                assert same.all() and (nd == rcnt).all(), (ef, same.mean(), int((nd != rcnt).sum()))
            else:       # the kernel's association: a near-tie may fall the other way
                assert same.mean() >= 0.99, (ef, order, same.mean())
                assert (nd[same] == rcnt[same]).mean() >= 0.99


@needs_ref
def test_live_reference_bruteforce_and_recall():
    c = get_corpus(n=20000, nq=300, dim=32)
    gt_ref, _ = rh.ref_bruteforce(c.base, c.queries[:100], 100)
    gt_orc, _ = rh.oracle_bruteforce(c.base, c.queries[:100], 100, order=rh.ORDER_REF)
    assert (gt_ref == gt_orc).mean() >= 0.999
    ref = rh.RefSlim(c.graph, c.dim, c.n)
    lab, _, _ = ref.search(c.queries[:100], 10, 50)
    r = rh.oracle_recall(c.base, c.queries[:100], lab, gt_ref, 10)
    plain = np.mean([len(set(a) & set(b[-10:])) / 10 for a, b in zip(lab, gt_ref)])
    assert abs(r - plain) < 1e-6 and r > 0.7


@needs_ref
@pytest.mark.parametrize("dim", [32, 96, 128, 768, 960])
@pytest.mark.parametrize("metric", [0, 1])
def test_ref_order_is_bit_exact(dim, metric):
    """HSO_ORDER_REF restates the association of the reference's DISTFUNC AS COMPILED into oracle/_ref
    (space_l2.h:25-54 / space_ip.h:146-204 under -Ofast: per-lane accumulation, then a tree fold of the 16
    lanes): bit-identical distances, so the oracle takes the same side of every near-tie the reference does.
    Holds for the x86-64-v4 (AVX-512) build; the AVX2 build sums in another order."""
    if not rh.ref_slim_path().endswith("_v4.so"):
        pytest.skip("host without AVX-512: oracle/_ref runs its x86-64-v3 build")
    rng = np.random.default_rng(dim * 2 + metric)
    a = rng.standard_normal((500, dim)).astype(np.float32)
    b = rng.standard_normal((500, dim)).astype(np.float32)
    if metric:
        a /= np.linalg.norm(a, axis=1, keepdims=True)
        b /= np.linalg.norm(b, axis=1, keepdims=True)
    r = np.array([rh.ref_dist(x, y, metric) for x, y in zip(a, b)], dtype=np.float32)
    o = np.array([rh.oracle_dist(x, y, metric, order=rh.ORDER_REF) for x, y in zip(a, b)], dtype=np.float32)
    assert np.array_equal(r.view(np.uint32), o.view(np.uint32))


@needs_ref
def test_live_reference_multithreaded_search_is_the_same():
    """The OpenMP loop of hnsw_slim_client_update_patch.cc:223-226 returns what the serial loop does."""
    c = get_corpus(n=20000, nq=300, dim=32)
    ref = rh.RefSlim(c.graph, c.dim, c.n)
    a, _, _ = ref.search(c.queries, 10, 64, 1)
    b, _, _ = ref.search(c.queries, 10, 64, 4)
    assert all(set(x) == set(y) for x, y in zip(a, b))


@needs_ref
@pytest.mark.parametrize("thr", [1, 2, 7])
def test_threshold_level_against_live_reference(thr):
    """threshold_level > 0 (layered beam, slim.h:222-316 + 2108-2113): identical k-subsets and
    distance-evaluation counts vs the reference on a reference-built index."""
    c = get_corpus(n=20000, nq=300, dim=32, threshold_level=thr)
    orc = rh.Oracle(c.graph, c.dim, c.metric)
    assert orc.info()["threshold_level"] == thr
    ref = rh.RefSlim(c.graph, c.dim, c.n, c.metric, counting=True)
    for ef in (10, 60, 150):
        lab, dist, nd, nh = orc.search(c.queries, 10, ef, order=rh.ORDER_REF, threads=1)
        rlab, rcnt = ref.counts(c.queries, 10, ef)
        same = np.array([set(a) == set(b) for a, b in zip(lab, rlab)])
        if rh.ref_slim_path().endswith("_v4.so"):
            assert same.all() and (nd == rcnt).all(), (thr, ef, same.mean(), int((nd != rcnt).sum()))
        else:
            assert same.mean() >= 0.995, (thr, ef, same.mean())
            assert (nd[same] == rcnt[same]).all()


def test_tie_events_are_reported():
    """hso_search_ties = hso_search + the per-query count of exact fp32 ties at the ef boundary (a result trimmed
    while the new worst carries the bit-identical distance).  On the golden corpus (distinct rows) there are none;
    on a corpus in which every row exists three times they are the rule; ids, distances and counters are those of
    hso_search either way."""
    import tempfile
    z = np.load(os.path.join(GOLDEN, "slim_l2_2k.npz"))
    q = z["queries"]
    orc = rh.Oracle(os.path.join(GOLDEN, "slim_l2_2k.graph"), 16)
    for ef in (10, 40, 100):
        a = orc.search(q, 10, ef, order=rh.ORDER_GPU, team=8)
        b = orc.search_ties(q, 10, ef, order=rh.ORDER_GPU, team=8)
        assert all(np.array_equal(x, y) for x, y in zip(a, b[:4]))
        assert int(b[4].sum()) == 0
    from hnsw_slim_b200 import capi
    rng = np.random.default_rng(3)
    rows = rng.standard_normal((700, 16)).astype(np.float32)
    base = np.repeat(rows, 3, axis=0)                            # every vector three times, bit for bit
    queries = rng.standard_normal((60, 16)).astype(np.float32)
    with tempfile.TemporaryDirectory() as td:
        g = os.path.join(td, "ties.graph")
        capi.build_slim_graph(base, g, M=8, ef_construction=60, threads=1)   # single-threaded: the same graph on every box
        orc = rh.Oracle(g, 16)
        a = orc.search(queries, 10, 12, order=rh.ORDER_GPU, team=8)
        b = orc.search_ties(queries, 10, 12, order=rh.ORDER_GPU, team=8)
        assert all(np.array_equal(x, y) for x, y in zip(a, b[:4]))
        assert (b[4] > 0).mean() > 0.5, b[4]


@pytest.mark.parametrize("name,metric", [("slim_l2_2k", 0), ("slim_ip_1k", 1)])
def test_pool_emulator_equals_the_reference_semantics(name, metric):
    """hso_search_pool restates the ENGINE's algorithm (one pool in 32 columns, the kernel's placement, tie and
    ghost rules); hso_search restates the REFERENCE's (two heaps).  They must agree to the bit — ids, distances,
    evaluation and hop counters — on every query without an exact fp32 tie at the ef boundary."""
    z = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    q = z["queries"]
    orc = rh.Oracle(os.path.join(GOLDEN, f"{name}.graph"), 16, metric)
    for ef in (10, 33, 64, 100, 129, 161, 200, 256):
        lab, dist, nd, nh, nt = orc.search_ties(q, 10, ef, order=rh.ORDER_GPU, team=8)
        pl, pd, pnd, pnh, png = orc.search_pool(q, 10, ef, team=8)
        clean = nt == 0
        assert clean.mean() > 0.9
        assert np.array_equal(pl[clean], lab[clean]) and np.array_equal(pd[clean].view(np.uint32), dist[clean].view(np.uint32))
        assert np.array_equal(pnd[clean], nd[clean]) and np.array_equal(pnh[clean], nh[clean])
    with pytest.raises(RuntimeError):
        orc.search_pool(q, 10, 300)                              # register pools only


def test_pool_emulator_on_a_live_corpus():
    """The same on a 20k x 128 corpus, plus the all-ties corpus where the two algorithms are ALLOWED to part:
    the emulator must still return a valid answer (sorted, distinct ids) with recall equal within 0.5 pp."""
    import tempfile
    from hnsw_slim_b200 import capi
    from hnsw_slim_b200.synth import make_dataset
    base, q = make_dataset(20000, 300, 128, rank=14, seed=2)
    with tempfile.TemporaryDirectory() as td:
        g = os.path.join(td, "g.graph")
        capi.build_slim_graph(base, g, M=16, ef_construction=100, threads=1)     # single-threaded: the same graph on every box
        orc = rh.Oracle(g, 128)
        for ef in (50, 100, 200):
            lab, dist, nd, nh, nt = orc.search_ties(q, 10, ef, order=rh.ORDER_GPU, team=8)
            pl, pd, pnd, pnh, _ = orc.search_pool(q, 10, ef, team=8)
            clean = nt == 0
            assert np.array_equal(pl[clean], lab[clean]) and np.array_equal(pnd[clean], nd[clean])
            assert np.array_equal(pnh[clean], nh[clean])
        rng = np.random.default_rng(3)
        rows = rng.standard_normal((700, 16)).astype(np.float32)
        tb = np.repeat(rows, 3, axis=0)
        tq = rng.standard_normal((60, 16)).astype(np.float32)
        g2 = os.path.join(td, "ties.graph")
        capi.build_slim_graph(tb, g2, M=8, ef_construction=60, threads=1)
        o2 = rh.Oracle(g2, 16)
        for ef in (12, 24, 40):
            lab, dist, *_ = o2.search_ties(tq, 10, ef, order=rh.ORDER_GPU, team=8)
            pl, pd, *_ = o2.search_pool(tq, 10, ef, team=8)
            assert (np.diff(pd, axis=1) >= 0).all()
            assert all(len(set(r)) == 10 for r in pl)
            # the same distance multiset on almost every row (ties only reorder equal distances)
            assert np.mean(np.all(pd.view(np.uint32) == dist.view(np.uint32), axis=1)) >= 0.9
