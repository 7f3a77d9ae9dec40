"""GPU parity: the CUDA traversal (through the C ABI) against the C oracle and the reference.

Bars (north_star): graph search reproduces the reference's recall@k within 0.5 pp at the same
graph and ef_search; returned distances within 1e-5 relative.  We assert more: against the
oracle run with the kernel's own fp32 association (HSO_ORDER_GPU) ids, distances and the
per-query distance-evaluation counts are BIT-EXACT (integer/index work is exact; only bitwise
distance ties may differ).
"""
import numpy as np
import pytest

from conftest import get_corpus, needs_ref
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset
from oracle import refharness as rh

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5   # north_star: distances within 1e-5 relative error


def _recall(found, gt_sets):
    return float(np.mean([len(set(f) & g) / len(g) for f, g in zip(found, gt_sets)]))


def check_against_oracle(c, k, ef, *, min_exact=0.999):
    ix = capi.Index(c.graph, c.dim, metric=c.metric)
    ix.set_ef(ef)
    lab, dist, cnt = ix.search(c.queries, k, counts=True)
    orc = rh.Oracle(c.graph, c.dim, c.metric)
    olab, odist, ond, onh = orc.search(c.queries, k, ef, order=rh.ORDER_GPU, team=8)
    same_rows = np.all(lab == olab, axis=1)
    # bit-exact ids, distances and counters (ties aside)
    assert same_rows.mean() >= min_exact, f"only {same_rows.mean():.4f} of rows identical to the oracle"
    assert np.array_equal(dist[same_rows].view(np.uint32), odist[same_rows].view(np.uint32))
    # counters: bit-exact as well.  (The test graphs are built single-threaded, hence identical on every box;
    # the one known way the two sides can part — an entry evicted from the result set whose distance EQUALS
    # the new lowerBound is still expanded by the reference but is gone from the pool here — needs an exact
    # fp32 tie at the ef boundary and is exercised on purpose by test_exact_ties_at_the_ef_boundary.)
    bad = np.nonzero(same_rows & ((cnt[:, 0] != ond) | (cnt[:, 1] != onh)))[0]
    msg = "; ".join(f"q{q}: gpu {cnt[q].tolist()} oracle [{ond[q]}, {onh[q]}]" for q in bad[:5])
    assert len(bad) == 0, f"per-query counters differ on {len(bad)} of {len(cnt)} identical rows: {msg}"
    # rows that differ must be explainable by ties: same distance multiset within tolerance
    for i in np.nonzero(~same_rows)[0]:
        fin = np.isfinite(odist[i])
        np.testing.assert_allclose(dist[i][fin], odist[i][fin], rtol=REL_TOL)
    return ix, lab, dist


@pytest.mark.parametrize("ef", [10, 50, 100, 200, 300])     # register pools (<= 64 / 128 / 256) and the smem pool
def test_small_l2_matches_oracle_bit_exact(small_corpus, ef):
    check_against_oracle(small_corpus, 10, ef)


@needs_ref
@pytest.mark.parametrize("ef", [50, 100])
def test_small_l2_matches_reference(small_corpus, ef):
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(ef)
    lab, dist = ix.search(c.queries, 10)
    ref = rh.RefSlim(c.graph, c.dim, c.n)
    rlab, _, _ = ref.search(c.queries, 10, ef)
    gt, _ = rh.ref_bruteforce(c.base, c.queries, 10)
    gts = [set(r) for r in gt]
    r_gpu, r_ref = _recall(lab, gts), _recall(rlab, gts)
    assert abs(r_gpu - r_ref) <= 0.005, (r_gpu, r_ref)          # 0.5 pp
    same = np.mean([set(a) == set(b) for a, b in zip(lab, rlab)])
    assert same >= 0.99, same
    # distances: recompute with the reference's own DISTFUNC
    for i in range(0, c.nq, 17):
        for j in range(10):
            d = rh.ref_dist(c.queries[i], c.base[lab[i, j]], c.metric)
            assert abs(d - dist[i, j]) <= REL_TOL * max(abs(d), 1e-30)


def test_exact_ties_at_the_ef_boundary(tmp_path):
    """Constructed exact ties.  Every vector of the corpus exists THREE times, so every distance the search
    sees exists three times bit for bit, also at the ef boundary.  The reference admits a neighbour iff
    `top_size < ef || lowerBound > dist` (slim.h:403-404, strict) and stops when the closest candidate is
    `> lowerBound` (slim.h:339-340, strict): a candidate whose distance EQUALS lowerBound is still expanded by
    the reference even after it was trimmed from the result heap, while the engine's pool has dropped it.
    Which of several equal-distance entries is trimmed / popped first is heap order in the reference and
    (lane, slot) order here.  This pins what that is allowed to change: the k returned DISTANCES (as a sorted
    multiset), never — only which of the identical copies carries a distance may differ, and with it the
    counters.  The graph comes from the engine's host builder, single-threaded, hence the same on every box."""
    rng = np.random.default_rng(123)
    distinct, copies, dim, nq, k = 2500, 3, 32, 400, 10
    d0, q = make_dataset(distinct, nq, dim, rank=8, seed=41)
    base = np.ascontiguousarray(np.repeat(d0, copies, axis=0)[rng.permutation(distinct * copies)])
    graph = str(tmp_path / "ties.graph")
    capi.build_slim_graph(base, graph, M=8, ef_construction=60, threads=1)
    orc = rh.Oracle(graph, dim)
    ix = capi.Index(graph, dim)
    true_d = np.sort(((base[None, :, :] - q[:, None, :]) ** 2).sum(-1), axis=1)[:, :k]    # exact, tie-aware yardstick
    for ef in (10, 12, 16, 24, 40):
        ix.set_ef(ef)
        lab, dist, cnt = ix.search(q, k, counts=True)
        olab, odist, ond, onh = orc.search(q, k, ef, order=rh.ORDER_GPU, team=8)
        assert (np.diff(dist, axis=1) >= 0).all()
        # every returned distance is the distance of the returned row (bitwise, GPU association)
        same_d = np.all(dist.view(np.uint32) == odist.view(np.uint32), axis=1)
        same_ids = np.all(lab == olab, axis=1)
        same_cnt = (cnt[:, 0] == ond) & (cnt[:, 1] == onh)
        # tie-aware recall: a returned distance counts when it is within the true k-th distance
        hit = lambda d: float(np.mean(d <= true_d[:, -1:] * (1 + 1e-6)))
        print(f"\nties ef={ef}: identical distance rows {same_d.mean():.4f}, identical id rows {same_ids.mean():.4f}, "
              f"identical counters {same_cnt.mean():.4f}, tie-aware recall gpu {hit(dist):.4f} oracle {hit(odist):.4f}")
        # the bound: the divergence may move WHICH copy is reported and how many hops it took, and in rare
        # cases reach one more / one fewer candidate — never more than 0.5 pp of recall, and at least 95 % of
        # the rows carry bit-identical distances even in this all-ties corpus (measured on a B200: 99.75 % at ef=10)
        assert same_d.mean() >= 0.95, (ef, same_d.mean())
        assert abs(hit(dist) - hit(odist)) <= 0.005, (ef, hit(dist), hit(odist))
        # where the ids agree, the distances agree bitwise
        assert np.array_equal(dist[same_ids].view(np.uint32), odist[same_ids].view(np.uint32))


@needs_ref
def test_c1_graph_against_live_reference(tmp_path):
    """The north-star bar on the REAL configuration (BASELINE.json configs[0]): SIFT-shaped 1M x 128, M=16,
    efc=200, graph built by the reference itself (omp addPoint + convertFromHNSW), ef_search=100, k=10, 2000
    queries — the engine's recall@10 within 0.5 pp of the live reference's searchKnn on the same graph, the
    neighbour sets themselves equal for >= 99 % of the queries, returned distances within 1e-5 relative of the
    reference's DISTFUNC, and bit-exact ids / distances / counters against the oracle."""
    from hnsw_slim_b200.synth import latent_gaussian
    n, dim, nq, k, ef = 1_000_000, 128, 2000, 10, 100
    base = latent_gaussian(n, dim, rank=14, seed=1)
    q = latent_gaussian(nq, dim, rank=14, seed=1, stream=1)
    graph = str(tmp_path / "c1.graph")
    rh.ref_slim_build(base, graph, M=16, ef_construction=200, branching="4")
    ix = capi.Index(graph, dim)
    ix.set_ef(ef)
    lab, dist, cnt = ix.search(q, k, counts=True)
    ref = rh.RefSlim(graph, dim, n)
    rlab, _, _ = ref.search(q, k, ef, 0)
    gt, _ = capi.bruteforce_knn(base, q, k)
    gts = [set(r) for r in gt]
    r_gpu, r_ref = _recall(lab, gts), _recall(rlab, gts)
    print(f"\nC1 1M x 128 ef=100: recall@10 engine {r_gpu:.4f}, live reference {r_ref:.4f}")
    assert r_gpu >= 0.95 and abs(r_gpu - r_ref) <= 0.005, (r_gpu, r_ref)
    same = np.mean([set(a) == set(b) for a, b in zip(lab, rlab)])
    assert same >= 0.99, same
    for i in range(0, nq, 40):
        for j in range(k):
            d = rh.ref_dist(q[i], base[lab[i, j]], 0)
            assert abs(d - dist[i, j]) <= REL_TOL * max(abs(d), 1e-30)
    orc = rh.Oracle(graph, dim)
    olab, odist, ond, onh = orc.search(q, k, ef, order=rh.ORDER_GPU, team=8)
    same_rows = np.all(lab == olab, axis=1)
    assert same_rows.mean() >= 0.999, same_rows.mean()
    assert np.array_equal(dist[same_rows].view(np.uint32), odist[same_rows].view(np.uint32))
    assert np.array_equal(cnt[same_rows, 0], ond[same_rows]) and np.array_equal(cnt[same_rows, 1], onh[same_rows])


@pytest.mark.parametrize("dim,rank", [(96, 12), (128, 14), (100, 12), (64, 8)])
def test_dims_l2(dim, rank):
    c = get_corpus(n=20000, nq=200, dim=dim, rank=rank)
    check_against_oracle(c, 10, 64)


def test_large_dim_generic_kernel():
    c = get_corpus(n=6000, nq=100, dim=960, rank=16, M=32)     # GIST-shaped rows, M=32 -> deg stride 64
    ix, lab, dist = check_against_oracle(c, 10, 100)
    assert ix.info()["deg0_stride"] in (32, 64)


def test_inner_product():
    c = get_corpus(n=20000, nq=200, dim=768, rank=16, M=32, metric=1)   # COHERE-shaped
    check_against_oracle(c, 10, 100)


def test_edge_cases(small_corpus):
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    # nq = 0 and empty results buffers
    lab, dist = ix.search(np.zeros((0, c.dim), np.float32), 10)
    assert lab.shape == (0, 10)
    # ef < k -> ef = max(ef, k)   (slim.h:2080)
    ix.set_ef(3)
    lab, dist = ix.search(c.queries[:50], 20)
    orc = rh.Oracle(c.graph, c.dim)
    olab, odist, _, _ = orc.search(c.queries[:50], 20, 3)
    assert np.array_equal(lab, olab)
    assert (np.diff(dist, axis=1) >= 0).all()                     # sortedness
    # single query, k = 1
    ix.set_ef(50)
    lab1, _ = ix.search(c.queries[:1], 1)
    olab1, _, _, _ = orc.search(c.queries[:1], 1, 50)
    assert np.array_equal(lab1, olab1)
    # a query that IS a base vector finds itself at distance 0
    lab, dist = ix.search(c.base[:64], 1)
    assert (dist[:, 0] == 0).all() and np.array_equal(lab[:, 0], np.arange(64, dtype=np.uint32))
    # idempotence + batch-split invariance
    ix.set_ef(80)
    a, _ = ix.search(c.queries, 10)
    b, _ = ix.search(c.queries, 10)
    h = c.nq // 2
    c1, _ = ix.search(c.queries[:h], 10)
    c2, _ = ix.search(c.queries[h:], 10)
    assert np.array_equal(a, b) and np.array_equal(a, np.vstack([c1, c2]))


def test_tiny_graphs():
    for n in (1, 2, 5, 40):
        c = get_corpus(n=n, nq=7, dim=32, M=4, efc=20)
        ix = capi.Index(c.graph, c.dim)
        ix.set_ef(16)
        k = 3
        lab, dist = ix.search(c.queries, k)
        orc = rh.Oracle(c.graph, c.dim)
        olab, odist, _, _ = orc.search(c.queries, k, 16)
        assert np.array_equal(lab, olab), n
        assert np.array_equal(np.isinf(dist), np.isinf(odist))


def test_hash_reset_keeps_results(small_corpus, monkeypatch):
    """A visited hash far too small forces resets: results must not change (only n_dist grows)."""
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(100)
    a, da, ca = ix.search(c.queries, 10, counts=True)
    monkeypatch.setenv("HS_HASH_BITS", "8")
    ix2 = capi.Index(c.graph, c.dim)
    ix2.set_ef(100)
    b, db, cb = ix2.search(c.queries, 10, counts=True)
    assert np.array_equal(a, b) and np.array_equal(da, db)
    assert (cb[:, 0] >= ca[:, 0]).all() and (cb[:, 0] > ca[:, 0]).any()


@pytest.mark.parametrize("dim,rank,metric", [(128, 14, 0), (96, 12, 0), (128, 14, 1)])
def test_ef_129_to_256_compact_pool_and_visited_table(dim, rank, metric):
    """ef 129..256 at 96 / 128-dim rows: register pools of 5 / 6 / 7 / 8 slots with the expanded mark in the id word
    (RegPool32C) and the compact 16-bit visited table (cv_test_and_set) — bit-exact ids, distances and per-query
    counters against the oracle, whichever home the visited set has."""
    c = get_corpus(n=30000, nq=200, dim=dim, rank=rank, metric=metric)
    orc = rh.Oracle(c.graph, c.dim, metric)
    ix = capi.Index(c.graph, c.dim, metric=metric)
    tie_queries = 0
    for ef in (129, 160, 161, 192, 193, 224, 225, 256):
        olab, odist, ond, onh, oties = orc.search_ties(c.queries, 10, ef, order=rh.ORDER_GPU, team=8)
        # Counters are compared on every query without an exact fp32 tie at the ef boundary (hso_search_ties: a
        # result trimmed while tying with the new worst one).  At such a tie the reference's heaps and the engine's
        # pool may take the two equal candidates in a different order, which can change what is expanded next
        # (DESIGN.md §3); ids and distances must match regardless.
        clean = oties == 0
        tie_queries += int((~clean).sum())
        for mode in (-1, 2, 3, 0, 1):                      # automatic (compact), compact, legacy automatic, smem32, global
            ix.set_tuning("visited_table", mode)
            ix.set_ef(ef)
            lab, dist, cnt = ix.search(c.queries, 10, counts=True)
            assert np.array_equal(lab, olab), (ef, mode)
            assert np.array_equal(dist.view(np.uint32), odist.view(np.uint32)), (ef, mode)
            bad = np.nonzero((cnt[:, 0] != ond) | (cnt[:, 1] != onh))[0]
            assert clean[bad].sum() == 0, (ef, mode, bad.tolist(), cnt[bad].tolist(), ond[bad].tolist(), onh[bad].tolist())
            assert len(bad) <= 1, (ef, mode, bad.tolist())
    assert tie_queries <= 16          # the exemption is the exception: a handful of the 1600 (query, ef) pairs


def test_engine_equals_its_cpu_restatement_on_every_query():
    """oracle/hs_oracle.c hso_search_pool restates the ENGINE's algorithm on the CPU — one pool in 32 columns, the
    kernel's placement, tie and ghost rules.  The kernel must equal it on EVERY query, exact ties included: ids,
    distance bits, evaluation and hop counters.  (Against the reference's two-heap semantics the same runs differ
    on one query — 81 at ef=161, where two candidates carry the bit-identical distance and the reference happens
    to expand them in the other order; test_ef_129_to_256_compact_pool_and_visited_table, DESIGN.md §3.)"""
    c = get_corpus(n=30000, nq=200, dim=128, rank=14, metric=1)
    orc = rh.Oracle(c.graph, c.dim, 1)
    ix = capi.Index(c.graph, c.dim, metric=1)
    differs_from_reference = 0
    for ef in (16, 64, 100, 129, 160, 161, 192, 224, 256):
        ix.set_ef(ef)
        lab, dist, cnt = ix.search(c.queries, 10, counts=True)
        pl, pd, pnd, pnh, _ = orc.search_pool(c.queries, 10, ef, team=8)
        assert np.array_equal(lab, pl), ef
        assert np.array_equal(dist.view(np.uint32), pd.view(np.uint32)), ef
        assert np.array_equal(cnt[:, 0], pnd) and np.array_equal(cnt[:, 1], pnh), ef
        _, _, ond, onh = orc.search(c.queries, 10, ef, order=rh.ORDER_GPU, team=8)
        differs_from_reference += int(((cnt[:, 0] != ond) | (cnt[:, 1] != onh)).sum())
    assert differs_from_reference <= 1


def test_compact_visited_table_reset_and_overflow():
    """The compact table's rare paths made common: an early load limit (reset + re-seed from the pool) and
    single-choice buckets (ids that find their bucket full go unrecorded and force a reset).  Results are the
    oracle's either way; only the evaluation counters may grow."""
    c = get_corpus(n=30000, nq=200, dim=128, rank=14)
    orc = rh.Oracle(c.graph, c.dim)
    ix = capi.Index(c.graph, c.dim)
    ix.set_tuning("visited_table", 2)
    for ef in (140, 256):
        olab, odist, ond, _ = orc.search(c.queries, 10, ef, order=rh.ORDER_GPU, team=8)
        ix.set_ef(ef)
        grew = []
        for flags in (9 | 16, 9 | 32, 9 | 16 | 32):
            ix.set_tuning("traverse_flags", flags)
            lab, dist, cnt = ix.search(c.queries, 10, counts=True)
            assert np.array_equal(lab, olab), (ef, flags)
            assert np.array_equal(dist.view(np.uint32), odist.view(np.uint32)), (ef, flags)
            assert (cnt[:, 0] >= ond).all(), (ef, flags)
            grew.append(bool((cnt[:, 0] > ond).any()))
        assert grew[0], ef                                  # the early limit did trigger resets
        ix.set_tuning("traverse_flags", 9)
    with pytest.raises(capi.HsError):
        ix.set_tuning("no_such_knob", 1)


def test_large_ef_shared_memory_pool(small_corpus):
    """The generic kernel (query in shared memory): register pools up to ef = 256 (2..8 slots per lane), the
    shared-memory pool above — and, forced by traverse_flags bit 6, at every ef: all bit-exact against the oracle."""
    for ef in (33, 64, 65, 128, 129, 300, 384, 385, 512, 513, 700):
        check_against_oracle(small_corpus, 10, ef)
    c = small_corpus
    orc = rh.Oracle(c.graph, c.dim, c.metric)
    ix = capi.Index(c.graph, c.dim, metric=c.metric)
    ix.set_tuning("traverse_flags", 9 | 64)
    for ef in (64, 200, 300, 512):
        ix.set_ef(ef)
        lab, dist, cnt = ix.search(c.queries, 10, counts=True)
        olab, odist, ond, onh = orc.search(c.queries, 10, ef, order=rh.ORDER_GPU, team=8)
        assert np.array_equal(lab, olab) and np.array_equal(dist.view(np.uint32), odist.view(np.uint32)), ef
        assert np.array_equal(cnt[:, 0], ond) and np.array_equal(cnt[:, 1], onh), ef


@pytest.mark.parametrize("thr", [1, 2, 7])
def test_threshold_level_layered_beam(thr):
    """threshold_level > 0: greedy descent stops above the threshold, then searchBaseLayer runs on
    levels min(thr, maxlevel) .. 1 (slim.h:222-316, 2108-2113) before the base layer.  thr = 7
    exceeds maxlevel of this corpus: no greedy descent at all."""
    c = get_corpus(n=20000, nq=300, dim=32, threshold_level=thr)
    info = capi.Index(c.graph, c.dim).info()
    assert info["threshold_level"] == thr
    for ef in (10, 60, 150, 300):
        check_against_oracle(c, 10, ef)
    # a visited hash too small for the layered beam is cleared and re-seeded: results identical
    import os
    os.environ["HS_HASH_BITS"] = "9"
    try:
        ix = capi.Index(c.graph, c.dim)
    finally:
        del os.environ["HS_HASH_BITS"]
    ix.set_ef(60)
    lab, dist = ix.search(c.queries, 10)
    olab, odist, _, _ = rh.Oracle(c.graph, c.dim).search(c.queries, 10, 60, order=rh.ORDER_GPU, team=8)
    assert (lab == olab).all(1).mean() >= 0.999


@needs_ref
def test_threshold_level_matches_reference():
    c = get_corpus(n=20000, nq=300, dim=32, threshold_level=1)
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(80)
    lab, _ = ix.search(c.queries, 10)
    ref = rh.RefSlim(c.graph, c.dim, c.n)
    rlab, _, _ = ref.search(c.queries, 10, 80)
    same = np.mean([set(a) == set(b) for a, b in zip(lab, rlab)])
    assert same >= 0.995, same


def test_k_larger_than_32(small_corpus):
    check_against_oracle(small_corpus, 100, 100)
    check_against_oracle(small_corpus, 64, 200)


def test_full_size_properties():
    """Size-independent properties on a 200k x 128 corpus (the oracle would take minutes here):
    sortedness, self-retrieval, recall monotone in ef, counters consistent, determinism."""
    n, nq, dim = 200000, 2000, 128
    base, q = make_dataset(n, nq, dim, rank=14)
    import tempfile, os
    with tempfile.TemporaryDirectory() as td:
        g = os.path.join(td, "g.graph")
        capi.build_slim_graph(base, g, M=16, ef_construction=100)
        ix = capi.Index(g, dim)
        gt, _ = capi.bruteforce_knn(base, q[:500], 10)
        prev = 0.0
        for ef in (20, 50, 100, 200):
            ix.set_ef(ef)
            lab, dist, cnt = ix.search(q, 10, counts=True)
            assert (np.diff(dist, axis=1) >= 0).all() and (lab < n).all()
            assert all(len(set(r)) == 10 for r in lab[:200])
            rec = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(lab[:500], gt)])
            assert rec >= prev - 0.002
            prev = rec
            assert (cnt[:, 0] >= cnt[:, 1]).all() and (cnt[:, 1] >= 1).all()
            # returned distances are the true distances of the returned rows
            i = np.arange(0, nq, 37)
            true = ((base[lab[i, 0]] - q[i]) ** 2).sum(1)
            np.testing.assert_allclose(dist[i, 0], true, rtol=1e-5)
        assert prev >= 0.95
        self_lab, self_d = ix.search(base[:1000], 1)
        found = self_lab[:, 0] == np.arange(1000, dtype=np.uint32)      # pruning may orphan a few nodes
        assert found.mean() >= 0.99, found.mean()
        assert (self_d[found, 0] == 0).all()
        a, _ = ix.search(q, 10)
        b, _ = ix.search(q[::-1].copy(), 10)
        assert np.array_equal(a, b[::-1])


def test_stats_counters(small_corpus):
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(50)
    ix.reset_stats()
    _, _, cnt = ix.search(c.queries, 10, counts=True)
    st = ix.stats()
    assert st["n_dist"] == int(cnt[:, 0].sum()) and st["n_hops"] == int(cnt[:, 1].sum())


def test_errors_are_loud(tmp_path):
    with pytest.raises(capi.HsError) as e:
        capi.Index(str(tmp_path / "missing.graph"), 32)
    assert e.value.code == -2
    bad = tmp_path / "bad.graph"
    bad.write_bytes(b"\x01" * 100)
    with pytest.raises(capi.HsError):
        capi.Index(str(bad), 32)


def test_batch_overlap_keeps_results(small_corpus):
    """hs_set_overlap: consecutive device-buffer batches on one stream may overlap (programmatic
    dependent launch + a ring of work counters); every batch still gets exactly its own results."""
    import torch
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(60)
    k, nq = 10, c.queries.shape[0]
    batches = [np.ascontiguousarray(np.roll(c.queries, s, axis=0)) for s in range(12)]
    want = [ix.search(b, k) for b in batches]
    ix.set_overlap(True)
    dq = [torch.from_numpy(b).cuda() for b in batches]
    dl = [torch.empty((nq, k), dtype=torch.int32, device="cuda") for _ in batches]
    dd = [torch.empty((nq, k), dtype=torch.float32, device="cuda") for _ in batches]
    torch.cuda.synchronize()
    s = torch.cuda.current_stream().cuda_stream
    for rep in range(3):
        for i in range(len(batches)):
            ix.search_device(dq[i].data_ptr(), nq, k, dl[i].data_ptr(), dd[i].data_ptr(), s)
    torch.cuda.synchronize()
    for i, (wl, wd) in enumerate(want):
        assert np.array_equal(dl[i].cpu().numpy().view(np.uint32), wl), i
        assert np.array_equal(dd[i].cpu().numpy().view(np.uint32), wd.view(np.uint32)), i


@pytest.mark.parametrize("dim,k", [(128, 10), (100, 10), (128, 40), (30, 7)])
def test_zero_copy_host_buffers_match_staged(dim, k):
    """hs_search_batch with pinned + mapped host buffers runs the kernel directly on them (no staging
    copies); pageable buffers go through the staged path.  Same results either way, also for a
    dimension that is not a multiple of 4 (scalar query loads) and k > 32 (two result flushes)."""
    import torch
    c = get_corpus(n=20000, nq=333, dim=dim)
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(80)
    want_l, want_d = ix.search(c.queries, k)                      # pageable numpy -> staged path
    nq = c.queries.shape[0]
    hq = torch.from_numpy(c.queries).pin_memory()
    hl = torch.full((nq, k), -1, dtype=torch.int32).pin_memory()
    hd = torch.zeros((nq, k), dtype=torch.float32).pin_memory()
    ix.search_ptr(hq.data_ptr(), nq, k, hl.data_ptr(), hd.data_ptr())
    assert np.array_equal(hl.numpy().view(np.uint32), want_l)
    assert np.array_equal(hd.numpy().view(np.uint32), want_d.view(np.uint32))
    # an unaligned view of a pinned buffer (queries start 4 bytes in): scalar loads, same results
    flat = torch.zeros(nq * dim + 1, dtype=torch.float32).pin_memory()
    flat[1:] = torch.from_numpy(c.queries).reshape(-1)
    hl.fill_(-1)
    ix.search_ptr(flat.data_ptr() + 4, nq, k, hl.data_ptr(), hd.data_ptr())
    assert np.array_equal(hl.numpy().view(np.uint32), want_l)


@pytest.mark.parametrize("pinned", [True, False])
def test_submit_wait_pipeline(small_corpus, pinned):
    """hs_search_batch_submit / hs_search_batch_wait: several host-buffer batches in flight on the
    handle's stream (zero-copy for pinned buffers, staged for pageable ones), overlap on."""
    import torch
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(60)
    k, nq = 10, c.queries.shape[0]
    batches = [np.ascontiguousarray(np.roll(c.queries, s, axis=0)) for s in range(6)]
    want = [ix.search(b, k) for b in batches]
    ix.set_overlap(True)
    hq = [torch.from_numpy(b) for b in batches]
    hl = [torch.full((nq, k), -1, dtype=torch.int32) for _ in batches]
    hd = [torch.zeros((nq, k), dtype=torch.float32) for _ in batches]
    if pinned:
        hq, hl, hd = [t.pin_memory() for t in hq], [t.pin_memory() for t in hl], [t.pin_memory() for t in hd]
    for rep in range(2):
        for i in range(len(batches)):
            ix.submit_ptr(hq[i].data_ptr(), nq, k, hl[i].data_ptr(), hd[i].data_ptr())
        ix.wait()
    for i, (wl, wd) in enumerate(want):
        assert np.array_equal(hl[i].numpy().view(np.uint32), wl), i
        assert np.array_equal(hd[i].numpy().view(np.uint32), wd.view(np.uint32)), i


def _index_with_env(c, **env):
    import os
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return capi.Index(c.graph, c.dim, metric=c.metric)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.mark.parametrize("ef", [40, 100, 200, 400])
def test_global_memory_visited_hash_same_results(small_corpus, ef):
    """HS_GHASH: the visited tables in global memory (the plan picks them for large ef / dim) and
    in shared memory give identical ids, distances and counters."""
    c = small_corpus
    a = _index_with_env(c, HS_GHASH=0)
    b = _index_with_env(c, HS_GHASH=1)
    a.set_ef(ef)
    b.set_ef(ef)
    la, da, ca = a.search(c.queries, 10, counts=True)
    lb, db, cb = b.search(c.queries, 10, counts=True)
    assert np.array_equal(la, lb) and np.array_equal(da.view(np.uint32), db.view(np.uint32))
    assert np.array_equal(ca, cb)


def test_global_memory_visited_hash_overlapping_batches(small_corpus):
    """Overlapping launches alternate between the two halves of the global visited scratch."""
    import torch
    c = small_corpus
    ix = _index_with_env(c, HS_GHASH=1)
    ix.set_ef(200)
    k = 10
    big = np.ascontiguousarray(np.tile(c.queries, (40, 1)))          # 12000 queries: the grid fills the GPU
    nq = big.shape[0]
    want_l, want_d = ix.search(big, k)
    ix.set_overlap(True)
    dq = torch.from_numpy(big).cuda()
    outs = [(torch.empty((nq, k), dtype=torch.int32, device="cuda"), torch.empty((nq, k), dtype=torch.float32, device="cuda"))
            for _ in range(5)]
    torch.cuda.synchronize()
    s = torch.cuda.current_stream().cuda_stream
    for dl, dd in outs:
        ix.search_device(dq.data_ptr(), nq, k, dl.data_ptr(), dd.data_ptr(), s)
    torch.cuda.synchronize()
    for dl, dd in outs:
        assert np.array_equal(dl.cpu().numpy().view(np.uint32), want_l)
        assert np.array_equal(dd.cpu().numpy().view(np.uint32), want_d.view(np.uint32))


def test_has_deleted_flag_without_marks(tmp_path):
    """has_deleted_elements_ = true in the header, no node marked: the reference runs the
    non-bare-bone template (slim.h:2114-2123), whose extra stop clause cannot fire — same results
    as the oracle's restatement of that template, and as the unflagged file."""
    import os
    from conftest import GOLDEN
    src = os.path.join(GOLDEN, "slim_l2_2k.graph")
    z = np.load(os.path.join(GOLDEN, "slim_l2_2k.npz"))
    img = bytearray(open(src, "rb").read())
    off = 6 * 8 + 3 * 4 + 4 * 8            # the bool after ef_construction (slim.h:717-739)
    assert img[off] == 0
    img[off] = 1
    flagged = str(tmp_path / "flagged.graph")
    open(flagged, "wb").write(bytes(img))
    dim, q = int(z["dim"]), z["queries"]
    ix = capi.Index(flagged, dim)
    assert ix.info()["has_deleted"] == 1
    plain = capi.Index(src, dim)
    for ef in (10, 40, 100):
        ix.set_ef(ef)
        plain.set_ef(ef)
        lab, dist = ix.search(q, 10)
        pl, pd = plain.search(q, 10)
        assert np.array_equal(lab, pl) and np.array_equal(dist.view(np.uint32), pd.view(np.uint32))
        ol, od, _, _ = rh.Oracle(flagged, dim).search(q, 10, ef, order=rh.ORDER_GPU, team=8)
        assert (np.all(lab == ol, axis=1)).mean() >= 0.98
    # a node that really carries the mark (byte 6 of its record, slim.h:1776-1781) is refused loudly
    hdr = off + 1
    img[hdr + 6] |= 1
    marked = str(tmp_path / "marked.graph")
    open(marked, "wb").write(bytes(img))
    with pytest.raises(capi.HsError):
        capi.Index(marked, dim)


def test_submit_wait_oldest_ring(small_corpus):
    """hs_search_batch_wait_oldest retires batches in submission order, also past the 16-entry
    completion ring."""
    import torch
    c = small_corpus
    ix = capi.Index(c.graph, c.dim)
    ix.set_ef(40)
    ix.set_overlap(True)
    k, nq = 10, c.queries.shape[0]
    nb, depth = 40, 3
    batches = [np.ascontiguousarray(np.roll(c.queries, s, axis=0)) for s in range(nb)]
    want = [ix.search(b, k)[0] for b in batches]
    hq = [torch.from_numpy(b).pin_memory() for b in batches]
    hl = [torch.full((nq, k), -1, dtype=torch.int32).pin_memory() for _ in range(depth)]
    got = []
    for i in range(nb):
        if i >= depth:
            ix.wait_oldest()
            got.append(hl[i % depth].numpy().view(np.uint32).copy())
        ix.submit_ptr(hq[i].data_ptr(), nq, k, hl[i % depth].data_ptr(), None)
    for i in range(nb - depth, nb):
        ix.wait_oldest()
        got.append(hl[i % depth].numpy().view(np.uint32).copy())
    ix.wait_oldest()                                   # nothing outstanding: returns at once
    for i in range(nb):
        assert np.array_equal(got[i], want[i]), i
    # 20 submits without any wait: the ring retires the oldest ones itself
    outs = [torch.full((nq, k), -1, dtype=torch.int32).pin_memory() for _ in range(20)]
    for i in range(20):
        ix.submit_ptr(hq[i].data_ptr(), nq, k, outs[i].data_ptr(), None)
    ix.wait()
    for i in range(20):
        assert np.array_equal(outs[i].numpy().view(np.uint32), want[i]), i


FUZZ = [
    # n,    dim, M,  metric, thr, branching, ef,  k,   kind,   prune
    (3000,  5,   4,  0,      0,   "4",       17,  3,   "slim", {}),     # tiny dim (scalar query loads), tiny M
    (3000,  17,  6,  1,      0,   "e",       33,  33,  "slim", {}),     # k > 32 with ef == k, inner product, odd dim
    (5000,  96,  24, 0,      0,   "16",      64,  10,  "slim", {}),     # CPL=3 register variant
    (5000,  128, 48, 0,      0,   "4",       128, 10,  "slim", dict(top_M0=96, low_m0=80, top_M=48, low_m=40)),  # 3 adjacency segments
    (4000,  64,  16, 1,      1,   "4",       100, 10,  "slim", {}),     # layered beam + inner product
    (4000,  200, 12, 0,      2,   "sqrt",    257, 20,  "slim", {}),     # shared-memory pool (ef > 256), generic dim
    (2000,  33,  8,  0,      0,   "4",       1000, 100, "slim", {}),    # ef half the index: hash resets likely, large k
    (300,   8,   8,  0,      0,   "4",       400, 10,  "slim", {}),     # ef larger than the index: every node visited
    (5000,  48,  24, 0,      0,   "4",       90,  10,  "hnsw", {}),     # un-pruned index, maxM0 = 48 -> two segments
    (3000,  20,  40, 1,      0,   "16",      200, 50,  "hnsw", {}),     # un-pruned, maxM0 = 80, upper rows of 40 ids
]


@pytest.mark.parametrize("n,dim,M,metric,thr,branching,ef,k,kind,prune", FUZZ)
def test_unusual_shapes_match_oracle(n, dim, M, metric, thr, branching, ef, k, kind, prune, tmp_path):
    """Bit-exact parity on shapes away from the benchmark configurations, graphs from the engine's
    own builders (also exercises them: the oracle must be able to read what they wrote)."""
    base, q = make_dataset(n, 150, dim, metric=metric, rank=min(dim, 6), seed=n + dim)
    g = str(tmp_path / "f.graph")
    if kind == "hnsw":
        capi.build_hnsw_graph(base, g, metric=metric, M=M, ef_construction=60, branching=branching)
        ix = capi.Index(g, dim, kind=capi.HS_KIND_HNSW, metric=metric)
        orc = rh.Oracle(g, dim, metric, hnsw=True)
    else:
        capi.build_slim_graph(base, g, metric=metric, M=M, ef_construction=60, branching=branching,
                              threshold_level=thr, **prune)
        ix = capi.Index(g, dim, metric=metric)
        orc = rh.Oracle(g, dim, metric)
    ix.set_ef(ef)
    lab, dist, cnt = ix.search(q, k, counts=True)
    ol, od, ond, onh = orc.search(q, k, ef, order=rh.ORDER_GPU, team=8)
    same = np.all(lab == ol, axis=1)
    assert same.mean() >= 0.99, same.mean()
    assert np.array_equal(dist[same].view(np.uint32), od[same].view(np.uint32))
    assert (cnt[same, 1] == onh[same]).mean() >= 0.99
    fin = np.isfinite(od)
    np.testing.assert_allclose(dist[fin], od[fin], rtol=REL_TOL, atol=1e-6)
