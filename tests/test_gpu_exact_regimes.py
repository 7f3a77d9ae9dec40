"""GPU: exact kNN across its numeric regimes and code paths, judged three ways.

For every case the fp32 scan kernel (bruteforce.cu) must return, bit for bit, what the oracle's
HSO_ORDER_SEQFMA brute force returns (wherever the oracle is affordable); the tcgen05 path
(bruteforce_tc.cu), streaming or with resident query tiles (HS_BF_QRES=1), must return the scan
kernel's rows bit for bit; and the rows must pass the float64 yardstick of exact_regimes.py.
Every tc case asserts that the tc path really ran (hs_debug_bf_tc_fallback() >= 0), so a silent
switch to the scan kernel cannot make it pass.

The matrix hits each boundary of the two kernels once rather than forming a product:
  * one 128-row tc tile (n = 128) and one extra row (n = 129) under HS_BF_TC=1; a second query tile
    with one live lane (nq = 129); nq = 1; many base splits with a ragged last one (nq = 5, n = 300k);
  * the L2 |x|^2 column in the last column of a k-block (dim 31, 63) or opening a new one (32);
    the last dims of resident-query mode (159 L2, 160 IP); dim 1 and 4; GIST's 960;
  * k = 16 / 17 (candidate heaps leave shared memory), 32 / 33, 100, 256, 512 (tc maximum),
    513 and 2048 (scan only), k == n;
  * the sampled prefilter ("phase A", n >= 8 max(16384, 512 k)) at k <= 32, k = 100 and k = 512.

Fallback rates (queries the tc path could not certify and handed to the scan kernel) are in
test_exact_regime's docstring.  On latent and ip_raw data they stay at or below nq / 10
(asserted); on integer, offset, outlier and constant data only correctness is asserted.
"""
import numpy as np
import pytest
import torch

from exact_regimes import check_topk, make_regime, same_bits
from hnsw_slim_b200 import capi
from oracle import refharness as rh

pytestmark = pytest.mark.gpu

ORACLE_BUDGET = 1e10           # n * nq * dim above which the CPU oracle is skipped
SQ = ("scan", "tc", "qres")    # qres only where kpad <= 160 (dim + 1 <= 160 for L2, dim <= 160 for IP)
TC = ("scan", "tc")

CASES = [
    # regime, metric, n, nq, dim, k, modes
    ("latent", 0, 128, 129, 128, 1, SQ),
    ("latent", 0, 129, 128, 31, 16, SQ),
    ("latent", 0, 128, 127, 32, 128, SQ),              # k == n
    ("latent", 1, 129, 1, 33, 17, SQ),
    ("latent", 0, 5003, 300, 63, 32, SQ),
    ("latent", 0, 5003, 129, 1, 33, SQ),
    ("latent", 0, 4099, 128, 4, 100, SQ),
    ("ip_raw", 1, 20011, 1000, 100, 10, SQ),
    ("ip_raw", 1, 6007, 129, 160, 256, SQ),
    ("latent", 0, 6007, 127, 159, 17, SQ),
    ("latent", 0, 20000, 129, 200, 512, TC),
    ("latent", 0, 3001, 33, 960, 100, TC),
    ("latent", 0, 5000, 64, 32, 513, ("scan", "tc_refused")),
    ("latent", 0, 4096, 16, 17, 2048, ("scan", "tc_refused")),
    ("latent", 1, 2048, 8, 8, 2048, ("scan",)),        # k == n at the scan maximum
    ("integer", 0, 20000, 500, 128, 10, SQ),
    ("integer", 0, 10007, 129, 32, 100, TC),
    ("offset", 0, 20000, 300, 128, 10, SQ),
    ("offset", 0, 8000, 128, 33, 17, TC),
    ("outlier", 0, 20000, 300, 128, 10, TC),
    ("outlier", 1, 9000, 129, 64, 32, TC),
    ("copies", 0, 30000, 300, 96, 16, SQ),
    ("copies", 1, 12000, 200, 768, 10, TC),
    ("constant", 0, 5000, 200, 16, 10, TC),
    ("constant", 1, 3000, 64, 128, 33, TC),
    # phase A (sampled prefilter) and many splits
    ("latent", 0, 131200, 1000, 32, 16, SQ),
    ("copies", 0, 131073, 300, 64, 32, TC),
    ("ip_raw", 1, 140001, 129, 128, 32, SQ),
    ("latent", 0, 409700, 200, 64, 100, TC),
    ("latent", 0, 2_100_001, 128, 16, 512, TC),
    ("latent", 0, 300_000, 5, 128, 10, TC),
    ("integer", 0, 200_000, 128, 128, 100, TC),
]


def case_id(c):
    regime, metric, n, nq, dim, k, modes = c
    return f"{regime}-{'ip' if metric else 'l2'}-n{n}-nq{nq}-d{dim}-k{k}-{'+'.join(modes[1:]) or 'scan'}"


def run(monkeypatch, base, q, k, metric, mode):
    """Rows of capi.bruteforce_knn with the path forced, and hs_debug_bf_tc_fallback() after it."""
    monkeypatch.setenv("HS_BF_TC", "0" if mode == "scan" else "1")
    monkeypatch.setenv("HS_BF_TC_STATS", "1")
    if mode == "qres":
        monkeypatch.setenv("HS_BF_QRES", "1")
    else:
        monkeypatch.delenv("HS_BF_QRES", raising=False)
    lab, dist = capi.bruteforce_knn(base, q, k, metric=metric)
    return lab, dist, capi.bf_tc_fallback()


def oracle_rows(base, q, k, metric):
    lab, dist = rh.oracle_bruteforce(base, q, k, metric=metric, order=rh.ORDER_SEQFMA, threads=0)
    return lab[:, ::-1], dist[:, ::-1]


def fallback_bound(regime, dim, nq):
    """nq / 10 on latent and ip_raw data.  Not at dim < 16, where neighbour gaps are of the order
    of the tc error bound, nor below 100 queries, where one fallback is already 1 %."""
    if regime in ("latent", "ip_raw") and dim >= 16 and nq >= 100:
        return nq // 10
    return None


@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_exact_regime(case, monkeypatch):
    """Fallback counts measured on a B200 (1000 W power limit), streaming and resident-query mode
    alike.  Not failures, but a note for work on the tc kernel:
      integer   0 of 500 (n 20000, dim 128, k 10), 0 of 129 (n 10007, dim 32, k 100),
                0 of 128 (n 200000, dim 128, k 100): a cluster's members spread over the base
                splits, so no split's heap overflows although the k-th boundary is tied
      offset    300 of 300 (dim 128), 128 of 128 (dim 33): with 1000 added to every coordinate
                score_eps is ~1e4, far above the gaps between neighbours
      outlier   300 of 300 (L2, dim 128); 14 of 129 (IP, dim 64)
      constant  every query (asserted)
      latent    0 everywhere except dim 1 (2 of 129); ip_raw 0 everywhere."""
    regime, metric, n, nq, dim, k, modes = case
    base, q = make_regime(regime, n, nq, dim, metric=metric)
    lab0, dist0, fb0 = run(monkeypatch, base, q, k, metric, "scan")
    assert fb0 == -1
    if n * nq * dim <= ORACLE_BUDGET:
        assert same_bits(lab0, dist0, *oracle_rows(base, q, k, metric)), "scan kernel != oracle (HSO_ORDER_SEQFMA)"
    check_topk(base, q, k, metric, lab0, dist0, device="cuda")
    for mode in modes[1:]:
        lab1, dist1, fb = run(monkeypatch, base, q, k, metric, mode)
        if mode == "tc_refused":                        # k > 512: the tc path declines, the scan kernel answers
            assert fb == -1
        else:
            assert fb >= 0, f"{mode}: the tcgen05 path did not run"
            print(f"[fallback] {case_id(case)} {mode}: {fb} of {nq}")
            bound = fallback_bound(regime, dim, nq)
            if bound is not None:
                assert fb <= bound, f"{mode}: {fb} of {nq} queries fell back to the scan kernel"
            if regime == "constant":
                assert fb == nq
        assert same_bits(lab1, dist1, lab0, dist0), f"{mode} != scan kernel"


def test_mixed_fallback_in_one_call(monkeypatch):
    """Half the queries sit on 300 identical rows (their heaps overflow and they go to the scan
    kernel through the fallback list), the other half certify on the tc path: both halves of one
    call must come back in their own rows."""
    n, nq, dim, k = 40000, 256, 64, 10
    base, q = make_regime("latent", n, nq, dim)
    base[1000:1300] = base[1000]
    q[: nq // 2] = base[1000] + np.float32(1e-3) * q[: nq // 2]
    lab0, dist0, _ = run(monkeypatch, base, q, k, 0, "scan")
    lab1, dist1, fb = run(monkeypatch, base, q, k, 0, "tc")
    assert nq // 2 <= fb < nq, fb
    assert same_bits(lab1, dist1, lab0, dist0)
    assert same_bits(lab0, dist0, *oracle_rows(base, q, k, 0))
    assert np.array_equal(lab0[: nq // 2], np.tile(np.arange(1000, 1000 + k, dtype=np.uint32), (nq // 2, 1)))


@pytest.mark.parametrize("tc", [False, True])
def test_device_entry_on_a_side_stream_equals_host_entry(tc, monkeypatch):
    n, nq, dim, k, metric = 40000, 300, 96, 100, 0
    base, q = make_regime("latent", n, nq, dim)
    want_l, want_d, _ = run(monkeypatch, base, q, k, metric, "tc" if tc else "scan")
    dev = torch.device("cuda")
    db, dq = torch.from_numpy(base).to(dev), torch.from_numpy(q).to(dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ol = torch.full((nq, k), -7, dtype=torch.int32, device=dev)
        od = torch.full((nq, k), -7.0, dtype=torch.float32, device=dev)
        capi.bruteforce_knn_device(db.data_ptr(), n, dim, dq.data_ptr(), nq, k, ol.data_ptr(), od.data_ptr(),
                                   metric=metric, stream=side.cuda_stream)
    fb = capi.bf_tc_fallback()                       # HS_BF_TC_STATS synchronises the stream
    side.synchronize()
    assert (fb >= 0) == tc
    assert same_bits(ol.cpu().numpy().view(np.uint32), od.cpu().numpy(), want_l, want_d)


def test_host_entry_rejects_k_above_n_when_the_base_is_empty():
    # regression: hs_bruteforce_knn returned HS_OK for n == 0 without writing the output rows
    q = np.ones((5, 8), np.float32)
    with pytest.raises(capi.HsError) as e:
        capi.bruteforce_knn(np.zeros((0, 8), np.float32), q, 10)
    assert e.value.code == -1
    lab, dist = capi.bruteforce_knn(np.zeros((0, 8), np.float32), np.zeros((0, 8), np.float32), 10)
    assert lab.shape == (0, 10) and dist.shape == (0, 10)
    with pytest.raises(capi.HsError) as e:
        capi.bruteforce_knn(np.ones((4, 8), np.float32), q, 5)
    assert e.value.code == -1


# ------------------------------------------------------------------ hs_topk_merge_device at its limits
def merge_reference(lab, dist, k):
    """Python sort of (float32 distance, label) over the valid entries of every part; padding
    (label 0xFFFFFFFF) skipped; fewer than k valid entries padded with (inf, 0xFFFFFFFF)."""
    parts, nq, kk = lab.shape
    out_l = np.full((nq, k), 0xFFFFFFFF, np.uint32)
    out_d = np.full((nq, k), np.inf, np.float32)
    for i in range(nq):
        l, d = lab[:, i].ravel(), dist[:, i].ravel()
        ok = l != 0xFFFFFFFF
        l, d = l[ok], d[ok]
        o = np.lexsort((l, d))[:k]
        out_l[i, : len(o)], out_d[i, : len(o)] = l[o], d[o]
    return out_l, out_d


def merge_on_device(lab, dist, k):
    parts, nq, _ = lab.shape
    tl = torch.from_numpy(np.ascontiguousarray(lab).view(np.int32)).cuda()
    td = torch.from_numpy(np.ascontiguousarray(dist)).cuda()
    ol = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    od = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    capi.topk_merge_device(tl.data_ptr(), td.data_ptr(), parts, nq, k, ol.data_ptr(), od.data_ptr(),
                           torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return ol.cpu().numpy().view(np.uint32), od.cpu().numpy()


@pytest.mark.parametrize("parts,nq,k,what", [
    (16, 5, 1024, "parts * k = 16384: P = 16384, 128 KB of shared memory, 256 threads"),
    (128, 3, 128, "parts * k = 16384 from many parts"),
    (1, 9, 1, "k = 1, one part"),
    (7, 40, 33, "negative distances"),
    (4, 6, 100, "all-padding rows"),
])
def test_topk_merge_limits(parts, nq, k, what):
    rng = np.random.default_rng(parts * 1000 + k)
    dist = (rng.standard_normal((parts, nq, k)) * 10).astype(np.float32)   # about half negative
    dist[rng.random(dist.shape) < 0.1] = -2.5                               # ties across parts
    dist[dist == 0] = 1.0                                                   # no -0.0 / +0.0 pairs
    lab = rng.choice(1 << 31, size=parts * nq * k, replace=False).astype(np.uint32).reshape(parts, nq, k)
    if what == "all-padding rows":
        lab[:, 0], dist[:, 0] = 0xFFFFFFFF, np.inf                          # query 0: nothing valid
        lab[:, 1, 1:], dist[:, 1, 1:] = 0xFFFFFFFF, np.inf                  # query 1: fewer than k valid
    got_l, got_d = merge_on_device(lab, dist, k)
    want_l, want_d = merge_reference(lab, dist, k)
    assert same_bits(got_l, got_d, want_l, want_d), what
    if what == "negative distances":
        assert (got_d < 0).any()


def test_topk_merge_rejects_more_than_16384_candidates():
    lab = np.zeros((5, 2, 3277), np.uint32)                  # 5 * 3277 = 16385
    with pytest.raises(capi.HsError):
        merge_on_device(lab, np.zeros(lab.shape, np.float32), 3277)


# ------------------------------------------------------------------ hs_recall at its limits
def recall_restated(base, q, knn, gt, K, metric):
    """SolveStrategy::recall (solve_strategy.h:67-103) as the kernel runs it: gt ids >= n are
    skipped, the rest re-ranked by (fp32 distance in the kernel's arithmetic, id), the first K
    intersected with knn as sets."""
    n, hits = base.shape[0], 0
    for i in range(q.shape[0]):
        ids = sorted(int(g) for g in gt[i] if g < n)
        ranked = sorted(ids, key=lambda g: (rh.oracle_dist(q[i], base[g], metric, order=rh.ORDER_SEQFMA), g))[:K]
        hits += len(set(ranked) & set(int(x) for x in knn[i]))
    return hits / (q.shape[0] * K)


@pytest.mark.parametrize("what", ["gt_k = 8192", "K == gt_k", "ip negative distances", "duplicate knn ids"])
def test_recall_limits(what):
    rng = np.random.default_rng(17)
    metric = 1 if what.startswith("ip") else 0
    n, nq, dim = 10000, 6, 24
    base, q = make_regime("ip_raw" if metric else "latent", n, nq, dim, metric=metric)
    gt_k, K = {"gt_k = 8192": (8192, 100), "K == gt_k": (64, 64)}.get(what, (200, 50))
    gt = np.stack([rng.permutation(n)[:gt_k] for _ in range(nq)]).astype(np.uint32)   # distinct ids, any order
    b64, q64 = base.astype(np.float64), q.astype(np.float64)
    d = np.stack([((b64[g] - qq) ** 2).sum(1) if metric == 0 else 1.0 - b64[g] @ qq for g, qq in zip(gt, q64)])
    knn = np.take_along_axis(gt, np.argsort(d, axis=1, kind="stable")[:, :K], 1)          # the right answers ...
    knn[rng.random(knn.shape) < 0.4] = n - 1                          # ... partly spoiled (repeats of n - 1)
    if what == "duplicate knn ids":
        knn[:, 1::2] = knn[:, 0::2][:, : knn[:, 1::2].shape[1]]
    if metric:
        assert (d < 0).any()
    got = capi.recall(base, q, knn, gt, K, metric=metric)
    assert abs(got - rh.oracle_recall(base, q, knn, gt, K, metric=metric)) < 1e-12, what
    assert abs(got - recall_restated(base, q, knn, gt, K, metric)) < 1e-12, what
    assert 0 < got < 1


def test_recall_skips_gt_ids_past_the_base():
    """gt ids >= n name no row: the kernel drops them from the re-ranked list (hso_recall has no n
    and would read past the base, so the comparison is with the Python restatement)."""
    rng = np.random.default_rng(5)
    n, nq, dim, gt_k, K = 3000, 12, 16, 40, 20
    base, q = make_regime("latent", n, nq, dim)
    gt, _ = capi.bruteforce_knn(base, q, gt_k)
    gt = gt.copy()
    gt[rng.random(gt.shape) < 0.3] = n + 5
    gt[0, :] = n + np.arange(gt_k)                                    # query 0: every gt id out of range
    knn = np.stack([r[rng.permutation(gt_k)][:K] for r in gt])
    knn[knn >= n] = 0
    got = capi.recall(base, q, knn, gt, K)
    assert abs(got - recall_restated(base, q, knn, gt, K, 0)) < 1e-12
    assert 0 < got < 1
