"""CPU: the regime generator and the float64 yardstick of tests/exact_regimes.py, which the GPU
exact-kNN tests (test_gpu_exact_regimes.py) rely on.  The oracle's HSO_ORDER_SEQFMA brute force —
the scan kernel's own arithmetic — must pass the yardstick on every regime, and corrupted copies of
its rows must fail it or the bitwise comparison with the oracle."""
import numpy as np
import pytest

from exact_regimes import REGIMES, check_topk, kth_gap, make_regime, outlier_label, same_bits, topk_problems
from oracle import refharness as rh


def oracle(base, q, k, metric):
    lab, dist = rh.oracle_bruteforce(base, q, k, metric=metric, order=rh.ORDER_SEQFMA)
    return np.ascontiguousarray(lab[:, ::-1]), np.ascontiguousarray(dist[:, ::-1])     # nearest first


@pytest.mark.parametrize("regime,metric,dim", [(r, 0, 37) for r in REGIMES] + [
    ("latent", 1, 37), ("ip_raw", 1, 37), ("outlier", 1, 37), ("copies", 1, 37), ("constant", 1, 37),
    ("integer", 0, 1), ("offset", 0, 128), ("ip_raw", 1, 160)])
@pytest.mark.parametrize("k", [1, 10, 33])
def test_oracle_passes_the_yardstick(regime, metric, dim, k):
    base, q = make_regime(regime, 1500, 40, dim, metric=metric)
    lab, dist = oracle(base, q, k, metric)
    check_topk(base, q, k, metric, lab, dist, device="cpu")


def test_regimes_are_deterministic():
    for r in REGIMES:
        a, b = make_regime(r, 700, 9, 20, seed=4), make_regime(r, 700, 9, 20, seed=4)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), r
        assert a[0].dtype == np.float32 and a[0].shape == (700, 20) and a[1].shape == (9, 20)
        assert not np.array_equal(a[0], make_regime(r, 700, 9, 20, seed=5)[0]), r


def test_regimes_are_what_their_names_say():
    n, nq, dim, k = 6000, 200, 64, 10
    # latent: distinct rows, no exact tie at the boundary
    base, q = make_regime("latent", n, nq, dim)
    lo, hi = kth_gap(base, q, k, 0, device="cpu")
    assert (lo < hi).all() and len(np.unique(base, axis=0)) == n
    # integer: SIFT-like values, exact ties at the k-th boundary on at least half of the queries
    base, q = make_regime("integer", n, nq, dim)
    for a in (base, q):
        assert a.min() >= 0 and a.max() <= 255 and np.array_equal(a, np.round(a))
    lo, hi = kth_gap(base, q, k, 0, device="cpu")
    assert np.array_equal(lo, np.round(lo)) and (lo == hi).mean() >= 0.5, (lo == hi).mean()
    # offset: |x|^2 dwarfs the neighbour distances (the cancellation of |x|^2 - 2<q,x>)
    base, q = make_regime("offset", n, nq, dim)
    assert abs(base.mean() - 1000) < 5 and abs(q.mean() - 1000) < 5
    lo, _ = kth_gap(base, q, k, 0, device="cpu")
    assert np.median((base.astype(np.float64) ** 2).sum(1)) > 1e4 * np.median(lo)
    # ip_raw: norms over 0.1 .. 10, some <q,x> > 1 (negative distances) and some positive distances
    base, q = make_regime("ip_raw", n, nq, dim, metric=1)
    norms = np.linalg.norm(base, axis=1)
    assert norms.min() < 0.15 and norms.max() > 7 and 0.1 <= norms.min() and norms.max() <= 10.01
    _, dist = oracle(base, q, k, 1)
    assert (dist < 0).mean() > 0.2 and (dist > 0).any()
    # outlier: one row 1e3 times the scale of the rest
    base, q = make_regime("outlier", n, nq, dim)
    norms = np.linalg.norm(base, axis=1)
    assert np.argmax(norms) == outlier_label(n) and norms.max() > 500 * np.median(norms)
    # copies: row i == row i + m == row i + 2m, so the k-th boundary falls inside a tie group
    base, q = make_regime("copies", n, nq, dim)
    m = n // 3
    assert np.array_equal(base[:m], base[m:2 * m]) and np.array_equal(base[:m], base[2 * m:])
    assert len(np.unique(base, axis=0)) == m
    lo, hi = kth_gap(base, q, k, 0, device="cpu")
    assert (lo == hi).all()                                  # k = 10 ends inside a group of 3
    # constant: one row n times
    base, q = make_regime("constant", n, nq, dim)
    assert (base == base[0]).all()


def tie_at_boundary(dist, k):
    """Queries whose k-th and (k+1)-th returned rows tie exactly (fp32, as the kernel computed them)."""
    return np.nonzero(dist[:, k - 1] == dist[:, k])[0]


def caught(base, q, k, metric, want, lab, dist):
    """(yardstick fails, bitwise comparison with the wanted rows fails)"""
    return bool(topk_problems(base, q, k, metric, lab, dist, device="cpu")), not same_bits(lab, dist, *want)


@pytest.mark.parametrize("regime,metric", [("integer", 0), ("copies", 0), ("copies", 1)])
def test_mutations_are_caught(regime, metric):
    k = 10
    base, q = make_regime(regime, 3000, 60, 48, metric=metric)
    lab1, dist1 = oracle(base, q, k + 1, metric)               # one row past the boundary
    want = (lab1[:, :k].copy(), dist1[:, :k].copy())
    assert not any(caught(base, q, k, metric, want, *want))

    # 1. the k-th and (k+1)-th members of a tie group swapped: same distance, wrong tie rule.  Only
    #    the bitwise comparison sees it (the yardstick cannot tell equal fp32 distances apart)
    ties = tie_at_boundary(dist1, k)
    assert len(ties) > 0
    i = ties[0]
    lab, dist = want[0].copy(), want[1].copy()
    lab[i, k - 1] = lab1[i, k]
    assert caught(base, q, k, metric, want, lab, dist)[1]

    # 2. two equal-distance labels inside the rows reversed: the (distance, label) order breaks
    i, j = next((i, j) for i in range(len(q)) for j in range(k - 1) if dist1[i, j] == dist1[i, j + 1])
    lab, dist = want[0].copy(), want[1].copy()
    lab[i, j], lab[i, j + 1] = lab[i, j + 1], lab[i, j]
    assert caught(base, q, k, metric, want, lab, dist) == (True, True)

    # 3. the last bit of one distance flipped: within the fp32 bound, so again the bitwise check
    lab, dist = want[0].copy(), want[1].copy()
    dist.view(np.uint32)[0, 0] ^= 1
    assert caught(base, q, k, metric, want, lab, dist)[1]


@pytest.mark.parametrize("regime,metric,dim", [("latent", 0, 32), ("latent", 1, 33), ("ip_raw", 1, 100),
                                               ("offset", 0, 64), ("integer", 0, 64)])
def test_boundary_row_replaced_by_the_next_is_caught(regime, metric, dim):
    """A boundary row replaced with the (k+1)-th row (its own distance): the returned row lies more
    than two bounds beyond the true k-th distance, and the yardstick says so."""
    k = 10
    base, q = make_regime(regime, 3000, 60, dim, metric=metric)
    lab1, dist1 = oracle(base, q, k + 1, metric)
    want = (lab1[:, :k].copy(), dist1[:, :k].copy())
    lo, hi = kth_gap(base, q, k, metric, device="cpu")
    d1 = dist1.astype(np.float64)
    i = int(np.argmax(np.minimum(hi - lo, lo - d1[:, 0])))    # clear gaps at the boundary and below it
    assert hi[i] > lo[i] > d1[i, 0]
    lab, dist = want[0].copy(), want[1].copy()
    lab[i, k - 1], dist[i, k - 1] = lab1[i, k], dist1[i, k]
    problems = topk_problems(base, q, k, metric, lab, dist, device="cpu")
    assert any(f"q{i}: label {lab1[i, k]} " in p and "farther" in p for p in problems), problems
    # the nearest row dropped for the (k+1)-th: reported missing
    lab, dist = want[0].copy(), want[1].copy()
    lab[i], dist[i] = lab1[i, 1:], dist1[i, 1:]
    problems = topk_problems(base, q, k, metric, lab, dist, device="cpu")
    assert any(f"q{i}: label {lab1[i, 0]} " in p and "missing" in p for p in problems), problems
    # ... and a wrong distance for a right row, by more than the bound, is caught too
    lab, dist = want[0].copy(), want[1].copy()
    dist[i, 0] = np.nextafter(dist[i, 0], np.float32(np.inf)) + abs(dist[i, 0]) * 1e-3 + 1e-3
    assert any("float64" in p and f"q{i} row 0" in p for p in topk_problems(base, q, k, metric, lab, dist, device="cpu"))
