"""Data regimes for the exact-kNN kernels and a float64 yardstick to judge their rows by.

Every regime is a deterministic function of (n, nq, dim, seed) and stresses a different part of
the exact paths (bruteforce.cu's fp32 scan, bruteforce_tc.cu's tcgen05 filter + re-scoring):

  latent    the latent-Gaussian corpus of synth.make_dataset (unit-normalised rows for IP)
  integer   values 0..255 stored as float32, as SIFT is: clusters of near-identical rows, so the
            distances are small exact integers and ties at the k-th boundary are common
  offset    1000 + a latent part: |x|^2 - 2<q,x> cancels catastrophically (tc error bound ~1e4)
  ip_raw    IP on unnormalised rows with norms spread over 0.1 .. 10: <q,x> > 1 happens, so some
            distances 1 - <q,x> are negative
  outlier   latent plus one row scaled by 1e3: the largest row norm (and the tc threshold) blows up
  copies    each row present 3 times, at labels i, i + m, i + 2m (m = ceil(n / 3)): members of a tie
            group land in different base splits
  constant  all rows equal: every candidate heap overflows

The yardstick computes distances in float64 as differences (L2) or as a float64 dot product (IP)
and bounds the error of the kernels' fp32 arithmetic (one fma chain in index order, u = 2^-24):
  L2: |d32 - d64| <= (dim + 3) u d64          IP: |d32 - d64| <= (dim + 1) u sum|q_i x_i| + u |d64|
check_topk judges result rows with it; bit-exactness against the oracle is checked separately.
"""
from __future__ import annotations

import numpy as np
import torch

from hnsw_slim_b200.synth import latent_gaussian

REGIMES = ("latent", "integer", "offset", "ip_raw", "outlier", "copies", "constant")
U = 2.0 ** -24


def outlier_label(n: int) -> int:
    return n // 2


def _latent(n, nq, dim, seed, normalize):
    rank = max(1, min(12, dim))
    base = latent_gaussian(n, dim, rank=rank, seed=seed, normalize=normalize)
    q = latent_gaussian(nq, dim, rank=rank, seed=seed, normalize=normalize, stream=1)
    return base, q


def make_regime(name: str, n: int, nq: int, dim: int, seed: int = 1, metric: int = 0):
    """(base[n, dim], queries[nq, dim]) float32 of the named regime.  `metric` matters only where
    the regime has an IP flavour (latent, outlier, copies, constant normalise for IP); ip_raw is
    meant for IP, integer and offset for L2."""
    rng = np.random.default_rng([seed, dim, 0xE8AC7])
    ip = metric == 1
    if name == "latent":
        return _latent(n, nq, dim, seed, ip)
    if name == "integer":
        # prototypes in 0..255, rows = prototype + sparse +-1/+-2 noise (clipped); half the queries
        # are perturbed base rows, half fresh members of a cluster
        n_proto = max(1, n // 64)
        proto = rng.integers(0, 256, (n_proto, dim))

        def members(cnt):
            noise = rng.integers(-2, 3, (cnt, dim)) * (rng.random((cnt, dim)) < 0.1)
            return proto[rng.integers(0, n_proto, cnt)] + noise

        base = np.clip(members(n), 0, 255).astype(np.float32)
        nq0 = nq // 2
        q0 = base[rng.integers(0, n, nq0)] + rng.integers(-1, 2, (nq0, dim)) * (rng.random((nq0, dim)) < 0.05)
        q = np.concatenate([q0, members(nq - nq0)])
        return base, np.clip(q, 0, 255).astype(np.float32)
    if name == "offset":
        base, q = _latent(n, nq, dim, seed, False)
        return (base + np.float32(1000)).astype(np.float32), (q + np.float32(1000)).astype(np.float32)
    if name == "ip_raw":
        base, q = _latent(n, nq, dim, seed, True)
        base *= (10.0 ** rng.uniform(-1, 1, (n, 1))).astype(np.float32)
        q *= (10.0 ** rng.uniform(-1, 1, (nq, 1))).astype(np.float32)
        return base, q
    if name == "outlier":
        base, q = _latent(n, nq, dim, seed, ip)
        base[outlier_label(n)] *= np.float32(1e3)
        return base, q
    if name == "copies":
        m = (n + 2) // 3
        proto, q = _latent(m, nq, dim, seed, ip)
        return np.ascontiguousarray(np.concatenate([proto, proto, proto])[:n]), q
    if name == "constant":
        proto, q = _latent(1, nq, dim, seed, ip)
        return np.repeat(proto, n, axis=0), q
    raise ValueError(f"unknown regime {name!r}")


def _device(device):
    if device is None:
        return torch.device("cuda" if torch.cuda.is_available() else "cpu")
    return torch.device(device)


def exact_block(base_t: torch.Tensor, q_t: torch.Tensor, metric: int):
    """float64 distances [nq, n] and their fp32 error bounds, for float64 tensors on one device."""
    dim = base_t.shape[1]
    if metric == 1:
        dot = q_t @ base_t.T
        d = 1.0 - dot
        tol = (dim + 1) * U * (q_t.abs() @ base_t.abs().T) + U * d.abs()
        return d, tol
    d = torch.empty((q_t.shape[0], base_t.shape[0]), dtype=torch.float64, device=base_t.device)
    step = max(1, (1 << 24) // max(1, q_t.shape[0] * dim))
    for r0 in range(0, base_t.shape[0], step):
        diff = q_t[:, None, :] - base_t[None, r0:r0 + step, :]
        d[:, r0:r0 + step] = (diff * diff).sum(-1)
    return d, (dim + 3) * U * d


def exact_rows(base, q, labels, metric: int, device=None):
    """float64 distances [nq, k] of the given rows and their error bounds."""
    dev = _device(device)
    b = torch.from_numpy(np.ascontiguousarray(base)).to(dev, torch.float64)
    qt = torch.from_numpy(np.ascontiguousarray(q)).to(dev, torch.float64)
    lab = torch.from_numpy(np.asarray(labels, dtype=np.int64)).to(dev)
    x = b[lab]                                              # [nq, k, dim]
    dim = b.shape[1]
    if metric == 1:
        d = 1.0 - (x * qt[:, None, :]).sum(-1)
        tol = (dim + 1) * U * (x.abs() * qt.abs()[:, None, :]).sum(-1) + U * d.abs()
    else:
        diff = x - qt[:, None, :]
        d = (diff * diff).sum(-1)
        tol = (dim + 3) * U * d
    return d.cpu().numpy(), tol.cpu().numpy()


def topk_problems(base, q, k: int, metric: int, labels, dists, device=None, limit: int = 5) -> list[str]:
    """What is wrong with result rows (labels, dists)[nq, k], nearest first, as judged in float64.
    Empty list = the rows are a correct top-k up to fp32 rounding:
      * rows sorted by (distance, label); labels distinct and < n;
      * every distance equals the float64 distance of its row within the fp32 bound;
      * no row missing that is more than two bounds closer than the true float64 k-th distance,
        and no returned row more than two bounds farther than it."""
    base = np.ascontiguousarray(base, dtype=np.float32)
    q = np.ascontiguousarray(q, dtype=np.float32)
    labels = np.asarray(labels)
    dists = np.asarray(dists, dtype=np.float32)
    n, nq = base.shape[0], q.shape[0]
    out: list[str] = []

    def bad(msg):
        if len(out) < limit:
            out.append(msg)

    if labels.shape != (nq, k) or dists.shape != (nq, k):
        return [f"shape {labels.shape} / {dists.shape}, want {(nq, k)}"]
    lab64 = labels.astype(np.int64)
    if (lab64 >= n).any() or (lab64 < 0).any():
        bad(f"labels out of range on queries {np.nonzero(((lab64 >= n) | (lab64 < 0)).any(1))[0][:8]}")
        return out
    for i in range(nq):
        if len(np.unique(lab64[i])) != k:
            bad(f"q{i}: repeated labels")
        dd, ll = dists[i].astype(np.float64), lab64[i]
        if ((dd[1:] < dd[:-1]) | ((dd[1:] == dd[:-1]) & (ll[1:] <= ll[:-1]))).any():
            bad(f"q{i}: rows not sorted by (distance, label)")
    d64, tol = exact_rows(base, q, lab64, metric, device)
    err = np.abs(dists.astype(np.float64) - d64)
    for i, j in zip(*np.nonzero(err > tol)):
        bad(f"q{i} row {j} (label {lab64[i, j]}): distance {dists[i, j]!r}, float64 {d64[i, j]!r}, bound {tol[i, j]:.3g}")

    dev = _device(device)
    b = torch.from_numpy(base).to(dev, torch.float64)
    qt = torch.from_numpy(q).to(dev, torch.float64)
    lab_t = torch.from_numpy(lab64).to(dev)
    step = max(1, min(nq, (1 << 25) // max(1, n)))
    for q0 in range(0, nq, step):
        D, T = exact_block(b, qt[q0:q0 + step], metric)
        kv, ki = torch.topk(D, k, dim=1, largest=False, sorted=True)
        kth, kth_tol = kv[:, -1:], T.gather(1, ki[:, -1:])
        returned = torch.zeros_like(D, dtype=torch.bool)
        returned.scatter_(1, lab_t[q0:q0 + step], True)
        missing = (~returned) & (D < kth - 2 * torch.maximum(T, kth_tol))
        far = returned & (D > kth + 2 * torch.maximum(T, kth_tol))
        for what, m in (("missing although closer than", missing), ("returned although farther than", far)):
            for i, j in torch.nonzero(m)[:limit].tolist():
                bad(f"q{q0 + i}: label {j} (float64 {D[i, j].item()!r}) {what} the k-th {kth[i, 0].item()!r}")
    return out


def check_topk(base, q, k: int, metric: int, labels, dists, device=None) -> None:
    problems = topk_problems(base, q, k, metric, labels, dists, device)
    assert not problems, "\n".join(problems)


def same_bits(lab_a, dist_a, lab_b, dist_b) -> bool:
    """Labels equal and distances equal bit for bit (what the scan kernel promises against the
    oracle's HSO_ORDER_SEQFMA, and the tc path against the scan kernel)."""
    da, db = np.ascontiguousarray(dist_a, np.float32), np.ascontiguousarray(dist_b, np.float32)
    return np.array_equal(np.asarray(lab_a, np.uint32), np.asarray(lab_b, np.uint32)) and \
        np.array_equal(da.view(np.uint32), db.view(np.uint32))


def kth_gap(base, q, k: int, metric: int, device=None):
    """float64 (k-th distance, (k+1)-th distance) per query: equal values are exact ties at the boundary."""
    dev = _device(device)
    D, _ = exact_block(torch.from_numpy(np.ascontiguousarray(base)).to(dev, torch.float64),
                       torch.from_numpy(np.ascontiguousarray(q)).to(dev, torch.float64), metric)
    v = torch.topk(D, k + 1, dim=1, largest=False, sorted=True).values
    return v[:, k - 1].cpu().numpy(), v[:, k].cpu().numpy()
