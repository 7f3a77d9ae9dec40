"""CPU: the yardsticks of tests/build_reference.py, which the GPU builder tests (test_gpu_build_exact.py) rely on.
The host builder's conversion (graph_build.cpp) must equal convert_reference list by list and its hnsw_slimq
payload must equal rotate_f32 + payload_reference bit for bit; planted corruptions must be caught."""
import ctypes as C

import numpy as np
import pytest

from build_reference import (build_host_pair, convert_reference, graph_lists, list_mismatches, nearest_centroid,
                             payload_reference, read_slimq_payload, rotate_f32, rotate_f64, rotation_bound,
                             rotation_shape)
from conftest import HAVE_GPU
from exact_regimes import U, make_regime
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset


def host_and_reference(base, tmp_path, metric, M, branching="4", **prune):
    hp, sp = build_host_pair(base, str(tmp_path), metric=metric, M=M, branching=branching, **prune)
    levels, hnsw = graph_lists(hp, base.shape[1], capi.HS_KIND_HNSW)
    _, slim = graph_lists(sp, base.shape[1])
    return hp, slim, convert_reference(levels, hnsw, base, metric, dict(prune, maxM=M, maxM0=2 * M))


NON_DEFAULT = dict(threshold_level=1, top_degree_percent=0.3, top_M0=40, low_m0=12, top_M=12, low_m=6)


@pytest.mark.parametrize("regime,n,dim,metric,M,prune", [
    ("integer", 3000, 32, 0, 8, {}),
    ("integer", 3000, 32, 1, 8, {}),
    ("integer", 3000, 64, 0, 16, NON_DEFAULT),
    ("integer", 2500, 48, 1, 12, dict(NON_DEFAULT, threshold_level=2)),
    ("copies", 3000, 200, 0, 8, {}),
    ("copies", 3000, 64, 1, 8, {}),
    ("constant", 2000, 32, 0, 8, {}),
    ("latent", 5000, 64, 0, 16, {}),
])
def test_host_conversion_equals_the_reference(regime, n, dim, metric, M, prune, tmp_path):
    base, _ = make_regime(regime, n, 1, dim, seed=3, metric=metric)
    _, slim, ref = host_and_reference(base, tmp_path, metric, M, **prune)
    print(f"{regime}: {len(ref.uncertain)} uncertain of {sum(len(x) for x in slim)} lists")
    assert list_mismatches(ref.lists, slim, ref.uncertain) == []
    if regime in ("integer", "constant"):
        assert not ref.uncertain                       # exact distances (or equal rows): nothing is left open
    if regime == "latent":
        assert len(ref.uncertain) < 0.1 * sum(len(x) for x in slim)
    if prune:                                          # the parameters reached both sides
        assert any(ref.thresholds[1:]) and len(ref.lists) > prune["threshold_level"]


def test_reference_detects_planted_corruptions(tmp_path):
    base, _ = make_regime("integer", 3000, 32, 32, seed=3)
    _, slim, ref = host_and_reference(base, tmp_path, 0, 8)
    assert list_mismatches(ref.lists, slim) == []
    # a dropped reverse edge: v kept u in its first prune, so u's list holds v through the union
    v, u = next((v, int(u)) for v, f in ref.first[0].items() for u in f
                if v in ref.lists[0][int(u)] and v not in ref.first[0][int(u)])
    bad = [{k: x.copy() for k, x in lv.items()} for lv in slim]
    bad[0][u] = bad[0][u][bad[0][u] != v]
    assert list_mismatches(ref.lists, bad) == [(u, 0)]
    # two kept neighbours swapped: same set, wrong order
    w = next(k for k, x in slim[0].items() if len(x) >= 2)
    bad = [{k: x.copy() for k, x in lv.items()} for lv in slim]
    bad[0][w][[0, 1]] = bad[0][w][[1, 0]]
    assert list_mismatches(ref.lists, bad) == [(w, 0)]


@pytest.mark.parametrize("dim", [64, 96, 100, 200, 960])
def test_host_payload_equals_the_reference(dim, tmp_path):
    n, nc = 1003, 16
    base, _ = make_dataset(n, 1, dim, rank=10, seed=2)
    centroids = base[np.random.default_rng(1).choice(n, nc, replace=False)].copy()
    base[[5, 7]] = centroids[[2, 0]]                   # zero residual: ip_resi == 0 -> the inf branch
    cid, gap, bound = nearest_centroid(base, centroids)
    assert (gap > bound).all()
    path = str(tmp_path / "q.graph")
    capi.build_slimq_graph(base, path, M=8, ef_construction=32, centroids=centroids, cluster_ids=cid, threads=1)
    f = read_slimq_payload(path)
    pd, _ = rotation_shape(dim)
    assert f["codes"].shape == (n, pd // 64) and np.array_equal(f["cluster"], cid)
    assert np.array_equal(rotate_f32(centroids, dim, pd, f["flip"]).view(np.uint32), f["centroids"].view(np.uint32))
    r32 = rotate_f32(base, dim, pd, f["flip"])
    ref = payload_reference(r32, f["centroids"], cid)
    assert np.array_equal(ref["codes"], f["codes"])
    for k in ("f_add", "f_rescale"):
        assert np.array_equal(ref[k].view(np.uint32), f[k].view(np.uint32)), k
    assert (f["f_add"][[5, 7]] == 0).all() and (f["f_rescale"][[5, 7]].view(np.uint32) == 0x80000000).all()
    # the float64 rotation is orthogonal; the fp32 one stays within its bound of it
    r64, c64 = rotate_f64(base, dim, pd, f["flip"]), rotate_f64(centroids, dim, pd, f["flip"])
    x64 = base.astype(np.float64)
    assert np.allclose(np.linalg.norm(r64, axis=1), np.linalg.norm(x64, axis=1), rtol=1e-13, atol=0)
    assert np.allclose(r64 @ c64.T, x64 @ centroids.astype(np.float64).T, rtol=0, atol=1e-11 * np.abs(x64).max() ** 2 * dim)
    bx, bc = rotation_bound(base, dim), rotation_bound(centroids, dim)
    assert (np.linalg.norm(r32 - r64, axis=1) <= bx).all()
    ip32 = r32.astype(np.float64) @ f["centroids"].astype(np.float64).T
    nx, ncn = np.linalg.norm(x64, axis=1), np.linalg.norm(centroids.astype(np.float64), axis=1)
    assert (np.abs(ip32 - r64 @ c64.T) <= bx[:, None] * ncn[None] + bc[None] * nx[:, None] + 2 * U * nx[:, None] * ncn).all()
    # every code bit whose float64 residual is clear of the bound has the float64 sign
    res64 = r64 - c64[cid]
    clear = np.abs(res64) > (bx + bc[cid])[:, None] + 2 * U * np.abs(res64)
    assert clear.mean() > 0.9
    assert ((res64 > 0) == (ref["residual"] > 0))[clear].all()


def test_reference_detects_a_flipped_code_bit(tmp_path):
    dim, n = 96, 500
    base, _ = make_dataset(n, 1, dim, rank=10, seed=4)
    centroids = base[:4].copy()
    cid, _, _ = nearest_centroid(base, centroids)
    path = str(tmp_path / "q.graph")
    capi.build_slimq_graph(base, path, M=8, ef_construction=32, centroids=centroids, cluster_ids=cid, threads=1)
    f = read_slimq_payload(path)
    ref = payload_reference(rotate_f32(base, dim, 128, f["flip"]), f["centroids"], cid)
    assert np.array_equal(ref["codes"], f["codes"])
    codes = f["codes"].copy()
    codes[17, 1] ^= np.uint64(1) << np.uint64(40)
    assert np.nonzero((codes != ref["codes"]).any(1))[0].tolist() == [17]


@pytest.mark.skipif(HAVE_GPU, reason="checks the no-device error path")
def test_debug_hooks_without_a_device(tmp_path):
    base, _ = make_regime("integer", 300, 1, 32, seed=3)
    hp, _ = build_host_pair(base, str(tmp_path))
    with pytest.raises(capi.HsError) as e:
        capi.Index.convert_gpu(hp, 32)
    assert e.value.code == -3 and "no CPU fallback" in str(e.value)
    L = capi.lib()
    p = capi.BuildParams()
    L.hs_build_params_default(C.byref(p))
    out = C.c_void_p()
    assert L.hs_debug_convert_gpu(hp.encode(), 32, 0, C.byref(p), 0, None) == -1
    assert L.hs_debug_convert_gpu(None, 32, 0, C.byref(p), 0, C.byref(out)) == -1 and not out.value
    assert L.hs_debug_convert_gpu(hp.encode(), 32, 7, C.byref(p), 0, C.byref(out)) == -1 and not out.value
    assert L.hs_debug_slimq_payload(None, None, None, None) == -1
    ix = capi.Index.__new__(capi.Index)                # no device, so no index: the handle is null
    ix._h = C.c_void_p()
    with pytest.raises(capi.HsError) as e:
        ix.slimq_payload()
    assert e.value.code == -1
