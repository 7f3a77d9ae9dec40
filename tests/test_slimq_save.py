"""CPU suite for saving hnsw_slimq indices: the f_error factor the file carries and the argument checks of
hs_save_index.

f_error is the third factor of every record (one_bit_code_with_factor, rabitq_impl.hpp:76-135).  No search path
reads it, so until hs_save_index wrote it back nothing checked it: the host builder's value must equal the float64
formula on payload_reference's residual within 1 ulp, and be 0 where the residual is 0 (the ip_resi == 0 -> inf
branch)."""
import ctypes as C

import numpy as np
import pytest

from build_reference import nearest_centroid, payload_reference, read_slimq_payload, rotate_f32, rotation_shape, ulp_distance
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset

HS_ERR_ARG = -1


def f_error_reference(residual: np.ndarray) -> np.ndarray:
    """f_error of one_bit_code_with_factor (rabitq_impl.hpp:76-135, L2) as build_slimq_graph computes it, from
    payload_reference's fp32 residual: the same sums in double, left to right, ip_resi == 0 -> inf, in float64."""
    r = np.asarray(residual, np.float32).astype(np.float64)
    pd = r.shape[1]
    xu = np.where(r > 0, 0.5, -0.5)
    l2 = np.cumsum(r * r, axis=1)[:, -1]
    ip_resi = np.cumsum(r * xu, axis=1)[:, -1]
    ip_resi = np.where(ip_resi == 0, np.inf, ip_resi)
    tmp_err = np.sqrt(l2) * 1.9 * np.sqrt(np.maximum(0.0, (l2 * (pd * 0.25) / (ip_resi * ip_resi) - 1.0) / (pd - 1)))
    return (2 * tmp_err).astype(np.float32)


@pytest.mark.parametrize("dim", [64, 96, 100, 128, 200, 960, 2048])
def test_host_f_error_equals_the_reference(dim, tmp_path):
    n, nc = (1003, 16) if dim < 2048 else (301, 8)
    base, _ = make_dataset(n, 1, dim, rank=10, seed=2)
    centroids = base[np.random.default_rng(1).choice(n, nc, replace=False)].copy()
    zero = [5, 7]
    base[zero] = centroids[[2, 0]]                     # zero residual: ip_resi == 0 -> the inf branch
    cid, gap, bound = nearest_centroid(base, centroids)
    assert (gap > bound).all()
    path = str(tmp_path / "q.graph")
    capi.build_slimq_graph(base, path, M=8, ef_construction=32, centroids=centroids, cluster_ids=cid, threads=1)
    f = read_slimq_payload(path)
    pd, _ = rotation_shape(dim)
    ref = payload_reference(rotate_f32(base, dim, pd, f["flip"]), f["centroids"], cid)
    assert np.array_equal(ref["codes"], f["codes"])
    ulps = ulp_distance(f["f_error"], f_error_reference(ref["residual"]))
    assert ulps.max() <= 1, (int(ulps.max()), int(np.argmax(ulps)))
    still = ~ref["residual"].any(axis=1)               # the rows above and the rows the centroids were taken from
    assert still[zero].all() and still.sum() < n // 10
    assert (f["f_error"][still].view(np.uint32) == 0).all()
    assert np.isfinite(f["f_error"]).all() and (f["f_error"][~still] > 0).all()


def test_reference_f_error_catches_a_changed_constant(tmp_path):
    """The formula's 1.9 and its pd - 1 denominator matter: a changed constant moves every factor by far more
    than 1 ulp."""
    dim, n = 96, 400
    base, _ = make_dataset(n, 1, dim, rank=10, seed=4)
    centroids = base[:4].copy()
    cid, _, _ = nearest_centroid(base, centroids)
    path = str(tmp_path / "q.graph")
    capi.build_slimq_graph(base, path, M=8, ef_construction=32, centroids=centroids, cluster_ids=cid, threads=1)
    f = read_slimq_payload(path)
    ref = payload_reference(rotate_f32(base, dim, 128, f["flip"]), f["centroids"], cid)
    moved = ulp_distance(f["f_error"] * np.float32(1.9 / 2.0), f_error_reference(ref["residual"]))
    assert (moved[4:] > 1000).all()


def test_save_index_argument_checks():
    """A null handle or a null path is refused before anything else is looked at (no device needed)."""
    L = capi.lib()
    assert L.hs_save_index(None, b"/tmp/never-written.graph") == HS_ERR_ARG
    assert L.hs_save_index(None, None) == HS_ERR_ARG
    assert L.hs_save_index(C.c_void_p(8), None) == HS_ERR_ARG     # the path check comes before the handle is read
    ix = capi.Index.__new__(capi.Index)
    ix._h = C.c_void_p()
    with pytest.raises(capi.HsError) as e:
        ix.save("/tmp/never-written.graph")
    assert e.value.code == HS_ERR_ARG
