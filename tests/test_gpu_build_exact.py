"""GPU suite: the device builder's deterministic steps (csrc/graph_gpu.cu) list by list and bit by bit.

Conversion: hs_debug_convert_gpu runs the builder's phase 2 (convertFromHNSW: prune_kernel, the reverse-edge
sort, merge_kernel) on the un-pruned lists of a single-threaded host HNSW build; hs_build_slim_graph converts
the same lists on the host.  On integer and equal-row data every list equals the host's and
convert_reference's, in order; on float data every list outside the reference's uncertain mask does.

Payload: hs_build_slimq_index_gpu's slimq_payload_kernel against the host file with the same centroids and
seed (flip bits, rotated centroids), the float64 nearest centroid, and rotate_f32 + payload_reference.

Phase 1 (the batched HNSW insert) follows another insertion schedule than the host builder by design and is
covered by test_gpu_build.py.

Measured on a B200 (power limit 1000 W): the float cases left 27 of 3983 lists uncertain (copies), 1630 of 26513
(latent-20k) and 61 of 26513 (ip_raw-20k), and every list matched; every f_add and f_rescale equalled the
reference bit for bit."""
import ctypes as C

import numpy as np
import pytest

from build_reference import (build_host_pair, convert_reference, graph_lists, list_mismatches, nearest_centroid,
                             payload_reference, read_slimq_payload, rotate_f32, rotation_shape, ulp_distance)
from exact_regimes import make_regime
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset

pytestmark = pytest.mark.gpu

HS_ERR_UNSUPPORTED = -5
NON_DEFAULT = dict(top_degree_percent=0.3, top_M0=40, low_m0=12, top_M=12, low_m=6)

# (regime, n, dim, metric, M, branching, pruning parameters): one boundary each
CONVERT_CASES = {
    "d128-cpl4": ("integer", 3000, 128, 0, 16, "4", {}),
    "d96-cpl3": ("integer", 3000, 96, 0, 16, "4", {}),
    "d64-smem": ("integer", 3000, 64, 0, 16, "4", {}),
    "d200-smem": ("integer", 3000, 200, 0, 16, "4", {}),
    "M32-second-segment": ("integer", 4000, 64, 0, 32, "4", dict(low_m0=40)),
    "M8-topM-above-maxM": ("integer", 3000, 32, 0, 8, "4", {}),
    "ip": ("integer", 3000, 32, 1, 8, "4", {}),
    "ip-threshold1": ("integer", 3000, 32, 1, 8, "4", dict(threshold_level=1)),
    "threshold1": ("integer", 3000, 64, 0, 16, "4", dict(threshold_level=1)),
    "threshold2": ("integer", 3000, 64, 0, 16, "4", dict(threshold_level=2)),
    "threshold-above-maxlevel": ("integer", 3000, 64, 0, 16, "4", dict(threshold_level=30)),
    "branching-e": ("integer", 3000, 64, 0, 16, "e", {}),
    "branching-sqrt": ("integer", 3000, 64, 0, 16, "sqrt", {}),
    "pct-and-degrees": ("integer", 3000, 64, 0, 16, "4", NON_DEFAULT),
    "copies": ("copies", 3000, 200, 0, 8, "4", {}),
    "constant": ("constant", 2000, 32, 0, 8, "4", {}),
    "n1": ("integer", 1, 64, 0, 16, "4", {}),
    "n2": ("integer", 2, 64, 0, 16, "4", {}),
    "n33": ("integer", 33, 64, 0, 16, "4", {}),
    "latent-20k": ("latent", 20000, 128, 0, 16, "4", {}),
    "ip_raw-20k": ("ip_raw", 20000, 64, 1, 16, "4", {}),
}


@pytest.mark.parametrize("case", list(CONVERT_CASES))
def test_gpu_conversion_equals_host_and_reference(case, tmp_path):
    regime, n, dim, metric, M, branching, prune = CONVERT_CASES[case]
    base, _ = make_regime(regime, n, 1, dim, seed=3, metric=metric)
    hp, sp = build_host_pair(base, str(tmp_path), metric=metric, M=M, branching=branching, **prune)
    levels, hnsw = graph_lists(hp, dim, capi.HS_KIND_HNSW)
    _, host = graph_lists(sp, dim)
    ref = convert_reference(levels, hnsw, base, metric, dict(prune, maxM=M, maxM0=2 * M))
    ix = capi.Index.convert_gpu(hp, dim, metric=metric, **prune)
    gp = str(tmp_path / "gpu.graph")
    ix.save(gp)
    _, gpu = graph_lists(gp, dim)
    total = sum(len(x) for x in host)
    print(f"{case}: {len(ref.uncertain)} uncertain of {total} lists")
    assert list_mismatches(ref.lists, host, ref.uncertain) == []
    bad = list_mismatches(ref.lists, gpu, ref.uncertain)
    assert bad == [], (len(bad), [(v, l, ref.lists[l][v].tolist(), gpu[l][v].tolist()) for v, l in bad[:3]])
    gi, hi = ix.info(), capi.HostGraph(sp, dim).info()
    keys = ["maxlevel", "enterpoint", "n_upper", "threshold_level", "maxM", "maxM0", "M"]
    if regime in ("integer", "constant"):
        assert not ref.uncertain                   # exact distances or equal rows: every list is decided
        keys += ["max_deg0", "sum_deg0"]
    assert {k: gi[k] for k in keys} == {k: hi[k] for k in keys}
    if case == "M32-second-segment":               # lists past 32 ids in the first prune and in the result
        assert max(len(x) for x in ref.first[0].values()) > 32 and gi["max_deg0"] > 32


def _convert_status(hp, dim, **prune):
    """hs_debug_convert_gpu's status, message and whether it handed out an index."""
    L = capi.lib()
    p = capi.BuildParams()
    L.hs_build_params_default(C.byref(p))
    for k, v in prune.items():
        setattr(p, k, v)
    out = C.c_void_p()
    rc = L.hs_debug_convert_gpu(hp.encode(), dim, 0, C.byref(p), 0, C.byref(out))
    return rc, L.hs_last_error().decode(), out.value


def test_gpu_conversion_errors(tmp_path):
    base, _ = make_regime("integer", 600, 1, 32, seed=3)
    hp, _ = build_host_pair(base, str(tmp_path), M=16)
    rc, msg, out = _convert_status(hp, 32, top_M0=65)
    assert rc == HS_ERR_UNSUPPORTED and "64" in msg and out is None
    wide = tmp_path / "m48"
    wide.mkdir()
    hp48, _ = build_host_pair(base, str(wide), M=48)
    rc, msg, out = _convert_status(hp48, 32)
    assert rc == HS_ERR_UNSUPPORTED and "64" in msg and out is None


def test_gpu_conversion_refuses_a_merge_set_over_capacity(tmp_path):
    """The origin among unit rows is every row's nearest neighbour, so every first prune keeps it and its
    reverse-edge union outgrows merge_kernel's 2048 slots: an error, not a truncated list.  The origin takes the
    row the level draw makes the entry point (levels depend on the seed and the row only), so that every search
    of both builders starts there; with seed 112 that row comes early (46), so the host builder, which inserts in
    row order, links nearly every row to the origin, as the device builder does by inserting it first."""
    dim, n, seed = 64, 4000, 112
    hub = np.random.default_rng(7).standard_normal((n, dim)).astype(np.float32)
    hub /= np.linalg.norm(hub, axis=1, keepdims=True)
    draw = tmp_path / "draw"
    draw.mkdir()
    levels, _ = graph_lists(build_host_pair(hub, str(draw), M=16, seed=seed)[0], dim, capi.HS_KIND_HNSW)
    ep = int(np.argmax(levels))                   # the first node of the top level
    hub[ep] = 0
    hp, _ = build_host_pair(hub, str(tmp_path), M=16, seed=seed)
    assert capi.HostGraph(hp, dim, kind=capi.HS_KIND_HNSW).info()["enterpoint"] == ep
    levels, hnsw = graph_lists(hp, dim, capi.HS_KIND_HNSW)
    ref = convert_reference(levels, hnsw, hub, 0, dict(maxM=16, maxM0=32))
    assert ref.merged[0][ep] > 2048, ref.merged[0][ep]
    rc, msg, out = _convert_status(hp, dim)
    assert rc == HS_ERR_UNSUPPORTED and "2048" in msg and out is None, (rc, msg)
    with pytest.raises(capi.HsError) as e:
        capi.Index.build_gpu(hub, M=16, ef_construction=64, seed=seed)
    assert e.value.code == HS_ERR_UNSUPPORTED and "2048" in str(e.value)


def _check_payload(base, centroids, tmp_path, seed=11, zero_rows=()):
    """GPU payload against the host file (same centroids and seed) and the reference.  -> the GPU payload and
    the reference's (f_add, f_rescale are within 1 ulp of it; the count that is not bit-equal is printed)."""
    n, dim = base.shape
    pd, _ = rotation_shape(dim)
    cid, gap, bound = nearest_centroid(base, centroids)
    hq = str(tmp_path / "hq.graph")
    capi.build_slimq_graph(base, hq, M=8, ef_construction=32, centroids=centroids, cluster_ids=cid, threads=1,
                           seed=seed)
    f = read_slimq_payload(hq)
    gpu = capi.Index.build_gpu(base, kind=capi.HS_KIND_SLIMQ, M=8, ef_construction=32, centroids=centroids, seed=seed)
    info = gpu.info()
    assert info["padded_dim_q"] == pd and info["num_cluster"] == len(centroids) and info["n"] == n
    g = gpu.slimq_payload()
    assert np.array_equal(g["flip"], f["flip"])
    assert np.array_equal(g["centroids"].view(np.uint32), f["centroids"].view(np.uint32))
    binding = gap > bound
    assert np.array_equal(g["cluster"][binding], cid[binding])
    assert (g["cluster"] < len(centroids)).all()
    ref = payload_reference(rotate_f32(base, dim, pd, f["flip"]), f["centroids"], g["cluster"])
    assert np.array_equal(g["codes"], ref["codes"]), np.nonzero((g["codes"] != ref["codes"]).any(1))[0][:8]
    off = 0
    for k in ("f_add", "f_rescale"):
        ulps = ulp_distance(g[k], ref[k])
        assert ulps.max() <= 1, (k, int(ulps.max()), np.argmax(ulps))
        off += int((g[k].view(np.uint32) != ref[k].view(np.uint32)).sum())
    for i in zero_rows:                           # residual 0: ip_resi == 0 takes the inf branch
        assert g["f_add"][i] == 0 and g["f_rescale"][i].view(np.uint32) == 0x80000000, i
        assert not g["codes"][i].any()
    # the loader's conversion of the host file's code words gives the same records
    loaded = capi.Index(hq, dim, kind=capi.HS_KIND_SLIMQ, raw_base=base).slimq_payload()
    for k in ("codes", "cluster", "flip"):
        assert np.array_equal(loaded[k], f[k]), k
    for k in ("f_add", "f_rescale", "centroids"):
        assert np.array_equal(loaded[k].view(np.uint32), f[k].view(np.uint32)), k
    print(f"dim {dim}, {len(centroids)} centroids: {int((~binding).sum())} near-tie rows, "
          f"{off} of {2 * n} factors 1 ulp off the reference")
    return g, ref


@pytest.mark.parametrize("dim,nc", [(64, 16), (96, 16), (100, 16), (128, 1), (128, 100), (200, 16), (960, 16),
                                    (1000, 16), (2048, 16)])
def test_gpu_payload_equals_host_and_reference(dim, nc, tmp_path):
    n = 2003                                      # not a multiple of the kernel's 4 rows per block
    base, _ = make_dataset(n, 1, dim, rank=10, seed=2)
    centroids = base[np.random.default_rng(1).choice(n, nc, replace=False)].copy()
    zero = [5, 7, n - 1]
    base[zero] = centroids[[min(2, nc - 1), 0, nc - 1]]
    _check_payload(base, centroids, tmp_path, zero_rows=zero)


def test_gpu_payload_many_centroids_and_duplicates(tmp_path):
    """4096 centroids (128 chunks of 32), three of them equal (3, 35, 100: three different chunks): rows nearest
    to that content belong to centroid 3."""
    n, dim, nc = 5001, 128, 4096
    base, _ = make_dataset(n, 1, dim, rank=10, seed=8)
    centroids = make_dataset(nc, 1, dim, rank=10, seed=9)[0]
    centroids[[35, 100]] = centroids[3]
    base[[10, 11, 12]] = centroids[[3, 35, 100]]
    g, _ = _check_payload(base, centroids, tmp_path, zero_rows=[10, 11, 12])
    assert (g["cluster"][[10, 11, 12]] == 3).all() and not np.isin(g["cluster"], [35, 100]).any()


def test_gpu_payload_exact_zero_residual_coordinates(tmp_path):
    """Integer rows around integer centroids in 64 dims: the fp32 rotation is exact (|x|_2 < 2^11, scale 1/8), so
    some residual coordinates are exactly 0 and must give bit 0 (r > 0 is the sign rule)."""
    n, dim = 3001, 64
    rng = np.random.default_rng(5)
    proto = rng.integers(0, 256, (40, dim))
    noise = rng.integers(-2, 3, (n, dim)) * (rng.random((n, dim)) < 0.1)
    base = np.clip(proto[rng.integers(0, 40, n)] + noise, 0, 255).astype(np.float32)
    centroids = proto.astype(np.float32)
    _, ref = _check_payload(base, centroids, tmp_path)
    assert (nearest_centroid(base, centroids)[2] == 0).all()      # exact distances: every row's argmin binds
    moved = (base != centroids[ref["cluster"]]).any(1)
    assert ((ref["residual"] == 0) & moved[:, None]).sum() > 0


@pytest.mark.parametrize("dim", [63, 2049])
def test_gpu_payload_refuses_dims_outside_the_rotator(dim):
    base, _ = make_dataset(100, 1, dim, rank=10, seed=2)
    with pytest.raises(capi.HsError) as e:
        capi.Index.build_gpu(base, kind=capi.HS_KIND_SLIMQ, M=8, ef_construction=32, centroids=base[:4])
    assert e.value.code == HS_ERR_UNSUPPORTED
