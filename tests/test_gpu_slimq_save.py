"""GPU suite: hs_save_index on hnsw_slimq indices (HierarchicalNSWSlimQ::saveIndex's format, slimq.h:1161-1216).

* Host-built files loaded with hs_load come back byte for byte.
* The reference-built goldens come back byte for byte except the 3-bit ex-code blocks (written as zeros) and the 8
  pointer bytes of each record; the saved file searches as the golden does.
* GPU-built indices (hs_build_slimq_index_gpu): the saved payload is the in-memory one bit for bit, f_error is the
  reference formula's, the lists are the device's, and the reopened file searches exactly as the in-memory index,
  for the engine, the C oracle and (where it is built) the reference's loadIndex + searchKnn.
"""
import numpy as np
import pytest

from build_reference import graph_lists, nearest_centroid, payload_reference, read_slimq_payload, rotate_f32, rotation_shape, ulp_distance
from hnsw_slim_b200 import capi, sharding
from hnsw_slim_b200.synth import make_dataset
from oracle import refharness as rh
from test_gpu_slimq import check_against_oracle
from test_oracle_slimq import GOLD, HAVE_REFQ, load_gold, same_sets
from test_slimq_save import f_error_reference

pytestmark = pytest.mark.gpu

SLIMQ = capi.HS_KIND_SLIMQ
HS_ERR_ARG, HS_ERR_IO, HS_ERR_UNSUPPORTED = -1, -2, -5


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


def _layout(raw):
    """-> n, record size, offset of the first record, offset of the ex block inside a record"""
    n, rec = (int(v) for v in np.frombuffer(raw, np.uint64, 2, 0))
    meta = np.frombuffer(raw, np.uint64, 9, 93)
    nc, pd, off_ex = int(meta[0]), int(meta[2]), int(meta[5])
    return n, rec, 166 + nc * pd * 4 + 4 * pd // 8, off_ex


# (dim, num_cluster, n, build parameters): the shapes of the round trip of host-built files
HOST_CASES = {
    "d64-nc16": (64, 16, 3000, {}),
    "d96-nc1": (96, 1, 3000, {}),
    "d100-nc16-threshold2": (100, 16, 3000, dict(threshold_level=2)),
    "d200-nc4096": (200, 4096, 5000, {}),
    "d960-nc16-e": (960, 16, 2000, dict(branching="e")),
    "d96-threshold0-e": (96, 16, 3000, dict(threshold_level=0, branching="e")),
}


@pytest.mark.parametrize("case", list(HOST_CASES))
def test_host_built_file_round_trips_byte_for_byte(case, tmp_path):
    dim, nc, n, kw = HOST_CASES[case]
    base, _ = make_dataset(n, 1, dim, rank=10, seed=5)
    rng = np.random.default_rng(6)
    centroids = base[rng.choice(n, nc, replace=False)].copy()
    labels = rng.permutation(n).astype(np.uint64) + 1000            # stored as 64 bits, kept as 32 on the device
    src, out = str(tmp_path / "src.graph"), str(tmp_path / "out.graph")
    capi.build_slimq_graph(base, src, M=16, ef_construction=64, centroids=centroids,
                           cluster_ids=nearest_centroid(base, centroids)[0], labels=labels, threads=1, seed=3, **kw)
    ix = capi.Index(src, dim, kind=SLIMQ, raw_base=base)
    ix.save(out)
    a, b = _read(src), _read(out)
    assert len(a) == len(b)
    diff = np.nonzero(np.frombuffer(a, np.uint8) != np.frombuffer(b, np.uint8))[0]
    assert diff.size == 0, f"{diff.size} bytes differ, first at {diff[:8].tolist()}"


@pytest.mark.parametrize("name", GOLD)
def test_reference_golden_round_trips(name, tmp_path):
    g, base, q, graph = load_gold(name)
    t = float(g["t_const"])
    out = str(tmp_path / "out.graph")
    capi.Index(graph, base.shape[1], kind=SLIMQ, raw_base=base).save(out)
    a, b = np.frombuffer(_read(graph), np.uint8), np.frombuffer(_read(out), np.uint8)
    assert a.size == b.size
    n, rec, el, off_ex = _layout(a.tobytes())
    free = np.zeros(a.size, bool)                       # bytes the save writes as zeros: pointer bytes and ex blocks
    recs = free[el:el + n * rec].reshape(n, rec)
    recs[:, 16:24] = True
    recs[:, off_ex:] = True
    assert np.array_equal(a[~free], b[~free]), np.nonzero((a != b) & ~free)[0][:8]
    assert not b[free].any()
    assert a[free].any()                                # the golden really has something there
    # the saved file, reloaded with the golden's t_const, searches as the oracle does on the original
    ix = capi.Index(out, base.shape[1], kind=SLIMQ, raw_base=base)
    ix.query_tconst = t
    o = rh.OracleQ(graph, base, t_const=t)
    for ef in (10, 40, 100, 200):
        check_against_oracle(ix, o, q, int(g["k"]), ef)


# (dim, num_cluster, M, pruning): the shapes of test_gpu_payload_equals_host_and_reference, M 8 and 32, threshold 2
GPU_CASES = {f"d{d}-nc{c}": (d, c, 16, {}) for d, c in [(64, 16), (96, 16), (100, 16), (128, 1), (128, 100), (200, 16),
                                                        (960, 16), (1000, 16), (2048, 16)]}
GPU_CASES.update({"d96-M8": (96, 16, 8, {}), "d96-M32": (96, 16, 32, {}),
                  "d128-threshold2": (128, 16, 16, dict(threshold_level=2))})


def _gpu_built(dim, nc, M, prune, *, n=2003, nq=200, seed=2, labels=None):
    base, q = make_dataset(n, nq, dim, rank=10, seed=seed)
    rng = np.random.default_rng(1)
    centroids = (base[rng.choice(n, nc, replace=False)] + 0.01 * rng.standard_normal((nc, dim))).astype(np.float32)
    # rows equal to a centroid (zero residual: ip_resi == 0 -> the inf branch), no two rows equal: equal rows tie
    # bit for bit, and the kernel and the oracle order tied pool entries differently (counters may then differ)
    zero = [5, 7, n - 1][:nc]
    base[zero] = centroids[:len(zero)]
    kw = dict(kind=SLIMQ, M=M, ef_construction=64, centroids=centroids, seed=11, labels=labels)
    return capi.Index.build_gpu(base, **kw, **prune), base, q, zero


def _same_search(a, b, q, ef, k):
    a.set_ef(ef)
    b.set_ef(ef)
    la, da, ca = a.search(q, k, counts=True)
    lb, db, cb = b.search(q, k, counts=True)
    assert np.array_equal(la, lb), (ef, k)
    assert np.array_equal(da.view(np.uint32), db.view(np.uint32)), (ef, k)
    assert np.array_equal(ca, cb), (ef, k)


@pytest.mark.parametrize("case", list(GPU_CASES))
def test_gpu_built_index_saves_what_it_searches(case, tmp_path):
    dim, nc, M, prune = GPU_CASES[case]
    gpu, base, q, zero = _gpu_built(dim, nc, M, prune)
    n, pd = base.shape[0], rotation_shape(dim)[0]
    path = str(tmp_path / "gpu.graph")
    gpu.save(path)

    # payload: the in-memory records, bit for bit; f_error within 1 ulp of the reference formula
    f, g = read_slimq_payload(path), gpu.slimq_payload()
    for k in ("codes", "cluster", "flip"):
        assert np.array_equal(f[k], g[k]), k
    for k in ("f_add", "f_rescale", "centroids"):
        assert np.array_equal(f[k].view(np.uint32), g[k].view(np.uint32)), k
    ref = payload_reference(rotate_f32(base, dim, pd, f["flip"]), f["centroids"], g["cluster"])
    ulps = ulp_distance(f["f_error"], f_error_reference(ref["residual"]))
    assert ulps.max() <= 1, (int(ulps.max()), int(np.argmax(ulps)))
    assert (f["f_error"][zero].view(np.uint32) == 0).all()
    raw = _read(path)
    _, rec, el, off_ex = _layout(raw)
    recs = np.frombuffer(raw, np.uint8, n * rec, el).reshape(n, rec)
    assert not recs[:, 16:24].any() and not recs[:, off_ex:].any()
    assert rec - off_ex == pd * 3 // 8 + 8

    # header and lists: those of the device graph, which the GPU hnsw_slim builder gives for the same rows and
    # seed (the phase-1 schedule is deterministic); that index is saved by the hnsw_slim writer
    info = gpu.info()
    hg = capi.HostGraph(path, dim, kind=SLIMQ).info()
    for k in ("n", "maxlevel", "threshold_level", "enterpoint", "M", "maxM", "maxM0", "ef_construction",
              "padded_dim_q", "num_cluster"):
        assert hg[k] == info[k], k
    slim_path = str(tmp_path / "slim.graph")
    capi.Index.build_gpu(base, M=M, ef_construction=64, seed=11, **prune).save(slim_path)
    lv_q, lists_q = graph_lists(path, dim, SLIMQ)
    lv_s, lists_s = graph_lists(slim_path, dim)
    assert np.array_equal(lv_q, lv_s)
    for l, (a, b) in enumerate(zip(lists_q, lists_s)):
        assert a.keys() == b.keys(), l
        bad = [v for v in a if not np.array_equal(a[v], b[v])]
        assert not bad, (l, bad[:5])
    hq = capi.HostGraph(path, dim, kind=SLIMQ)
    assert [hq.node(i)[1] for i in range(n)] == list(range(n))

    # reopened with the build's rows: the same rows, distance bits and counters
    again = capi.Index(path, dim, kind=SLIMQ, raw_base=base)
    assert again.query_tconst == gpu.query_tconst
    assert again.info()["device_bytes"] == info["device_bytes"]
    for ef in (10, 100, 300):
        for k in sorted({10, ef}):
            _same_search(gpu, again, q, ef, k)

    # the C oracle on the saved file against the in-memory index
    o = rh.OracleQ(path, base, t_const=gpu.query_tconst)
    for ef in (10, 100):
        check_against_oracle(gpu, o, q, 10, ef)

    # the reference's loadIndex + searchKnn on the saved file
    if HAVE_REFQ:
        r = rh.RefSlimQ(path, base)
        assert r.info["n"] == n and r.info["ex_bits"] == 3
        gpu.query_tconst = r.t_const
        for ef in (50, 100):
            gpu.set_ef(ef)
            lab, _ = gpu.search(q, 10)
            rlab, _ = r.search(q, 10, ef)
            assert same_sets(lab, rlab).mean() >= 0.95, ef


def test_saving_is_idempotent(tmp_path):
    gpu, base, q, _ = _gpu_built(96, 16, 16, {})
    p1, p2, p3 = (str(tmp_path / f"{i}.graph") for i in range(3))
    gpu.save(p1)
    gpu.save(p2)
    gpu.set_ef(100)
    gpu.search(q, 10)
    gpu.query_tconst = 1.5 * gpu.query_tconst
    gpu.set_ef(37)
    gpu.search(q, 5, counts=True)
    gpu.save(p3)
    assert _read(p1) == _read(p2) == _read(p3)
    # a loaded index saved twice, around searches, too
    ix = capi.Index(p1, 96, kind=SLIMQ, raw_base=base)
    ix.set_ef(200)
    ix.search(q, 50)
    ix.query_tconst = 0.5
    ix.save(p2)
    assert _read(p2) == _read(p1)


def test_saved_gpu_built_shards_open_as_a_sharded_index(tmp_path):
    import torch
    n, nq, dim, k, ef = 12000, 300, 96, 10, 80
    base, q = make_dataset(n, nq, dim, rank=10, seed=21)
    ranges = sharding.shard_ranges(n, 2)
    shards, paths, raws = [], [], []
    for s, (lo, hi) in enumerate(ranges):
        ix = capi.Index.build_gpu(base[lo:hi], kind=SLIMQ, M=16, ef_construction=100, seed=5 + s,
                                  labels=np.arange(lo, hi, dtype=np.uint64))
        p = str(tmp_path / f"s{s}.graph")
        ix.save(p)
        shards.append(ix)
        paths.append(p)
        raws.append(base[lo:hi])
    dq = torch.from_numpy(q).cuda()
    results = []
    for sx in (sharding.ShardedIndex.from_indices(shards, dim),
               sharding.ShardedIndex(paths, dim, kind=SLIMQ, raw_bases=raws)):
        sx.set_ef(ef)
        lab, dist = sx.search(dq, nq, k)
        sx.join()
        results.append((lab.cpu().numpy().view(np.uint32), dist.cpu().numpy()))
        sx.close()
    (la, da), (lb, db) = results
    assert np.array_equal(la, lb)
    assert np.array_equal(da.view(np.uint32), db.view(np.uint32))
    assert la.max() >= ranges[1][0] and la.min() < ranges[0][1]       # both shards contribute global labels


def test_save_errors(tmp_path):
    gpu, _, _, _ = _gpu_built(64, 4, 16, {}, n=500)
    bad = str(tmp_path / "no-such-dir" / "x.graph")
    with pytest.raises(capi.HsError) as e:
        gpu.save(bad)
    assert e.value.code == HS_ERR_IO and bad in str(e.value)
    assert capi.lib().hs_save_index(gpu.handle, None) == HS_ERR_ARG
    base, _ = make_dataset(500, 1, 32, rank=10, seed=3)
    hp = str(tmp_path / "hnsw.graph")
    capi.build_hnsw_graph(base, hp, M=8, ef_construction=32, threads=1)
    h = capi.Index(hp, 32, kind=capi.HS_KIND_HNSW)
    with pytest.raises(capi.HsError) as e:
        h.save(str(tmp_path / "h.graph"))
    assert e.value.code == HS_ERR_UNSUPPORTED
    assert not (tmp_path / "h.graph").exists()
