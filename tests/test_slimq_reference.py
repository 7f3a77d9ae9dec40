"""CPU: the hnsw_slimq oracle (oracle/hs_oracle_slimq.c) against the float64 query-side reference of
slimq_reference.py, on single-threaded host-built indices at padded dims 64 to 2048 with 1, 16 and 4096 clusters.

The oracle is what traverse_slimq.cu must equal bit for bit, and it was written next to the kernel.  Here it is
judged by things that were not: rotate_f32, the float64 codes, scalars and estimator, and the statistics of the
estimate against the exact distance, which holds whatever association or bit layout either side uses.

Measured with latent data and k-means centroids (3000 rows, 64 queries x 429 nodes): the rms relative error of the
estimate is 0.73 to 0.78 / sqrt(padded_dim) and its mean below 0.004 at every dim."""
import numpy as np
import pytest

from build_reference import read_slimq_payload, rotate_f32, rotation_shape
from hnsw_slim_b200 import capi
from hnsw_slim_b200.synth import make_dataset
from oracle import refharness as rh
from slimq_reference import (check_preparation, estimate, host_index, ip_ppc, pack_planes, query_codes,
                             query_scalars, relative_error_stats, statistics_hold, true_l2, unpack_planes)

# (dim, clusters): every dim with 16 clusters, and 1 and 4096 clusters at a few of them
CASES = [(64, 16), (96, 16), (130, 16), (200, 16), (960, 16), (1000, 16), (2048, 16),
         (96, 1), (1000, 1), (130, 4096), (2048, 4096)]
NQ = 8
NQ_STATS = 64         # the per-query bias of the estimate has sd ~0.02 at dim 64: 64 queries average it


class Case:
    def __init__(self, dim, nc, directory):
        n = 5000 if nc > 1000 else 3000
        self.dim, self.nc = dim, nc
        self.base, q = make_dataset(n, NQ, dim, rank=10, seed=dim + nc)
        self.qs = make_dataset(n, NQ_STATS, dim, rank=10, seed=dim + nc)[1]      # for the statistics
        self.path = f"{directory}/q.graph"
        self.cen, self.cid = host_index(self.path, self.base, nc)
        self.pay = read_slimq_payload(self.path)
        self.pd = rotation_shape(dim)[0]
        self.t = capi.slimq_default_tconst(self.pd)
        self.o = rh.OracleQ(self.path, self.base, t_const=self.t)
        # ordinary queries, a base row, a centroid and a constant vector
        self.q = np.concatenate([q, self.base[:1], self.cen[:1], np.full((1, dim), 0.25, np.float32)])
        self.nodes = np.arange(0, n, 7)
        self.at_centroid = np.nonzero(self.pay["f_rescale"].view(np.uint32) == 0x80000000)[0]


_cases = {}


@pytest.fixture
def case(request, tmp_path_factory):
    key = request.param
    if key not in _cases:
        _cases[key] = Case(*key, tmp_path_factory.mktemp(f"slimq{key[0]}_{key[1]}"))
    return _cases[key]


def ids(c):
    return f"d{c[0]}-c{c[1]}"


@pytest.mark.parametrize("case", CASES, ids=ids, indirect=True)
def test_oracle_preparation_equals_the_reference(case):
    rot, planes, scal, q2c = case.o.prep(case.q)
    assert np.array_equal(case.o.rotate(case.q).view(np.uint32), rotate_f32(case.q, case.dim, case.pd,
                                                                             case.pay["flip"]).view(np.uint32))
    masked = check_preparation(case.q, case.dim, case.pay, case.t, rot, planes, scal, q2c)
    # the oracle's own codes and planes are one layout
    _, _, codes = case.o.quantize(rot)
    assert np.array_equal(pack_planes(codes), planes) and np.array_equal(unpack_planes(planes, case.pd), codes)
    print(f"d{case.dim} c{case.nc}: {masked} masked plane dimensions of {case.q.size // case.dim * case.pd}")
    assert masked <= 0.01 * rot.size
    assert case.nc == 1 or (q2c[NQ + 1, 0] == 0)          # the centroid query sits on centroid 0


@pytest.mark.parametrize("case", CASES, ids=ids, indirect=True)
def test_oracle_estimates_within_the_bound(case):
    rot, planes, scal, q2c = case.o.prep(case.q)
    nodes = np.concatenate([case.nodes, case.at_centroid[:50]])
    if case.nc > 1000:
        assert len(case.at_centroid) > 0
    for i in range(len(case.q)):
        qc = unpack_planes(planes[i:i + 1], case.pd)[0]
        ip, ppc = ip_ppc(case.pay["codes"][nodes], qc)
        want, bound = estimate(case.pay["f_add"][nodes], case.pay["f_rescale"][nodes], case.pay["cluster"][nodes],
                               ip, ppc, *(float(v) for v in scal[i]), q2c[i])
        got = case.o.est(nodes, planes[i], scal[i], q2c[i]).astype(np.float64)
        assert (np.abs(got - want) <= bound).all(), (i, np.max(np.abs(got - want) / bound))
        at = np.isin(nodes, case.at_centroid)                 # f_add = 0, f_rescale = -0: exactly q2c^2
        assert np.array_equal(got[at], (q2c[i][case.pay["cluster"][nodes[at]]] ** 2).astype(np.float64))


def estimates(case, planes, scal, q2c):
    return np.stack([case.o.est(case.nodes, planes[i], scal[i], q2c[i]) for i in range(NQ_STATS)])


def exact(case):
    return np.stack([true_l2(case.base, case.qs[i], case.nodes) for i in range(NQ_STATS)])


@pytest.mark.parametrize("case", [c for c in CASES if c[1] == 16], ids=ids, indirect=True)
def test_estimator_estimates_the_distance(case):
    _, planes, scal, q2c = case.o.prep(case.qs)
    est, d = estimates(case, planes, scal, q2c), exact(case)
    mean, rms = relative_error_stats(est, d)
    print(f"d{case.dim}: mean {mean:+.4f} rms {rms:.4f} = {rms * np.sqrt(case.pd):.2f} / sqrt(pd)")
    assert statistics_hold(est, d, case.pd), (mean, rms)
    # the float64 estimator with the float64 scalars obeys the same statistics
    rot = rotate_f32(case.qs, case.dim, case.pd, case.pay["flip"])
    codes, _ = query_codes(rot, case.t)
    s = query_scalars(rot, codes, case.pay["centroids"])
    e64 = np.stack([estimate(case.pay["f_add"][case.nodes], case.pay["f_rescale"][case.nodes],
                             case.pay["cluster"][case.nodes], *ip_ppc(case.pay["codes"][case.nodes], codes[i]),
                             s["delta"][i], s["vl"][i], s["k1xsumq"][i], s["q2c"][i])[0] for i in range(NQ_STATS)])
    assert statistics_hold(e64, d, case.pd)


def swap_halves(p):
    return (p << np.uint64(32)) | (p >> np.uint64(32))


def reverse_bits(p):
    by = np.ascontiguousarray(p, np.uint64).astype(">u8").view(np.uint8).reshape(-1, 8)
    bits = np.unpackbits(by, axis=1, bitorder="big")[:, ::-1]
    return np.packbits(bits, axis=1, bitorder="big").view(">u8").astype(np.uint64).reshape(p.shape)


@pytest.mark.parametrize("case", [(96, 16), (960, 16)], ids=ids, indirect=True)
def test_reference_detects_planted_corruptions(case):
    """Each corruption of the query planes must fail the comparison with the reference layout; those the estimate
    can see must also fail the statistics.  Reversing the bit order of every word on BOTH sides (planes and node
    codes) leaves every estimate unchanged, so only the layout comparison catches it."""
    rot, planes, scal, q2c = case.o.prep(case.qs)
    d = exact(case)
    _, _, codes = case.o.quantize(rot)
    shifted = pack_planes(np.minimum(codes + 1, 15))
    for name, bad in [("swapped halves", swap_halves(planes)), ("reversed bits", reverse_bits(planes)),
                      ("code + 1", shifted)]:
        with pytest.raises(AssertionError):
            check_preparation(case.qs, case.dim, case.pay, case.t, rot, bad, scal, q2c)
        assert not statistics_hold(estimates(case, bad, scal, q2c), d, case.pd), name
    # both sides reversed: ip is unchanged (the statistics are blind to it)
    i = 0
    ip, ppc = ip_ppc(case.pay["codes"][case.nodes], codes[i])
    ip2, ppc2 = ip_ppc(reverse_bits(case.pay["codes"][case.nodes]), unpack_planes(reverse_bits(planes[:1]),
                                                                                 case.pd)[0])
    assert np.array_equal(ip, ip2) and np.array_equal(ppc, ppc2)
    # and the unmodified planes pass
    check_preparation(case.qs, case.dim, case.pay, case.t, rot, planes, scal, q2c)


@pytest.mark.parametrize("case", [(96, 16), (200, 4096), (2048, 16)], ids=ids, indirect=True)
@pytest.mark.parametrize("scale", [0.0, 1e-30])
def test_zero_query(case, scale):
    """A zero query, or one whose squares underflow, has norm 0.  The reference's fp32 quantiser divides 0 by 0 and
    every estimate is NaN, so its search walks the whole reachable graph.  The oracle (and the kernel) take
    cosv = 0: finite scalars, estimates f_add + |c|^2, and a search as long as an ordinary query's.
    Queries that overflow the fp32 norm (coordinates around 1e19 and above) still give NaN; they are out of scope."""
    z = (case.q[:1] * np.float32(scale)).astype(np.float32)
    assert (z == 0).all() or (np.float32(z.ravel()[np.abs(z).argmax()]) ** 2 == 0)
    rot, planes, scal, q2c = case.o.prep(z)
    assert np.isfinite(scal).all() and scal[0, 0] == 0 and scal[0, 1] == 0
    check_preparation(z, case.dim, case.pay, case.t, rot, planes, scal, q2c)
    for ef in (10, 100):
        _, _, _, nh, _ = case.o.search(case.q[:NQ], 10, ef)
        lab, dist, _, nhz, _ = case.o.search(z, 10, ef)
        assert nhz[0] <= 3 * np.median(nh), (ef, nhz[0], np.median(nh))
        assert (lab != 0xFFFFFFFF).all() and np.isfinite(dist).all()
    # the estimate of a node is f_add + |c|^2 + f_rescale * k1xsumq, and k1xsumq = -0.5 * sum(q') is (about) 0
    n = case.nodes
    want, bound = estimate(case.pay["f_add"][n], case.pay["f_rescale"][n], case.pay["cluster"][n], 0, 0, 0.0, 0.0,
                           float(scal[0, 2]), q2c[0])
    got = case.o.est(n, planes[0], scal[0], q2c[0]).astype(np.float64)
    assert (np.abs(got - want) <= bound).all()
