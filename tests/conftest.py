"""Shared fixtures.  `-m "not gpu"` runs on the CPU container (oracle, loader, ABI);
`-m gpu` runs on a B200 and calls the CUDA path through the C ABI.

Corpus graphs are built single-threaded, so that every machine sees the same graph, and cached
under a temp dir: with the REFERENCE builder where the compiled reference (oracle/_ref) exists,
with the engine's own host builder (hs_build_slim_graph) elsewhere.  Tests that run the reference
itself skip without it; the golden tests check the small fixtures in tests/golden/, which hold
outputs the reference produced on those fixtures only.
"""
from __future__ import annotations

import hashlib
import os
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from hnsw_slim_b200 import build as hs_build  # noqa: E402
from hnsw_slim_b200 import capi as hs_capi  # noqa: E402
from hnsw_slim_b200.synth import make_dataset  # noqa: E402
from oracle import refharness as rh  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
CACHE = os.environ.get("HS_TEST_CACHE", os.path.join(tempfile.gettempdir(), "hs_test_cache"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def _have_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


HAVE_GPU = _have_gpu()
HAVE_REF = rh.ref_slim_path() is not None


def pytest_collection_modifyitems(config, items):
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords and not HAVE_GPU:
            item.add_marker(skip_gpu)


@pytest.fixture(scope="session", autouse=True)
def _built_libraries():
    """The engine (.so) and the C oracle must exist; build them if the tree is fresh."""
    hs_build.build()
    rh.build(ref=rh.have_reference_tree() and not (HAVE_REF and rh.ref_hnsw_path()), oracle=True)
    yield


needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref (compiled reference) not available on this host")
needs_ref_hnsw = pytest.mark.skipif(rh.ref_hnsw_path() is None, reason="oracle/_ref/libhsref_hnsw_*.so not available on this host")


class Corpus:
    """A synthetic corpus + a single-threaded .graph over it (reference builder if present, else the engine's)."""

    def __init__(self, n, nq, dim, metric=0, M=16, efc=200, rank=8, branching="4", seed=1, **prune):
        self.n, self.nq, self.dim, self.metric, self.M = n, nq, dim, metric, M
        self.base, self.queries = make_dataset(n, nq, dim, metric=metric, rank=rank, seed=seed)
        # built SINGLE-THREADED: a multi-threaded build gives a different graph on every run, and a parity
        # suite must see the same graph (and the same distance ties) on every box
        builder = "reference" if HAVE_REF else "engine"
        key = hashlib.sha1(repr(("1thread", builder, n, dim, metric, M, efc, rank, branching, seed,
                                 sorted(prune.items()))).encode()).hexdigest()[:16]
        os.makedirs(CACHE, exist_ok=True)
        self.graph = os.path.join(CACHE, f"slim_{key}.graph")
        if not os.path.exists(self.graph):
            tmp = self.graph + f".tmp{os.getpid()}"
            if HAVE_REF:
                rh.ref_slim_build(self.base, tmp, metric=metric, M=M, ef_construction=efc, branching=branching,
                                  threads=1, **prune)
            else:
                hs_capi.build_slim_graph(self.base, tmp, metric=metric, M=M, ef_construction=efc, branching=branching,
                                         threads=1, **prune)
            os.replace(tmp, self.graph)


_corpora: dict = {}


def get_corpus(**kw) -> Corpus:
    key = repr(sorted(kw.items()))
    if key not in _corpora:
        _corpora[key] = Corpus(**kw)
    return _corpora[key]


@pytest.fixture(scope="session")
def small_corpus():
    """20k x 32, L2, M=16: CPL=1 kernel variant, finishes in ~1 s on the CPU."""
    return get_corpus(n=20000, nq=300, dim=32)
