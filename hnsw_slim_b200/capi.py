"""ctypes binding of include/hnswslim_b200.h (libhnswslim_b200.so).

This is the only way Python (tests, bench.py) reaches the engine: every call goes through
the same C ABI a C++ host links against.  There is no fallback: if the shared library is
missing, or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

HS_KIND_SLIM, HS_KIND_SLIMQ, HS_KIND_HNSW = 0, 1, 2
HS_METRIC_L2, HS_METRIC_IP = 0, 1

EXPORTS = [
    "hs_load", "hs_load_memory", "hs_free", "hs_set_ef", "hs_get_info", "hs_search_batch",
    "hs_search_batch_counts", "hs_search_batch_submit", "hs_search_batch_wait", "hs_search_batch_wait_oldest", "hs_pin_host", "hs_unpin_host", "hs_search_batch_device", "hs_stats", "hs_reset_stats", "hs_bruteforce_knn",
    "hs_bruteforce_knn_device", "hs_topk_merge_device", "hs_recall", "hs_last_error", "hs_abi_version",
    "hs_debug_flatten", "hs_debug_free", "hs_debug_info", "hs_debug_row", "hs_debug_node",
    "hs_build_params_default", "hs_build_slim_graph", "hs_build_hnsw_graph",
    "hs_get_query_tconst", "hs_set_query_tconst", "hs_slimq_prepare", "hs_build_slimq_graph",
    "hs_slimq_default_tconst", "hs_debug_bf_tc_fallback", "hs_set_overlap",
    "hs_search_batch_device_scatter", "hs_exchange_create", "hs_exchange_handle", "hs_exchange_connect",
    "hs_exchange_search", "hs_exchange_signal_and_wait", "hs_exchange_tables", "hs_exchange_free",
    "hs_shardgroup_create", "hs_shardgroup_handle", "hs_shardgroup_connect", "hs_shardgroup_connect_local",
    "hs_shardgroup_submit", "hs_shardgroup_wait_oldest", "hs_shardgroup_wait", "hs_shardgroup_streams",
    "hs_shardgroup_free", "hs_build_slim_index_gpu", "hs_save_index", "hs_build_slimq_index_gpu",
    "hs_load_reserve", "hs_patch_apply", "hs_debug_patch",
    "hs_service_create", "hs_service_query", "hs_service_set_ef", "hs_service_patch", "hs_service_get_stats",
    "hs_service_free", "hs_debug_service_create", "hs_set_tuning", "hs_debug_convert_gpu", "hs_debug_slimq_payload",
]
HS_PATCH_INLINE_ROWS = 1


class HsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"hnswslim_b200 error {code}: {msg}")
        self.code = code


class IndexInfo(C.Structure):
    _fields_ = [("n", C.c_uint64), ("dim", C.c_uint64), ("dim_padded", C.c_uint64), ("M", C.c_uint64),
                ("maxM", C.c_uint64), ("maxM0", C.c_uint64), ("ef_construction", C.c_uint64),
                ("maxlevel", C.c_int32), ("threshold_level", C.c_int32), ("enterpoint", C.c_uint32),
                ("has_deleted", C.c_int32), ("kind", C.c_int32), ("metric", C.c_int32),
                ("deg0_stride", C.c_uint32), ("max_deg0", C.c_uint32), ("upper_stride", C.c_uint32),
                ("n_upper", C.c_uint32), ("sum_deg0", C.c_uint64), ("device_bytes", C.c_uint64),
                ("ef", C.c_uint64), ("padded_dim_q", C.c_uint64), ("num_cluster", C.c_uint64)]

    def as_dict(self) -> dict:
        return {f: getattr(self, f) for f, _ in self._fields_}


class PatchInfo(C.Structure):
    _fields_ = [("n_before", C.c_uint64), ("n_after", C.c_uint64), ("changed_old", C.c_uint64),
                ("changed_new", C.c_uint64), ("bytes_consumed", C.c_uint64), ("rows_written", C.c_uint64),
                ("upper_rebuilt", C.c_uint64)]

    def as_dict(self) -> dict:
        return {f: int(getattr(self, f)) for f, _ in self._fields_}


class ServiceStats(C.Structure):
    _fields_ = [("batches", C.c_uint64), ("queries", C.c_uint64), ("max_batch", C.c_uint64), ("patches", C.c_uint64),
                ("busy_seconds", C.c_double)]


SERVICE_BACKEND = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p)


def _patch_args(stream: bytes, rows, row_labels, inline: bool):
    buf = np.frombuffer(stream, dtype=np.uint8)
    r = _f32(rows) if rows is not None else None
    rl = np.ascontiguousarray(row_labels, dtype=np.uint64) if row_labels is not None else None
    if rl is not None:
        assert r is not None and rl.shape[0] == r.shape[0]
    keep = (buf, r, rl)
    return keep, (buf.ctypes.data, buf.size, HS_PATCH_INLINE_ROWS if inline else 0,
                  r.ctypes.data if r is not None else None, rl.ctypes.data if rl is not None else None,
                  r.shape[0] if r is not None else 0)


class BuildParams(C.Structure):
    _fields_ = [("M", C.c_uint64), ("ef_construction", C.c_uint64), ("branching_factor", C.c_char_p),
                ("threshold_level", C.c_int32), ("top_degree_percent0", C.c_float),
                ("top_degree_percent", C.c_float), ("top_M0", C.c_uint64), ("low_m0", C.c_uint64),
                ("top_M", C.c_uint64), ("low_m", C.c_uint64), ("threads", C.c_int32), ("seed", C.c_uint64)]


_lib = None


def lib_path() -> str:
    return _build.LIB


def lib():
    """The loaded shared library (raises if it was not built — no fallback)."""
    global _lib
    if _lib is None:
        path = os.environ.get("HS_LIB_PATH", _build.LIB)     # HS_LIB_PATH: tuning variants (build.py --variant)
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} is missing: run `python -m hnsw_slim_b200.build` (nvcc, sm_100a). "
                "hnsw_slim_b200 has no CPU / PyTorch fallback.")
        L = C.CDLL(path)
        vp, sz, i32 = C.c_void_p, C.c_size_t, C.c_int
        L.hs_last_error.restype = C.c_char_p
        L.hs_abi_version.restype = i32
        L.hs_load.argtypes = [C.c_char_p, i32, i32, sz, vp, sz, i32, C.POINTER(vp)]
        L.hs_load_memory.argtypes = [vp, sz, i32, i32, sz, vp, sz, i32, C.POINTER(vp)]
        L.hs_free.argtypes = [vp]
        L.hs_free.restype = None
        L.hs_set_ef.argtypes = [vp, sz]
        L.hs_get_info.argtypes = [vp, C.POINTER(IndexInfo)]
        L.hs_search_batch.argtypes = [vp, vp, sz, sz, vp, vp]
        L.hs_search_batch_counts.argtypes = [vp, vp, sz, sz, vp, vp, vp]
        L.hs_search_batch_submit.argtypes = [vp, vp, sz, sz, vp, vp]
        L.hs_search_batch_wait.argtypes = [vp]
        L.hs_search_batch_wait_oldest.argtypes = [vp]
        L.hs_pin_host.argtypes = [vp, sz]
        L.hs_unpin_host.argtypes = [vp]
        L.hs_search_batch_device.argtypes = [vp, vp, sz, sz, vp, vp, vp]
        L.hs_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.hs_reset_stats.argtypes = [vp]
        L.hs_bruteforce_knn.argtypes = [vp, sz, sz, vp, sz, sz, i32, i32, vp, vp]
        L.hs_bruteforce_knn_device.argtypes = [vp, sz, sz, vp, sz, sz, i32, vp, vp, vp]
        L.hs_topk_merge_device.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp]
        L.hs_recall.argtypes = [vp, sz, sz, vp, sz, vp, sz, vp, sz, i32, i32, C.POINTER(C.c_double)]
        L.hs_debug_flatten.argtypes = [C.c_char_p, i32, sz, C.POINTER(vp)]
        L.hs_debug_free.argtypes = [vp]
        L.hs_debug_free.restype = None
        L.hs_debug_info.argtypes = [vp, C.POINTER(IndexInfo)]
        L.hs_debug_row.argtypes = [vp, C.c_uint32, i32, vp, i32]
        L.hs_debug_node.argtypes = [vp, C.c_uint32, C.POINTER(i32), C.POINTER(C.c_uint32), vp]
        L.hs_build_params_default.argtypes = [C.POINTER(BuildParams)]
        L.hs_build_params_default.restype = None
        L.hs_build_slim_graph.argtypes = [vp, sz, sz, i32, C.POINTER(BuildParams), vp, C.c_char_p]
        L.hs_build_hnsw_graph.argtypes = [vp, sz, sz, i32, C.POINTER(BuildParams), vp, C.c_char_p]
        L.hs_build_slimq_graph.argtypes = [vp, sz, sz, C.POINTER(BuildParams), vp, sz, vp, vp, C.c_char_p]
        L.hs_slimq_default_tconst.argtypes = [sz]
        L.hs_set_overlap.argtypes = [vp, i32]
        L.hs_search_batch_device_scatter.argtypes = [vp, vp, sz, sz, vp, vp, sz, sz, vp]
        L.hs_exchange_create.argtypes = [i32, i32, i32, sz, sz, sz, C.POINTER(vp)]
        L.hs_exchange_handle.argtypes = [vp, vp]
        L.hs_exchange_connect.argtypes = [vp, vp]
        L.hs_exchange_search.argtypes = [vp, vp, vp, sz, sz, sz, C.c_uint32, vp]
        L.hs_exchange_signal_and_wait.argtypes = [vp, C.c_uint32, vp]
        L.hs_exchange_tables.argtypes = [vp, C.c_uint32, C.POINTER(vp), C.POINTER(vp)]
        L.hs_exchange_free.argtypes = [vp]
        L.hs_exchange_free.restype = None
        L.hs_build_slim_index_gpu.argtypes = [vp, sz, sz, i32, C.POINTER(BuildParams), vp, i32, C.POINTER(vp)]
        L.hs_save_index.argtypes = [vp, C.c_char_p]
        L.hs_build_slimq_index_gpu.argtypes = [vp, sz, sz, C.POINTER(BuildParams), vp, sz, vp, i32, C.POINTER(vp)]
        L.hs_shardgroup_create.argtypes = [vp, sz, i32, i32, sz, sz, i32, C.POINTER(vp)]
        L.hs_shardgroup_handle.argtypes = [vp, vp]
        L.hs_shardgroup_connect.argtypes = [vp, vp]
        L.hs_shardgroup_connect_local.argtypes = [vp, sz]
        L.hs_shardgroup_submit.argtypes = [vp, vp, sz, vp, vp]
        L.hs_shardgroup_wait_oldest.argtypes = [vp]
        L.hs_shardgroup_wait.argtypes = [vp]
        L.hs_shardgroup_streams.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
        L.hs_shardgroup_free.argtypes = [vp]
        L.hs_shardgroup_free.restype = None
        L.hs_load_reserve.argtypes = [C.c_char_p, i32, i32, sz, sz, i32, C.POINTER(vp)]
        L.hs_patch_apply.argtypes = [vp, vp, sz, C.c_uint, vp, vp, sz, C.POINTER(PatchInfo)]
        L.hs_debug_patch.argtypes = [vp, vp, sz, C.c_uint, vp, vp, sz, C.POINTER(PatchInfo)]
        L.hs_service_create.argtypes = [vp, sz, C.c_uint, sz, C.POINTER(vp)]
        L.hs_debug_service_create.argtypes = [SERVICE_BACKEND, vp, sz, sz, C.c_uint, sz, C.POINTER(vp)]
        L.hs_service_query.argtypes = [vp, vp, sz, vp, vp]
        L.hs_service_set_ef.argtypes = [vp, sz]
        L.hs_service_patch.argtypes = [vp, vp, sz, C.c_uint, vp, vp, sz, C.POINTER(PatchInfo)]
        L.hs_service_get_stats.argtypes = [vp, C.POINTER(ServiceStats)]
        L.hs_service_free.argtypes = [vp]
        L.hs_service_free.restype = None
        L.hs_set_tuning.argtypes = [vp, C.c_char_p, C.c_longlong]
        L.hs_get_query_tconst.argtypes = [vp, C.POINTER(C.c_double)]
        L.hs_set_query_tconst.argtypes = [vp, C.c_double]
        L.hs_slimq_prepare.argtypes = [vp, vp, sz, vp, vp, vp, vp]
        L.hs_debug_convert_gpu.argtypes = [C.c_char_p, sz, i32, C.POINTER(BuildParams), i32, C.POINTER(vp)]
        L.hs_debug_slimq_payload.argtypes = [vp, vp, vp, vp]
        for name in EXPORTS:
            if name not in ("hs_last_error", "hs_free", "hs_debug_free", "hs_build_params_default", "hs_exchange_free",
                            "hs_shardgroup_free", "hs_service_free",
                            "hs_slimq_default_tconst", "hs_debug_bf_tc_fallback"):
                getattr(L, name).restype = i32
        L.hs_slimq_default_tconst.restype = C.c_double
        L.hs_debug_bf_tc_fallback.restype = C.c_longlong
        L.hs_debug_bf_tc_fallback.argtypes = []
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise HsError(rc, lib().hs_last_error().decode(errors="replace"))


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


class Index:
    """An HBM-resident HNSW-Slim index (hs_index*)."""

    def __init__(self, graph_path: str, dim: int, *, kind: int = HS_KIND_SLIM, metric: int = HS_METRIC_L2,
                 raw_base: np.ndarray | None = None, device: int = 0):
        self._h = C.c_void_p()
        raw = _f32(raw_base) if raw_base is not None else None
        _check(lib().hs_load(graph_path.encode(), kind, metric, dim,
                             raw.ctypes.data if raw is not None else None,
                             raw.shape[0] if raw is not None else 0, device, C.byref(self._h)))
        self.dim = dim

    @classmethod
    def load_reserve(cls, graph_path: str, dim: int, max_elements: int, *, metric: int = HS_METRIC_L2,
                     device: int = 0) -> "Index":
        """hs_load_reserve: loadIndex(path, space, max_elements) with room for delta patches (slim.h:753-761)."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        _check(lib().hs_load_reserve(graph_path.encode(), HS_KIND_SLIM, metric, dim, max_elements, device,
                                     C.byref(self._h)))
        self.dim = dim
        return self

    def patch(self, stream: bytes, *, rows=None, row_labels=None, inline: bool = False) -> dict:
        """hs_patch_apply: patchFromStream (slim.h:2206-2388) on the HBM-resident index.  rows[label] (or, with
        row_labels, the row whose label matches) supply the vectors of new nodes unless they are inline."""
        keep, args = _patch_args(stream, rows, row_labels, inline)
        info = PatchInfo()
        _check(lib().hs_patch_apply(self._h, *args, C.byref(info)))
        del keep
        return info.as_dict()

    @classmethod
    def from_bytes(cls, image: bytes, dim: int, *, kind: int = HS_KIND_SLIM, metric: int = HS_METRIC_L2,
                   device: int = 0) -> "Index":
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        buf = np.frombuffer(image, dtype=np.uint8)
        _check(lib().hs_load_memory(buf.ctypes.data, buf.size, kind, metric, dim, None, 0, device,
                                    C.byref(self._h)))
        self.dim = dim
        return self

    @classmethod
    def build_gpu(cls, base, *, metric: int = HS_METRIC_L2, M: int = 16, ef_construction: int = 200,
                  branching: str = "4", labels=None, seed: int = 100, device: int = 0, base_ptr: int | None = None,
                  n: int | None = None, dim: int | None = None, kind: int = HS_KIND_SLIM, centroids=None,
                  num_cluster: int = 16, **prune) -> "Index":
        """hs_build_slim_index_gpu / hs_build_slimq_index_gpu (kind = HS_KIND_SLIMQ): HNSW build + HNSW-Slim
        conversion (+ RaBitQ codes) on the device.  `base` is a host array, or pass base_ptr / n / dim for rows
        that already live in device memory."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        if base_ptr is None:
            b = _f32(base)
            base_ptr, n, dim = b.ctypes.data, b.shape[0], b.shape[1]
        p = BuildParams()
        lib().hs_build_params_default(C.byref(p))
        p.M, p.ef_construction, p.branching_factor = M, ef_construction, branching.encode()
        p.seed = seed
        for k_, v in prune.items():
            setattr(p, k_, v)
        lab = None
        if labels is not None:
            labels = np.ascontiguousarray(labels, dtype=np.uint64)
            lab = labels.ctypes.data
        if kind == HS_KIND_SLIMQ:
            cen = None
            if centroids is not None:
                centroids = _f32(centroids)
                num_cluster, cen = centroids.shape[0], centroids.ctypes.data
            _check(lib().hs_build_slimq_index_gpu(base_ptr, n, dim, C.byref(p), cen, num_cluster, lab, device,
                                                  C.byref(self._h)))
        else:
            _check(lib().hs_build_slim_index_gpu(base_ptr, n, dim, metric, C.byref(p), lab, device, C.byref(self._h)))
        self.dim = dim
        return self

    @classmethod
    def convert_gpu(cls, hnsw_path: str, dim: int, *, metric: int = HS_METRIC_L2, device: int = 0,
                    **prune) -> "Index":
        """hs_debug_convert_gpu: the device builder's convertFromHNSW (phase 2) over the lists of an
        hs_build_hnsw_graph file; `prune` sets threshold_level, top_degree_percent, top_M0, low_m0, top_M, low_m."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        p = BuildParams()
        lib().hs_build_params_default(C.byref(p))
        for k_, v in prune.items():
            setattr(p, k_, v)
        _check(lib().hs_debug_convert_gpu(hnsw_path.encode(), dim, metric, C.byref(p), device, C.byref(self._h)))
        self.dim = dim
        return self

    def save(self, path: str) -> None:
        """hs_save_index: the reference's saveIndex format, hnsw_slim (slim.h:717-751) or hnsw_slimq
        (slimq.h:1161-1216).  An hnsw_slimq file is written with zero ex-code blocks and holds no raw rows: open it
        again with the same rows, in the same order, as raw_base (for a GPU-built index, the builder's input)."""
        _check(lib().hs_save_index(self._h, path.encode()))

    def slimq_payload(self) -> dict:
        """hs_debug_slimq_payload (hnsw_slimq): per node codes[n, words] (MSB-first u64 words), f_add[n],
        f_rescale[n], cluster[n]; the rotated centroids[num_cluster, padded_dim] and the rotator flip bytes."""
        info = self.info()
        n, pd, nc = info["n"], info["padded_dim_q"], info["num_cluster"]
        words = pd // 64
        rec = np.zeros((n, words + 2), np.uint64)
        cent = np.zeros((nc, pd), np.float32)
        flip = np.zeros(4 * pd // 8, np.uint8)
        _check(lib().hs_debug_slimq_payload(self._h, rec.ctypes.data, cent.ctypes.data, flip.ctypes.data))
        fac = rec[:, words].copy().view(np.float32).reshape(n, 2)
        return {"codes": rec[:, :words].copy(), "f_add": fac[:, 0].copy(), "f_rescale": fac[:, 1].copy(),
                "cluster": (rec[:, words + 1] & np.uint64(0xFFFFFFFF)).astype(np.uint32),
                "centroids": cent, "flip": flip}

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hs_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def info(self) -> dict:
        s = IndexInfo()
        _check(lib().hs_get_info(self._h, C.byref(s)))
        return s.as_dict()

    def set_ef(self, ef: int) -> None:
        _check(lib().hs_set_ef(self._h, ef))

    def set_tuning(self, name: str, value: int) -> None:
        """hs_set_tuning: "visited_table", "hash_bits", "traverse_flags", "slimq_flags", "zero_copy" (see the header)."""
        _check(lib().hs_set_tuning(self._h, name.encode(), int(value)))

    def set_overlap(self, on: bool) -> None:
        """hs_set_overlap: consecutive device-buffer batches on one stream may overlap (see the header)."""
        _check(lib().hs_set_overlap(self._h, int(bool(on))))

    def search(self, queries, k: int, *, want_dists: bool = True, counts: bool = False):
        """Host buffers in/out (hs_search_batch).  -> labels[nq,k], dists[nq,k] (, counts[nq,2])."""
        q = _f32(queries)
        assert q.ndim == 2 and q.shape[1] == self.dim
        nq = q.shape[0]
        lab = np.empty((nq, k), dtype=np.uint32)
        dist = np.empty((nq, k), dtype=np.float32) if want_dists else None
        if counts:
            cnt = np.zeros((nq, 2), dtype=np.uint32)
            _check(lib().hs_search_batch_counts(self._h, q.ctypes.data, nq, k, lab.ctypes.data,
                                                dist.ctypes.data if want_dists else None, cnt.ctypes.data))
            return lab, dist, cnt
        _check(lib().hs_search_batch(self._h, q.ctypes.data, nq, k, lab.ctypes.data,
                                     dist.ctypes.data if want_dists else None))
        return lab, dist

    def search_ptr(self, q_ptr: int, nq: int, k: int, lab_ptr: int, dist_ptr: int | None) -> None:
        """hs_search_batch on raw HOST pointers (e.g. pinned torch tensors)."""
        _check(lib().hs_search_batch(self._h, q_ptr, nq, k, lab_ptr, dist_ptr))

    def submit_ptr(self, q_ptr: int, nq: int, k: int, lab_ptr: int, dist_ptr: int | None) -> None:
        """hs_search_batch_submit: enqueue a host-buffer batch, return at once (see wait())."""
        _check(lib().hs_search_batch_submit(self._h, q_ptr, nq, k, lab_ptr, dist_ptr))

    def wait(self) -> None:
        """hs_search_batch_wait: block until every submitted batch is complete."""
        _check(lib().hs_search_batch_wait(self._h))

    def wait_oldest(self) -> None:
        """hs_search_batch_wait_oldest: block until the oldest outstanding submitted batch is complete."""
        _check(lib().hs_search_batch_wait_oldest(self._h))

    def search_device(self, d_queries: int, nq: int, k: int, d_labels: int, d_dists: int | None,
                      stream: int = 0) -> None:
        """Device pointers, asynchronous on `stream` (hs_search_batch_device)."""
        _check(lib().hs_search_batch_device(self._h, d_queries, nq, k, d_labels, d_dists, stream))

    # ---- hnsw_slimq only ----
    @property
    def query_tconst(self) -> float:
        t = C.c_double(0)
        _check(lib().hs_get_query_tconst(self._h, C.byref(t)))
        return t.value

    @query_tconst.setter
    def query_tconst(self, t: float) -> None:
        _check(lib().hs_set_query_tconst(self._h, float(t)))

    def slimq_prepare(self, queries):
        """hs_slimq_prepare -> rotated[nq,pd], planes[nq,pd/64*4] u64, scal[nq,3], q2c[nq,ncl]."""
        q = _f32(queries)
        assert q.ndim == 2 and q.shape[1] == self.dim
        info = self.info()
        nq, pd, nc = q.shape[0], info["padded_dim_q"], info["num_cluster"]
        rot = np.zeros((nq, pd), np.float32)
        planes = np.zeros((nq, pd // 64 * 4), np.uint64)
        scal = np.zeros((nq, 3), np.float32)
        q2c = np.zeros((nq, nc), np.float32)
        _check(lib().hs_slimq_prepare(self._h, q.ctypes.data, nq, rot.ctypes.data, planes.ctypes.data,
                                      scal.ctypes.data, q2c.ctypes.data))
        return rot, planes, scal, q2c

    def stats(self) -> dict:
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(lib().hs_stats(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"n_dist": a.value, "n_hops": b.value, "n_rerank": c.value}

    def reset_stats(self) -> None:
        _check(lib().hs_reset_stats(self._h))


class Exchange:
    """hs_exchange: the gather tables + flags of one rank for the fused sharded exchange."""

    def __init__(self, device: int, world: int, rank: int, slots: int, nq_max: int, k: int):
        self._h = C.c_void_p()
        _check(lib().hs_exchange_create(device, world, rank, slots, nq_max, k, C.byref(self._h)))
        self.world, self.rank, self.slots, self.k = world, rank, slots, k

    def handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        _check(lib().hs_exchange_handle(self._h, buf))
        return buf.raw

    def connect(self, handles: bytes) -> None:
        assert len(handles) == 64 * self.world
        _check(lib().hs_exchange_connect(self._h, handles))

    def search(self, index: "Index", d_queries: int, nq: int, slot: int, seq: int, stream: int = 0) -> None:
        _check(lib().hs_exchange_search(self._h, index.handle, d_queries, nq, self.k, slot, seq, stream))

    def signal_and_wait(self, seq: int, stream: int = 0) -> None:
        _check(lib().hs_exchange_signal_and_wait(self._h, seq, stream))

    def tables(self, seq: int):
        l, d = C.c_void_p(), C.c_void_p()
        _check(lib().hs_exchange_tables(self._h, seq, C.byref(l), C.byref(d)))
        return l.value, d.value

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hs_exchange_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ShardGroup:
    """hs_shardgroup: one rank's local shards + gather tables + streams of the pipelined sharded search."""

    def __init__(self, shards, world: int, rank: int, nq_max: int, k: int, depth: int = 4):
        self._h = C.c_void_p()
        self._shards = list(shards)                       # keep the indices alive: the group borrows them
        arr = (C.c_void_p * len(self._shards))(*[s.handle for s in self._shards])
        _check(lib().hs_shardgroup_create(arr, len(self._shards), world, rank, nq_max, k, depth, C.byref(self._h)))
        self.world, self.rank, self.k, self.nq_max, self.depth = world, rank, k, nq_max, depth

    def handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        _check(lib().hs_shardgroup_handle(self._h, buf))
        return buf.raw

    def connect(self, handles: bytes | None) -> None:
        assert self.world == 1 or len(handles) == 64 * self.world
        _check(lib().hs_shardgroup_connect(self._h, handles))

    @staticmethod
    def connect_local(groups) -> None:
        """One process driving all GPUs: groups[r] = rank r."""
        arr = (C.c_void_p * len(groups))(*[g._h for g in groups])
        _check(lib().hs_shardgroup_connect_local(arr, len(groups)))

    def submit(self, q_ptr: int, nq: int, lab_ptr: int, dist_ptr: int | None) -> None:
        _check(lib().hs_shardgroup_submit(self._h, q_ptr, nq, lab_ptr, dist_ptr))

    def wait_oldest(self) -> None:
        _check(lib().hs_shardgroup_wait_oldest(self._h))

    def wait(self) -> None:
        _check(lib().hs_shardgroup_wait(self._h))

    def streams(self):
        a, b = C.c_void_p(), C.c_void_p()
        _check(lib().hs_shardgroup_streams(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hs_shardgroup_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def search_device_scatter(index: "Index", d_queries: int, nq: int, k: int, label_dsts, dist_dsts, slot: int,
                          stream: int = 0) -> None:
    """hs_search_batch_device_scatter: rows go to slot `slot` of every destination table."""
    n = len(label_dsts)
    la = (C.c_void_p * n)(*label_dsts)
    da = (C.c_void_p * n)(*dist_dsts)
    _check(lib().hs_search_batch_device_scatter(index.handle, d_queries, nq, k, la, da, n, slot, stream))


def build_slim_graph(base, path: str, *, metric: int = HS_METRIC_L2, M: int = 16, ef_construction: int = 200,
                     branching: str = "4", threads: int = 0, labels=None, seed: int = 100, **prune) -> None:
    """hs_build_slim_graph: host-side HNSW build + HNSW-Slim pruning -> reference-format .graph."""
    b = _f32(base)
    p = BuildParams()
    lib().hs_build_params_default(C.byref(p))
    p.M, p.ef_construction, p.branching_factor = M, ef_construction, branching.encode()
    p.threads, p.seed = threads, seed
    for k_, v in prune.items():
        setattr(p, k_, v)
    lab = None
    if labels is not None:
        labels = np.ascontiguousarray(labels, dtype=np.uint64)
        lab = labels.ctypes.data
    _check(lib().hs_build_slim_graph(b.ctypes.data, b.shape[0], b.shape[1], metric, C.byref(p), lab, path.encode()))


def build_hnsw_graph(base, path: str, *, metric: int = HS_METRIC_L2, M: int = 16, ef_construction: int = 200,
                     branching: str = "4", threads: int = 0, labels=None, seed: int = 100) -> None:
    """hs_build_hnsw_graph: host-side HNSW build -> upstream-format .graph of the `hnsw` strategy."""
    b = _f32(base)
    p = BuildParams()
    lib().hs_build_params_default(C.byref(p))
    p.M, p.ef_construction, p.branching_factor = M, ef_construction, branching.encode()
    p.threads, p.seed = threads, seed
    lab = None
    if labels is not None:
        labels = np.ascontiguousarray(labels, dtype=np.uint64)
        lab = labels.ctypes.data
    _check(lib().hs_build_hnsw_graph(b.ctypes.data, b.shape[0], b.shape[1], metric, C.byref(p), lab, path.encode()))


def build_slimq_graph(base, path: str, *, M: int = 16, ef_construction: int = 200, branching: str = "4",
                      threads: int = 0, labels=None, seed: int = 100, centroids=None, cluster_ids=None,
                      num_cluster: int = 16, **prune) -> None:
    """hs_build_slimq_graph: HNSW + HNSW-Slim pruning + RaBitQ codes -> reference-format hnsw_slimq .graph."""
    b = _f32(base)
    p = BuildParams()
    lib().hs_build_params_default(C.byref(p))
    p.M, p.ef_construction, p.branching_factor = M, ef_construction, branching.encode()
    p.threads, p.seed = threads, seed
    for k_, v in prune.items():
        setattr(p, k_, v)
    lab = cen = cid = None
    if labels is not None:
        labels = np.ascontiguousarray(labels, dtype=np.uint64)
        lab = labels.ctypes.data
    if centroids is not None:
        centroids = _f32(centroids)
        cluster_ids = np.ascontiguousarray(cluster_ids, dtype=np.uint32)
        num_cluster = centroids.shape[0]
        cen, cid = centroids.ctypes.data, cluster_ids.ctypes.data
    _check(lib().hs_build_slimq_graph(b.ctypes.data, b.shape[0], b.shape[1], C.byref(p), cen, num_cluster, cid,
                                      lab, path.encode()))


def slimq_default_tconst(padded_dim: int) -> float:
    return float(lib().hs_slimq_default_tconst(padded_dim))


class Service:
    """hs_service: single-query serving in front of the batched search (the /query, /setEf and update handlers of
    hnsw_slim_server.cc:69-142).  `backend` is an Index, or — CPU tests — a python function
    f(queries[nq, dim], k) -> (labels[nq, k], dists[nq, k]) standing in for hs_search_batch."""

    def __init__(self, backend, *, max_batch: int = 4096, max_wait_us: int = 0, k_max: int = 100, dim: int | None = None):
        self._h = C.c_void_p()
        self._cb = None
        if isinstance(backend, Index):
            self.dim = backend.dim
            self._index = backend                      # keep it alive: the service borrows the handle
            _check(lib().hs_service_create(backend.handle, max_batch, max_wait_us, k_max, C.byref(self._h)))
        else:
            assert dim is not None
            self.dim = dim

            def trampoline(_ctx, qp, nq, k, lp, dp):
                try:
                    q = np.ctypeslib.as_array(C.cast(qp, C.POINTER(C.c_float)), shape=(nq, dim))
                    lab, dist = backend(q.copy(), k)
                    np.ctypeslib.as_array(C.cast(lp, C.POINTER(C.c_uint32)), shape=(nq, k))[:] = lab
                    np.ctypeslib.as_array(C.cast(dp, C.POINTER(C.c_float)), shape=(nq, k))[:] = dist
                    return 0
                except Exception:                      # noqa: BLE001 — reported through the C status code
                    return -2

            self._cb = SERVICE_BACKEND(trampoline)
            _check(lib().hs_debug_service_create(self._cb, None, dim, max_batch, max_wait_us, k_max, C.byref(self._h)))

    def query(self, vec, k: int, want_dists: bool = False):
        v = _f32(vec)
        assert v.shape == (self.dim,)
        lab = np.empty(k, dtype=np.uint32)
        dist = np.empty(k, dtype=np.float32) if want_dists else None
        _check(lib().hs_service_query(self._h, v.ctypes.data, k, lab.ctypes.data, dist.ctypes.data if want_dists else None))
        return (lab, dist) if want_dists else lab

    def set_ef(self, ef: int) -> None:
        _check(lib().hs_service_set_ef(self._h, ef))

    def patch(self, stream: bytes, *, rows=None, row_labels=None, inline: bool = False) -> dict:
        keep, args = _patch_args(stream, rows, row_labels, inline)
        info = PatchInfo()
        _check(lib().hs_service_patch(self._h, *args, C.byref(info)))
        del keep
        return info.as_dict()

    def stats(self) -> dict:
        s = ServiceStats()
        _check(lib().hs_service_get_stats(self._h, C.byref(s)))
        return {f: getattr(s, f) for f, _ in s._fields_}

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hs_service_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostGraph:
    """Host-side flattened .graph (hs_debug_flatten) — loader inspection, no GPU needed."""

    def __init__(self, graph_path: str, dim: int, kind: int = HS_KIND_SLIM):
        self._h = C.c_void_p()
        _check(lib().hs_debug_flatten(graph_path.encode(), kind, dim, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().hs_debug_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> dict:
        s = IndexInfo()
        _check(lib().hs_debug_info(self._h, C.byref(s)))
        return s.as_dict()

    def patch(self, stream: bytes, *, rows=None, row_labels=None, inline: bool = False) -> dict:
        """hs_debug_patch: hs_patch_apply on the host image (same parser, validation and re-slotting)."""
        keep, args = _patch_args(stream, rows, row_labels, inline)
        info = PatchInfo()
        _check(lib().hs_debug_patch(self._h, *args, C.byref(info)))
        del keep
        return info.as_dict()

    def row(self, node: int, level: int) -> np.ndarray:
        """Valid ids of the node's level-`level` row (padding stripped; checks it is a suffix)."""
        out = np.full(1024, 0xFFFFFFFF, dtype=np.uint32)
        stride = lib().hs_debug_row(self._h, node, level, out.ctypes.data, 1024)
        if stride < 0:
            _check(stride)
        r = out[:stride]
        valid = r != 0xFFFFFFFF
        cnt = int(valid.sum())
        assert valid[:cnt].all(), "padding must follow the valid ids"
        return r[:cnt].copy()

    def node(self, i: int):
        lvl, lab = C.c_int(0), C.c_uint32(0)
        info = self.info()
        vec = np.zeros(info["dim_padded"], dtype=np.float32)
        _check(lib().hs_debug_node(self._h, i, C.byref(lvl), C.byref(lab), vec.ctypes.data))
        return lvl.value, lab.value, vec


def bruteforce_knn(base, queries, k: int, *, metric: int = HS_METRIC_L2, device: int = 0):
    """Exact kNN, nearest first (hs_bruteforce_knn).  -> labels[nq,k], dists[nq,k]."""
    b, q = _f32(base), _f32(queries)
    lab = np.empty((q.shape[0], k), dtype=np.uint32)
    dist = np.empty((q.shape[0], k), dtype=np.float32)
    _check(lib().hs_bruteforce_knn(b.ctypes.data, b.shape[0], b.shape[1], q.ctypes.data, q.shape[0], k, metric,
                                   device, lab.ctypes.data, dist.ctypes.data))
    return lab, dist


def bf_tc_fallback() -> int:
    """hs_debug_bf_tc_fallback(): see include/hnswslim_b200.h (needs HS_BF_TC_STATS=1)."""
    return int(lib().hs_debug_bf_tc_fallback())


def bruteforce_knn_device(d_base: int, n: int, dim: int, d_queries: int, nq: int, k: int, d_labels: int,
                          d_dists: int | None, *, metric: int = HS_METRIC_L2, stream: int = 0) -> None:
    _check(lib().hs_bruteforce_knn_device(d_base, n, dim, d_queries, nq, k, metric, d_labels, d_dists, stream))


def topk_merge_device(d_labels_in: int, d_dists_in: int, n_parts: int, nq: int, k: int, d_labels_out: int,
                      d_dists_out: int | None, stream: int = 0) -> None:
    _check(lib().hs_topk_merge_device(d_labels_in, d_dists_in, n_parts, nq, k, d_labels_out, d_dists_out, stream))


def recall(base, queries, knn, gt, K: int | None = None, *, metric: int = HS_METRIC_L2, device: int = 0) -> float:
    """SolveStrategy::recall on the device (hs_recall)."""
    b, q = _f32(base), _f32(queries)
    knn = np.ascontiguousarray(knn, dtype=np.uint32)
    gt = np.ascontiguousarray(gt, dtype=np.uint32)
    K = K or knn.shape[1]
    out = C.c_double(0)
    _check(lib().hs_recall(b.ctypes.data, b.shape[0], b.shape[1], q.ctypes.data, q.shape[0], knn.ctypes.data, K,
                           gt.ctypes.data, gt.shape[1], metric, device, C.byref(out)))
    return out.value
