"""ctypes binding of libdawn_b200.so with the method names of `usearch::ffi::Index`.

The reference drives its index through the `usearch::ffi` cxx bridge
(/root/reference/src/search/search_provider.rs:32-42,102,115-117,133,149,178,214,246,280-284):

    new_index(&IndexOptions) -> Index
    index.reserve(n) / add(label, &[f32]) / search(&[f32], k) -> Matches{labels, distances}
    index.size() / capacity() / dimensions() / save(path) / load(path) / view(path)

This module exposes the same names over the C ABI in include/dawn_index.h so that the
parity tests read like calls into the reference.  Errors surface as `DawnError`
(the cxx bridge maps C++ exceptions to `Result::Err`).

There is no CPU fallback: importing works anywhere, but creating an index without the
built library or without a B200 raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

EM_LEN = 384  # src/search/vector.rs:26
MAX_K = 120

_HERE = os.path.dirname(os.path.abspath(__file__))
# DAWN_B200_LIB: load another build of the same library (A/B of kernel changes on one box); never a fallback
LIB_PATH = os.environ.get("DAWN_B200_LIB") or os.path.join(_HERE, "lib", "libdawn_b200.so")

_vp = C.c_void_p


class DawnError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libdawn_b200 error {code}: {message}")
        self.code = code


class MetricKind:  # usearch::ffi::MetricKind (search_provider.rs:37)
    IP = 0


class ScalarKind:  # usearch::ffi::ScalarKind (search_provider.rs:38); storage precision
    F16 = 0
    I8 = 1
    F32 = 2  # the reference's own setting: f32 vectors kept as given, exact f32 distances


class _Options(C.Structure):
    _fields_ = [
        ("dimensions", C.c_uint32),
        ("metric", C.c_uint32),
        ("scalar", C.c_uint32),
        ("device", C.c_int32),
        ("capacity", C.c_uint64),
        ("flags", C.c_uint32),
        ("reserved_", C.c_uint32),
    ]


class Profile(C.Structure):
    _fields_ = [
        ("scan_launches", C.c_uint64),
        ("scan_ms", C.c_double),
        ("finalize_launches", C.c_uint64),
        ("finalize_ms", C.c_double),
        ("queries", C.c_uint64),
        ("uncertified", C.c_uint64),
        ("escalations", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("gemm_batches", C.c_uint64),
        ("gemm_ms", C.c_double),
        ("device_uncertified", C.c_uint64),
        ("device_status", C.c_uint64),
        ("max_selection_error", C.c_double),
        ("shadow_batches", C.c_uint64),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class ScoreError(C.Structure):
    _fields_ = [
        ("max_mma_vs_f64", C.c_double),
        ("max_seq_vs_f64", C.c_double),
        ("max_mma_vs_seq", C.c_double),
        ("max_err_over_eps_q", C.c_double),
        ("pairs", C.c_uint64),
        ("hist", C.c_uint64 * 40),
        ("scan_eps", C.c_float),
        ("gemm_accum_slack", C.c_float),
        ("i8_dequant_slack", C.c_float),
        ("reserved_", C.c_float),
    ]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n not in ("hist", "reserved_")}
        d["hist"] = list(self.hist)
        return d


class MultiStats(C.Structure):
    _fields_ = [
        ("searches", C.c_uint64),
        ("nccl_exchanges", C.c_uint64),
        ("peer_exchanges", C.c_uint64),
        ("exact_reruns", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("last_search_ms", C.c_double),
        ("last_exchange_ms", C.c_double),
        ("nccl_ready", C.c_uint32),
        ("reserved_", C.c_uint32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved_"}


@dataclass
class IndexOptions:
    """usearch::ffi::IndexOptions as the reference fills it (search_provider.rs:35-42).
    connectivity / expansion_* are accepted and ignored: the search is exact."""

    dimensions: int = EM_LEN
    metric: int = MetricKind.IP
    quantization: int = ScalarKind.F16
    connectivity: int = 0
    expansion_add: int = 0
    expansion_search: int = 0
    device: int = 0
    capacity: int = 0


@dataclass
class Matches:
    """usearch::ffi::Matches (search_provider.rs:221): labels and distances, ascending."""

    labels: np.ndarray
    distances: np.ndarray


_lib = None


def load_library() -> C.CDLL:
    """Load libdawn_b200.so; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DawnError(-5, f"{LIB_PATH} is missing: run `make -C dawnsearch_b200/csrc` "
                            "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.dawn_last_error.restype = C.c_char_p
    L.dawn_version.restype = C.c_char_p
    L.dawn_index_create.argtypes = [C.POINTER(_Options), C.POINTER(_vp)]
    L.dawn_index_free.argtypes = [_vp]
    L.dawn_index_free.restype = None
    L.dawn_index_reserve.argtypes = [_vp, C.c_size_t]
    L.dawn_index_add.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_index_add_batch.argtypes = [_vp, _vp, _vp, C.c_size_t]
    L.dawn_index_remove.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_index_remove_batch.argtypes = [_vp, _vp, C.c_size_t, _vp]
    L.dawn_index_search.argtypes = [_vp, _vp, C.c_size_t, _vp, _vp, _vp]
    L.dawn_index_search_batch.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, _vp, _vp, _vp]
    L.dawn_index_search_device.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, _vp, _vp, _vp, _vp, _vp]
    L.dawn_index_search_device_limit.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, C.c_float, _vp, _vp, _vp, _vp, _vp]
    L.dawn_merge_results_device.argtypes = [C.c_int, _vp, _vp, _vp, C.c_size_t, C.c_size_t, C.c_size_t,
                                            C.c_size_t, _vp, _vp, _vp, _vp]
    for name in ("dawn_index_size", "dawn_index_capacity", "dawn_index_dimensions"):
        getattr(L, name).argtypes = [_vp]
        getattr(L, name).restype = C.c_size_t
    L.dawn_index_save.argtypes = [_vp, C.c_char_p]
    L.dawn_index_load.argtypes = [_vp, C.c_char_p]
    L.dawn_index_get.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_index_add_synthetic.argtypes = [_vp, C.c_uint64, C.c_uint64, C.c_size_t]
    L.dawn_index_set_profiling.argtypes = [_vp, C.c_int]
    L.dawn_index_set_option.argtypes = [_vp, C.c_char_p, C.c_int64]
    L.dawn_index_get_profile.argtypes = [_vp, C.POINTER(Profile), C.c_int]
    L.dawn_debug_gemm_score_error.argtypes = [_vp, _vp, C.c_size_t, C.POINTER(ScoreError)]
    L.dawn_vector_length.argtypes = [_vp]
    L.dawn_vector_length.restype = C.c_float
    L.dawn_is_normalized.argtypes = [_vp]
    L.dawn_normalize.argtypes = [_vp]
    L.dawn_normalize.restype = None
    L.dawn_encode_i24.argtypes = [_vp, _vp]
    L.dawn_encode_i24.restype = None
    L.dawn_decode_i24.argtypes = [_vp, _vp]
    L.dawn_index_search_limit.argtypes = [_vp, _vp, C.c_size_t, C.c_float, _vp, _vp, _vp]
    L.dawn_index_search_batch_limit.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, C.c_float, _vp, _vp, _vp]
    L.dawn_index_verify.argtypes = [_vp, _vp, _vp, _vp]
    L.dawn_index_search_i24.argtypes = [_vp, _vp, C.c_size_t, C.c_int, C.c_float, _vp, _vp, _vp]
    L.dawn_index_get_i24.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_index_add_page_entries.argtypes = [_vp, _vp, C.c_size_t, C.c_uint64, _vp]
    L.dawn_batcher_create.argtypes = [_vp, C.c_size_t, C.c_uint32, C.POINTER(_vp)]
    L.dawn_batcher_create_multi.argtypes = [_vp, C.c_size_t, C.c_uint32, C.POINTER(_vp)]
    L.dawn_batcher_search.argtypes = [_vp, _vp, C.c_size_t, _vp, _vp, _vp]
    L.dawn_batcher_stats.argtypes = [_vp, _vp, _vp, _vp]
    L.dawn_batcher_last_error.restype = C.c_char_p
    L.dawn_batcher_free.argtypes = [_vp]
    L.dawn_batcher_free.restype = None
    L.dawn_multi_create.argtypes = [_vp, C.c_size_t, C.c_uint32, C.POINTER(_vp)]
    L.dawn_multi_free.argtypes = [_vp]
    L.dawn_multi_free.restype = None
    L.dawn_multi_reserve.argtypes = [_vp, C.c_size_t]
    L.dawn_multi_add.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_multi_add_batch.argtypes = [_vp, _vp, _vp, C.c_size_t]
    L.dawn_multi_add_synthetic.argtypes = [_vp, C.c_uint64, C.c_uint64, C.c_size_t]
    L.dawn_multi_remove.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_multi_remove_batch.argtypes = [_vp, _vp, C.c_size_t, _vp]
    L.dawn_multi_search.argtypes = [_vp, _vp, C.c_size_t, _vp, _vp, _vp]
    L.dawn_multi_search_batch.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, _vp, _vp, _vp]
    L.dawn_multi_search_batch_limit.argtypes = [_vp, _vp, C.c_size_t, C.c_size_t, C.c_float, _vp, _vp, _vp]
    L.dawn_multi_search_limit.argtypes = [_vp, _vp, C.c_size_t, C.c_float, _vp, _vp, _vp]
    for name in ("dawn_multi_size", "dawn_multi_capacity", "dawn_multi_shards"):
        getattr(L, name).argtypes = [_vp]
        getattr(L, name).restype = C.c_size_t
    L.dawn_multi_last_error.restype = C.c_char_p
    L.dawn_multi_set_option.argtypes = [_vp, C.c_char_p, C.c_int64]
    L.dawn_multi_get_stats.argtypes = [_vp, C.POINTER(MultiStats)]
    L.dawn_multi_save.argtypes = [_vp, C.c_char_p]
    L.dawn_multi_load.argtypes = [_vp, C.c_char_p]
    L.dawn_multi_get.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_multi_get_i24.argtypes = [_vp, C.c_uint64, _vp]
    L.dawn_multi_verify.argtypes = [_vp, _vp, _vp, _vp]
    L.dawn_multi_search_i24.argtypes = [_vp, _vp, C.c_size_t, C.c_int, C.c_float, _vp, _vp, _vp]
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise DawnError(rc, load_library().dawn_last_error().decode("utf-8", "replace"))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_vp)


class Index:
    """Device-resident exact index; method names follow usearch::ffi::Index."""

    def __init__(self, options: IndexOptions):
        L = load_library()
        if options.quantization not in (ScalarKind.F16, ScalarKind.I8, ScalarKind.F32):
            raise DawnError(-1, "quantization must be ScalarKind.F16, ScalarKind.I8 or ScalarKind.F32")
        o = _Options(options.dimensions, options.metric, options.quantization, options.device,
                     options.capacity, 0, 0)
        h = _vp()
        _check(L.dawn_index_create(C.byref(o), C.byref(h)))
        self._h = h
        self._L = L
        self.device = options.device

    # -- lifetime ------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.dawn_index_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- usearch::ffi::Index surface --------------------------------------------------
    def reserve(self, capacity: int) -> None:  # search_provider.rs:133,282
        _check(self._L.dawn_index_reserve(self._h, capacity))

    def add(self, label: int, vector) -> None:  # search_provider.rs:149,284
        v = np.ascontiguousarray(vector, dtype=np.float32)
        if v.shape != (EM_LEN,):
            raise DawnError(-1, f"vector must have {EM_LEN} dimensions, got {v.shape}")
        _check(self._L.dawn_index_add(self._h, int(label), _ptr(v)))

    def add_batch(self, labels, vectors) -> None:
        lab = np.ascontiguousarray(labels, dtype=np.uint64)
        v = np.ascontiguousarray(vectors, dtype=np.float32).reshape(-1, EM_LEN)
        if lab.shape[0] != v.shape[0]:
            raise DawnError(-1, "labels and vectors differ in length")
        _check(self._L.dawn_index_add_batch(self._h, _ptr(lab), _ptr(v), v.shape[0]))

    def remove(self, label: int) -> int:
        """Remove every stored vector with this label; returns how many were removed (0 if none)."""
        n = C.c_size_t(0)
        _check(self._L.dawn_index_remove(self._h, int(label), C.byref(n)))
        return int(n.value)

    def remove_batch(self, labels) -> int:
        """Remove every stored vector whose label is listed (repeats and absent labels are fine); returns the rows removed.
        An update is remove(label) followed by add(label, vector)."""
        lab = np.ascontiguousarray(labels, dtype=np.uint64).reshape(-1)
        n = C.c_size_t(0)
        _check(self._L.dawn_index_remove_batch(self._h, _ptr(lab), lab.shape[0], C.byref(n)))
        return int(n.value)

    def search(self, query, count: int) -> Matches:  # search_provider.rs:214
        q = np.ascontiguousarray(query, dtype=np.float32)
        if q.shape != (EM_LEN,):
            raise DawnError(-1, f"query must have {EM_LEN} dimensions, got {q.shape}")
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        _check(self._L.dawn_index_search(self._h, _ptr(q), count, _ptr(labels), _ptr(dist), C.byref(n)))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())

    def search_batch(self, queries, count: int):
        """-> (labels[B,count], distances[B,count], counts[B]); rows valid up to counts[b]."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        b = q.shape[0]
        labels = np.zeros((b, max(count, 1)), dtype=np.uint64)
        dist = np.zeros((b, max(count, 1)), dtype=np.float32)
        counts = np.zeros(b, dtype=np.uint64)
        _check(self._L.dawn_index_search_batch(self._h, _ptr(q), b, count, _ptr(labels), _ptr(dist),
                                               _ptr(counts)))
        return labels, dist, counts.astype(np.int64)

    def size(self) -> int:  # search_provider.rs:246,280
        return int(self._L.dawn_index_size(self._h))

    def capacity(self) -> int:  # search_provider.rs:280
        return int(self._L.dawn_index_capacity(self._h))

    def dimensions(self) -> int:
        return int(self._L.dawn_index_dimensions(self._h))

    def save(self, path: str) -> None:  # search_provider.rs:117,178
        _check(self._L.dawn_index_save(self._h, os.fsencode(path)))

    def load(self, path: str) -> None:  # search_provider.rs:115
        _check(self._L.dawn_index_load(self._h, os.fsencode(path)))

    view = load  # examples_old/search_usearch.rs:47 (a device index is always a copy)

    # -- additions ---------------------------------------------------------------------
    def get(self, label: int) -> np.ndarray:  # SearchProvider::embedding_for_page, :183-195
        out = np.zeros(EM_LEN, dtype=np.float32)
        _check(self._L.dawn_index_get(self._h, int(label), _ptr(out)))
        return out

    def search_limit(self, query, count: int, distance_limit: float) -> Matches:
        """Hits with distance >= distance_limit are dropped (src/net/udp_service.rs:196-199)."""
        q = np.ascontiguousarray(query, dtype=np.float32)
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        _check(self._L.dawn_index_search_limit(self._h, _ptr(q), count, distance_limit, _ptr(labels), _ptr(dist),
                                               C.byref(n)))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())

    def search_batch_limit(self, queries, count: int, distance_limit: float):
        """Batch form of search_limit (one limit for every query)."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        b = q.shape[0]
        labels = np.zeros((b, max(count, 1)), dtype=np.uint64)
        dist = np.zeros((b, max(count, 1)), dtype=np.float32)
        counts = np.zeros(b, dtype=np.uint64)
        _check(self._L.dawn_index_search_batch_limit(self._h, _ptr(q), b, count, distance_limit, _ptr(labels),
                                                     _ptr(dist), _ptr(counts)))
        return labels, dist, counts.astype(np.int64)

    def verify(self) -> dict:
        """SearchProvider::verify over the device corpus (search_provider.rs:289-327): norm gate on every stored row."""
        bad = C.c_size_t(0)
        lo, hi = C.c_float(0), C.c_float(0)
        _check(self._L.dawn_index_verify(self._h, C.byref(bad), C.byref(lo), C.byref(hi)))
        return {"bad_rows": int(bad.value), "min_norm": float(lo.value), "max_norm": float(hi.value)}

    def search_i24(self, query1152: bytes, count: int, distance_limit=None) -> Matches:
        """The peer side of UdpPacket::Search: raw i24 query bytes, optional distance_limit."""
        buf = np.frombuffer(query1152, dtype=np.uint8).copy()
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        _check(self._L.dawn_index_search_i24(self._h, _ptr(buf), count, int(distance_limit is not None),
                                             float(distance_limit or 0.0), _ptr(labels), _ptr(dist), C.byref(n)))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())

    def get_i24(self, label: int) -> bytes:
        out = np.zeros(EM_LEN * 3, dtype=np.uint8)
        _check(self._L.dawn_index_get_i24(self._h, int(label), _ptr(out)))
        return out.tobytes()

    def add_page_entries(self, entries: bytes, first_label: int) -> int:
        """Bulk load of a legacy `.emb` file (1568-byte PageEntry records); returns #skipped."""
        buf = np.frombuffer(entries, dtype=np.uint8)
        if buf.shape[0] % 1568:
            raise DawnError(-1, "a .emb file is a whole number of 1568-byte PageEntry records")
        skipped = C.c_size_t(0)
        _check(self._L.dawn_index_add_page_entries(self._h, _ptr(buf), buf.shape[0] // 1568, first_label,
                                                   C.byref(skipped)))
        return int(skipped.value)

    def add_synthetic(self, seed: int, first_row: int, n: int) -> None:
        _check(self._L.dawn_index_add_synthetic(self._h, seed, first_row, n))

    def search_device(self, d_queries: int, batch: int, count: int, d_labels: int, d_dist: int,
                      d_counts: int, d_flags: int, stream: int = 0, distance_limit=None) -> None:
        """Raw device-pointer entry point (ints are CUDA device addresses); only enqueues.
        distance_limit: hits with distance >= limit are cut from the counts on the device (udp_service.rs:196-199)."""
        if distance_limit is None:
            _check(self._L.dawn_index_search_device(self._h, d_queries, batch, count, d_labels, d_dist,
                                                    d_counts, d_flags, stream))
        else:
            _check(self._L.dawn_index_search_device_limit(self._h, d_queries, batch, count, float(distance_limit), d_labels,
                                                          d_dist, d_counts, d_flags, stream))

    def debug_gemm_score_error(self, queries, acc: "ScoreError") -> None:
        """Accumulate tensor-core score errors over every (query,row) pair (index of <= 2048 rows); see dawn_index.h."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        _check(self._L.dawn_debug_gemm_score_error(self._h, _ptr(q), q.shape[0], C.byref(acc)))

    def set_option(self, key: str, value: int) -> None:
        """'gemm_min_batch', 'gemm_min_rows', 'force_path' (0 auto, 1 scan, 2 tensor-core)."""
        _check(self._L.dawn_index_set_option(self._h, key.encode(), int(value)))

    def set_profiling(self, enable: bool) -> None:
        _check(self._L.dawn_index_set_profiling(self._h, int(enable)))

    def profile(self, reset: bool = False) -> dict:
        p = Profile()
        _check(self._L.dawn_index_get_profile(self._h, C.byref(p), int(reset)))
        return p.as_dict()


# ---- host mirrors of src/search/vector.rs (no GPU needed) ---------------------------------------


def is_normalized(v) -> bool:  # vector.rs:185-192
    a = np.ascontiguousarray(v, dtype=np.float32)
    return bool(load_library().dawn_is_normalized(_ptr(a)))


def normalize(v) -> np.ndarray:  # vector.rs:194-197
    a = np.ascontiguousarray(v, dtype=np.float32).copy()
    load_library().dawn_normalize(_ptr(a))
    return a


def encode_i24(v) -> bytes:  # vector.rs:74-86 (to24)
    a = np.ascontiguousarray(v, dtype=np.float32)
    out = np.zeros(EM_LEN * 3, dtype=np.uint8)
    load_library().dawn_encode_i24(_ptr(a), _ptr(out))
    return out.tobytes()


def decode_i24(data: bytes) -> np.ndarray:  # vector.rs:52-72 (from24); raises if not normalised
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    if buf.shape[0] != EM_LEN * 3:
        raise DawnError(-1, "an i24 embedding is 1152 bytes")
    out = np.zeros(EM_LEN, dtype=np.float32)
    if load_library().dawn_decode_i24(_ptr(buf), _ptr(out)) != 0:
        raise DawnError(-1, "Embedding is not normalized")
    return out


class Batcher:
    """Micro-batching front (SURVEY 8f-1): `search` may be called from many threads at once.
    `index` is an Index or a MultiIndex (one process, several GPUs)."""

    def __init__(self, index, max_batch: int = 256, max_wait_us: int = 200):
        self._L = load_library()
        h = _vp()
        if isinstance(index, MultiIndex):
            _check(self._L.dawn_batcher_create_multi(index._h, max_batch, max_wait_us, C.byref(h)))
        else:
            _check(self._L.dawn_batcher_create(index._h, max_batch, max_wait_us, C.byref(h)))
        self._h = h
        self._index = index  # keep the index alive

    def search(self, query, count: int) -> Matches:
        q = np.ascontiguousarray(query, dtype=np.float32)
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        rc = self._L.dawn_batcher_search(self._h, _ptr(q), count, _ptr(labels), _ptr(dist), C.byref(n))
        if rc != 0:
            raise DawnError(rc, self._L.dawn_batcher_last_error().decode("utf-8", "replace"))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())

    def stats(self) -> dict:
        b, q, m = C.c_uint64(), C.c_uint64(), C.c_uint64()
        _check(self._L.dawn_batcher_stats(self._h, C.byref(b), C.byref(q), C.byref(m)))
        return {"batches": b.value, "queries": q.value, "largest_batch": m.value}

    def close(self):
        if getattr(self, "_h", None):
            self._L.dawn_batcher_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiIndex:
    """Several GPUs, one process: one shard per listed device, searched concurrently, merged on the
    first device (include/dawn_index.h: dawn_multi_*).  Same method names as `Index`."""

    def __init__(self, devices, quantization: int = ScalarKind.F16):
        # The library binds NCCL at run time and prefers one that is already mapped.  In a Python process that will also
        # import torch, torch's bundled NCCL has to be the one: it is newer than the system copy and the dynamic loader
        # shares libnccl.so.2 by SONAME.  (A Rust / C++ host has no such concern.)
        if len(set(devices)) > 1:
            import importlib.util
            if importlib.util.find_spec("torch") is not None:
                import torch  # noqa: F401
        self._L = load_library()
        dev = (C.c_int * len(devices))(*devices)
        h = _vp()
        self._check(self._L.dawn_multi_create(dev, len(devices), quantization, C.byref(h)))
        self._h = h

    def _check(self, rc):
        if rc != 0:
            raise DawnError(rc, self._L.dawn_multi_last_error().decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "_h", None):
            self._L.dawn_multi_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reserve(self, capacity: int) -> None:
        self._check(self._L.dawn_multi_reserve(self._h, capacity))

    def add(self, label: int, vector) -> None:
        v = np.ascontiguousarray(vector, dtype=np.float32)
        self._check(self._L.dawn_multi_add(self._h, int(label), _ptr(v)))

    def add_batch(self, labels, vectors) -> None:
        lab = np.ascontiguousarray(labels, dtype=np.uint64)
        v = np.ascontiguousarray(vectors, dtype=np.float32).reshape(-1, EM_LEN)
        self._check(self._L.dawn_multi_add_batch(self._h, _ptr(lab), _ptr(v), v.shape[0]))

    def add_synthetic(self, seed: int, first_row: int, n: int) -> None:
        self._check(self._L.dawn_multi_add_synthetic(self._h, seed, first_row, n))

    def remove(self, label: int) -> int:
        """Remove the label's vectors from every shard; returns the rows removed."""
        n = C.c_size_t(0)
        self._check(self._L.dawn_multi_remove(self._h, int(label), C.byref(n)))
        return int(n.value)

    def remove_batch(self, labels) -> int:
        lab = np.ascontiguousarray(labels, dtype=np.uint64).reshape(-1)
        n = C.c_size_t(0)
        self._check(self._L.dawn_multi_remove_batch(self._h, _ptr(lab), lab.shape[0], C.byref(n)))
        return int(n.value)

    def search(self, query, count: int) -> Matches:
        q = np.ascontiguousarray(query, dtype=np.float32)
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        self._check(self._L.dawn_multi_search(self._h, _ptr(q), count, _ptr(labels), _ptr(dist), C.byref(n)))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())

    def search_batch(self, queries, count: int):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        b = q.shape[0]
        labels = np.zeros((b, max(count, 1)), dtype=np.uint64)
        dist = np.zeros((b, max(count, 1)), dtype=np.float32)
        counts = np.zeros(b, dtype=np.uint64)
        self._check(self._L.dawn_multi_search_batch(self._h, _ptr(q), b, count, _ptr(labels), _ptr(dist), _ptr(counts)))
        return labels, dist, counts.astype(np.int64)

    def search_batch_limit(self, queries, count: int, distance_limit: float):
        """search_batch with UdpPacket::Search's distance_limit applied on every shard before the exchange."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        b = q.shape[0]
        labels = np.zeros((b, max(count, 1)), dtype=np.uint64)
        dist = np.zeros((b, max(count, 1)), dtype=np.float32)
        counts = np.zeros(b, dtype=np.uint64)
        self._check(self._L.dawn_multi_search_batch_limit(self._h, _ptr(q), b, count, float(distance_limit), _ptr(labels),
                                                          _ptr(dist), _ptr(counts)))
        return labels, dist, counts.astype(np.int64)

    def size(self) -> int:
        return int(self._L.dawn_multi_size(self._h))

    def capacity(self) -> int:
        return int(self._L.dawn_multi_capacity(self._h))

    def shards(self) -> int:
        return int(self._L.dawn_multi_shards(self._h))

    def set_option(self, key: str, value: int) -> None:
        """'exchange': 0 auto, 1 peer copies, 2 NCCL all-gather; other keys go to every shard's index."""
        self._check(self._L.dawn_multi_set_option(self._h, key.encode(), int(value)))

    def stats(self) -> dict:
        st = MultiStats()
        self._check(self._L.dawn_multi_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    def save(self, path: str) -> None:
        """One file for the whole handle (include/dawn_index.h: dawn_multi_save); searches go on while it is written."""
        self._check(self._L.dawn_multi_save(self._h, os.fsencode(path)))

    def load(self, path: str) -> None:
        """A dawn_multi_save file or a single-index file, onto this handle's shards, whatever their number."""
        self._check(self._L.dawn_multi_load(self._h, os.fsencode(path)))

    view = load

    def get(self, label: int) -> np.ndarray:
        out = np.zeros(EM_LEN, dtype=np.float32)
        self._check(self._L.dawn_multi_get(self._h, int(label), _ptr(out)))
        return out

    def get_i24(self, label: int) -> bytes:
        out = np.zeros(EM_LEN * 3, dtype=np.uint8)
        self._check(self._L.dawn_multi_get_i24(self._h, int(label), _ptr(out)))
        return out.tobytes()

    def verify(self) -> dict:
        bad = C.c_size_t(0)
        lo, hi = C.c_float(0), C.c_float(0)
        self._check(self._L.dawn_multi_verify(self._h, C.byref(bad), C.byref(lo), C.byref(hi)))
        return {"bad_rows": int(bad.value), "min_norm": float(lo.value), "max_norm": float(hi.value)}

    def search_i24(self, query1152: bytes, count: int, distance_limit=None) -> Matches:
        buf = np.frombuffer(query1152, dtype=np.uint8).copy()
        labels = np.zeros(max(count, 1), dtype=np.uint64)
        dist = np.zeros(max(count, 1), dtype=np.float32)
        n = C.c_size_t(0)
        self._check(self._L.dawn_multi_search_i24(self._h, _ptr(buf), count, int(distance_limit is not None),
                                                  float(distance_limit or 0.0), _ptr(labels), _ptr(dist), C.byref(n)))
        return Matches(labels[: n.value].copy(), dist[: n.value].copy())


def new_index(options: IndexOptions | None = None) -> Index:
    """usearch::ffi::new_index (search_provider.rs:102)."""
    return Index(options or IndexOptions())


def merge_results_device(device: int, d_labels: int, d_dist: int, d_counts: int, n_lists: int,
                         batch: int, k: int, d_labels_out: int, d_dist_out: int, d_counts_out: int,
                         stream: int = 0, list_stride_bytes: int = 0) -> None:
    _check(load_library().dawn_merge_results_device(device, d_labels, d_dist, d_counts, n_lists,
                                                    list_stride_bytes, batch, k, d_labels_out, d_dist_out,
                                                    d_counts_out, stream))
