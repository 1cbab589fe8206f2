"""ctypes loader for the C oracle plus an independent numpy restatement.

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs; the product package
(dawnsearch_b200) must never import this module.

PARITY UNPINNED: the reference has no tests or golden vectors for this path
(/root/reference/.github/workflows/build.yml:32); see dawn_oracle.h.

The numpy functions restate the same semantics a second time, independently of
the C code (src/search/vector.rs:128-134 order: one f32 multiply and one f32 add
per element, in index order), so the two can be checked against each other.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

EM_LEN = 384  # src/search/vector.rs:26
_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "build", "libdawn_oracle.so")
_lib = None

_u64p = C.POINTER(C.c_uint64)
_f32p = C.POINTER(C.c_float)
_u16p = C.POINTER(C.c_uint16)
_i8p = C.POINTER(C.c_int8)
_u8p = C.POINTER(C.c_uint8)


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (gcc only)."""
    if force or not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(os.path.join(_HERE, f)) > os.path.getmtime(_LIB_PATH)
        for f in os.listdir(_HERE)
        if f.endswith((".c", ".h")) or f == "Makefile"
    ):
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True)
    return _LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.dawn_oracle_distance_l2sq.restype = C.c_float
        L.dawn_oracle_distance_ip.restype = C.c_float
        L.dawn_oracle_distance_cosine.restype = C.c_float
        L.dawn_oracle_vector_length.restype = C.c_float
        L.dawn_oracle_is_normalized.restype = C.c_int
        L.dawn_oracle_f32_to_i16.restype = C.c_int16
        L.dawn_oracle_f32_to_i16.argtypes = [C.c_float]
        L.dawn_oracle_distance_i16.restype = C.c_uint64
        L.dawn_oracle_distance_ip_i16.restype = C.c_uint64
        L.dawn_oracle_distance_reduced.restype = C.c_float
        L.dawn_oracle_distance_i8.restype = C.c_uint32
        L.dawn_oracle_from24.restype = C.c_int
        L.dawn_oracle_f32_to_f16.restype = C.c_uint16
        L.dawn_oracle_f32_to_f16.argtypes = [C.c_float]
        L.dawn_oracle_f16_to_f32.restype = C.c_float
        L.dawn_oracle_f16_to_f32.argtypes = [C.c_uint16]
        L.dawn_oracle_store_f16.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.dawn_oracle_store_i8.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.dawn_oracle_synth_row_f32.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
        L.dawn_oracle_synth_rows_f16.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p]
        for name in ("dawn_oracle_search_f16", "dawn_oracle_search_f32"):
            f = getattr(L, name)
            f.restype = C.c_size_t
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                          C.c_void_p, C.c_void_p]
        L.dawn_oracle_search_i8.restype = C.c_size_t
        L.dawn_oracle_search_i8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                            C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.dawn_oracle_score_f16.restype = C.c_float
        L.dawn_oracle_score_f16.argtypes = [C.c_void_p, C.c_void_p]
        L.dawn_oracle_best_new.restype = C.c_void_p
        L.dawn_oracle_best_new.argtypes = [C.c_size_t]
        L.dawn_oracle_best_free.argtypes = [C.c_void_p]
        L.dawn_oracle_best_insert.restype = C.c_int
        L.dawn_oracle_best_insert.argtypes = [C.c_void_p, C.c_uint64, C.c_float]
        L.dawn_oracle_best_sort.argtypes = [C.c_void_p]
        L.dawn_oracle_best_len.restype = C.c_size_t
        L.dawn_oracle_best_len.argtypes = [C.c_void_p]
        L.dawn_oracle_best_worst_distance.restype = C.c_float
        L.dawn_oracle_best_worst_distance.argtypes = [C.c_void_p]
        L.dawn_oracle_best_get.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.dawn_cpu_scan_f16.restype = C.c_int
        L.dawn_cpu_scan_f16.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                        C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
        L.dawn_cpu_scan_threads_default.restype = C.c_int
        if hasattr(L, "dawn_hnsw_new"):
            L.dawn_hnsw_new.restype = C.c_void_p
            L.dawn_hnsw_new.argtypes = [C.c_size_t, C.c_size_t, C.c_size_t, C.c_uint64]
            L.dawn_hnsw_free.argtypes = [C.c_void_p]
            L.dawn_hnsw_add.restype = C.c_int
            L.dawn_hnsw_add.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
            L.dawn_hnsw_search.restype = C.c_size_t
            L.dawn_hnsw_search.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                           C.c_void_p]
            L.dawn_hnsw_size.restype = C.c_size_t
            L.dawn_hnsw_size.argtypes = [C.c_void_p]
            L.dawn_hnsw_set_ef_search.argtypes = [C.c_void_p, C.c_size_t]
            L.dawn_hnsw_add_batch.restype = C.c_int
            L.dawn_hnsw_add_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
            L.dawn_hnsw_search_batch.restype = C.c_int
            L.dawn_hnsw_search_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int,
                                                 C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


# ----------------------------------------------------------------- C-backed API


def distance_cosine(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().dawn_oracle_distance_cosine(_p(a), _p(b)))


def distance_ip(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().dawn_oracle_distance_ip(_p(a), _p(b)))


def distance_l2sq(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().dawn_oracle_distance_l2sq(_p(a), _p(b)))


def vector_length(v) -> float:
    v = _f32(v)
    return float(lib().dawn_oracle_vector_length(_p(v)))


def is_normalized(v) -> bool:
    v = _f32(v)
    return bool(lib().dawn_oracle_is_normalized(_p(v)))


def normalize(v) -> np.ndarray:
    v = _f32(v).copy()
    lib().dawn_oracle_normalize(_p(v))
    return v


def to24(v) -> bytes:
    v = _f32(v)
    out = np.zeros(EM_LEN * 3, dtype=np.uint8)
    lib().dawn_oracle_to24(_p(v), _p(out))
    return out.tobytes()


def from24(data: bytes):
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    out = np.zeros(EM_LEN, dtype=np.float32)
    ok = lib().dawn_oracle_from24(_p(buf), _p(out))
    return out, bool(ok)


def store_f16(rows) -> np.ndarray:
    rows = _f32(rows).reshape(-1, EM_LEN)
    out = np.empty(rows.shape, dtype=np.uint16)
    lib().dawn_oracle_store_f16(_p(rows), rows.shape[0], _p(out))
    return out.view(np.float16)


def store_i8(rows):
    rows = _f32(rows).reshape(-1, EM_LEN)
    out = np.empty(rows.shape, dtype=np.int8)
    scales = np.empty(rows.shape[0], dtype=np.float32)
    lib().dawn_oracle_store_i8(_p(rows), rows.shape[0], _p(out), _p(scales))
    return out, scales


def synth_rows_f32(seed: int, first_row: int, n: int) -> np.ndarray:
    out = np.empty((n, EM_LEN), dtype=np.float32)
    L = lib()
    for i in range(n):
        L.dawn_oracle_synth_row_f32(seed, first_row + i, C.c_void_p(out[i].ctypes.data))
    return out


def synth_rows_f16(seed: int, first_row: int, n: int) -> np.ndarray:
    out = np.empty((n, EM_LEN), dtype=np.uint16)
    L = lib()
    if n < 20000:
        L.dawn_oracle_synth_rows_f16(seed, first_row, n, _p(out))
    else:  # rows are independent: slice over host threads (ctypes drops the GIL)
        from concurrent.futures import ThreadPoolExecutor

        nt = max(1, min(os.cpu_count() or 1, 64))
        step = (n + nt - 1) // nt

        def work(t):
            a, b = t * step, min(n, (t + 1) * step)
            if b > a:
                L.dawn_oracle_synth_rows_f16(seed, first_row + a, b - a, C.c_void_p(out[a:b].ctypes.data))

        with ThreadPoolExecutor(nt) as ex:
            list(ex.map(work, range(nt)))
    return out.view(np.float16)


def _labels_arg(labels, n):
    if labels is None:
        return None, None
    labels = np.ascontiguousarray(labels, dtype=np.uint64)
    assert labels.shape[0] == n
    return labels, _p(labels)


def search_f16(corpus_f16, labels, query, k):
    """Exact top-k over fp16-stored rows -> (labels[count], distances[count])."""
    corpus = np.ascontiguousarray(corpus_f16).view(np.uint16).reshape(-1, EM_LEN)
    n = corpus.shape[0]
    keep, lp = _labels_arg(labels, n)
    q = _f32(query)
    lo = np.zeros(max(k, 1), dtype=np.uint64)
    do = np.zeros(max(k, 1), dtype=np.float32)
    cnt = lib().dawn_oracle_search_f16(_p(corpus), lp, n, _p(q), k, _p(lo), _p(do))
    return lo[:cnt].copy(), do[:cnt].copy()


def search_f32(corpus_f32, labels, query, k):
    corpus = _f32(corpus_f32).reshape(-1, EM_LEN)
    n = corpus.shape[0]
    keep, lp = _labels_arg(labels, n)
    q = _f32(query)
    lo = np.zeros(max(k, 1), dtype=np.uint64)
    do = np.zeros(max(k, 1), dtype=np.float32)
    cnt = lib().dawn_oracle_search_f32(_p(corpus), lp, n, _p(q), k, _p(lo), _p(do))
    return lo[:cnt].copy(), do[:cnt].copy()


def search_i8(corpus_i8, scales, labels, query, k):
    corpus = np.ascontiguousarray(corpus_i8, dtype=np.int8).reshape(-1, EM_LEN)
    scales = _f32(scales)
    n = corpus.shape[0]
    keep, lp = _labels_arg(labels, n)
    q = _f32(query)
    lo = np.zeros(max(k, 1), dtype=np.uint64)
    do = np.zeros(max(k, 1), dtype=np.float32)
    cnt = lib().dawn_oracle_search_i8(_p(corpus), _p(scales), lp, n, _p(q), k, _p(lo), _p(do))
    return lo[:cnt].copy(), do[:cnt].copy()


def score_f16(row_f16, query) -> float:
    row = np.ascontiguousarray(row_f16).view(np.uint16)
    q = _f32(query)
    return float(lib().dawn_oracle_score_f16(_p(row), _p(q)))


def cpu_scan_f16(corpus_f16, labels, queries, k, threads=0):
    """Threaded SIMD exact scan; same results as search_f16 per query.
    Returns (labels[nq,k], distances[nq,k], counts[nq], certified)."""
    corpus = np.ascontiguousarray(corpus_f16).view(np.uint16).reshape(-1, EM_LEN)
    n = corpus.shape[0]
    keep, lp = _labels_arg(labels, n)
    q = _f32(queries).reshape(-1, EM_LEN)
    nq = q.shape[0]
    lo = np.zeros((nq, max(k, 1)), dtype=np.uint64)
    do = np.zeros((nq, max(k, 1)), dtype=np.float32)
    cnt = np.zeros(nq, dtype=np.uint64)
    cert = C.c_int(1)
    rc = lib().dawn_cpu_scan_f16(_p(corpus), lp, n, _p(q), nq, k, threads, _p(lo), _p(do), _p(cnt),
                                 C.byref(cert))
    assert rc == 0
    return lo, do, cnt.astype(np.int64), bool(cert.value)


def cpu_threads() -> int:
    return int(lib().dawn_cpu_scan_threads_default())


class BestResults:
    """src/search/best_results.rs restated (C-backed)."""

    def __init__(self, size: int):
        self._h = lib().dawn_oracle_best_new(size)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().dawn_oracle_best_free(self._h)
            self._h = None

    def insert(self, id_: int, distance: float) -> bool:
        return bool(lib().dawn_oracle_best_insert(self._h, id_, distance))

    def sort(self):
        lib().dawn_oracle_best_sort(self._h)

    def __len__(self):
        return int(lib().dawn_oracle_best_len(self._h))

    def worst_distance(self) -> float:
        return float(lib().dawn_oracle_best_worst_distance(self._h))

    def results(self):
        out = []
        i_ = C.c_uint64()
        d_ = C.c_float()
        for i in range(len(self)):
            lib().dawn_oracle_best_get(self._h, i, C.byref(i_), C.byref(d_))
            out.append((int(i_.value), float(d_.value)))
        return out


class Hnsw:
    """HNSW restatement (NOT USearch 0.22.3; see hnsw_restatement.c): the reference's kind of
    index with USearch's defaults (M=16, efConstruction=128, efSearch=64, IP on f32)."""

    def __init__(self, M: int = 16, ef_construction: int = 128, ef_search: int = 64, seed: int = 1):
        self._h = lib().dawn_hnsw_new(M, ef_construction, ef_search, seed)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().dawn_hnsw_free(self._h)
            self._h = None

    def add(self, label: int, vector) -> None:
        v = _f32(vector)
        lib().dawn_hnsw_add(self._h, int(label), _p(v))

    def add_batch(self, labels, vectors) -> None:
        vectors = _f32(vectors).reshape(-1, EM_LEN)
        lab = np.ascontiguousarray(labels, dtype=np.uint64)
        assert lib().dawn_hnsw_add_batch(self._h, _p(lab), _p(vectors), vectors.shape[0]) == 0

    def search_batch(self, queries, k: int, threads: int = 1):
        """nq independent searches on `threads` threads -> (labels[nq,k], distances[nq,k], counts[nq])."""
        q = _f32(queries).reshape(-1, EM_LEN)
        nq = q.shape[0]
        lo = np.zeros((nq, max(k, 1)), dtype=np.uint64)
        do = np.zeros((nq, max(k, 1)), dtype=np.float32)
        cnt = np.zeros(nq, dtype=np.uint64)
        assert lib().dawn_hnsw_search_batch(self._h, _p(q), nq, k, threads, _p(lo), _p(do), _p(cnt)) == 0
        return lo, do, cnt.astype(np.int64)

    def search(self, query, k: int):
        q = _f32(query)
        lo = np.zeros(max(k, 1), dtype=np.uint64)
        do = np.zeros(max(k, 1), dtype=np.float32)
        n = lib().dawn_hnsw_search(self._h, _p(q), k, _p(lo), _p(do))
        return lo[:n].copy(), do[:n].copy()

    def size(self) -> int:
        return int(lib().dawn_hnsw_size(self._h))

    def set_ef_search(self, ef: int) -> None:
        lib().dawn_hnsw_set_ef_search(self._h, ef)


# ------------------------------------------------------- numpy restatement


_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def np_mix64(z: np.ndarray) -> np.ndarray:
    z = z.astype(np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
    return z ^ (z >> np.uint64(31))


def np_synth_rows_f32(seed: int, first_row: int, n: int) -> np.ndarray:
    """Synthetic corpus rows: integer hash -> Irwin-Hall(4) integer -> exact int64 sum of
    squares -> IEEE f64 1/sqrt and multiply -> f32.  Every step is an exactly rounded
    IEEE operation or integer arithmetic, so CPU (C, numpy) and GPU agree bit for bit."""
    rows = (np.arange(n, dtype=np.uint64) + np.uint64(first_row))[:, None]
    cols = np.arange(EM_LEN, dtype=np.uint64)[None, :]
    with np.errstate(over="ignore"):
        idx = rows * np.uint64(EM_LEN) + cols + np.uint64(1)
        h = np_mix64(np.uint64(seed) + _GOLD * idx)
    m = np.uint64(0xFFFF)
    s = (h & m) + ((h >> np.uint64(16)) & m) + ((h >> np.uint64(32)) & m) + (h >> np.uint64(48))
    raw = s.astype(np.int64) - 131070
    sumsq = (raw * raw).sum(axis=1)
    zero = sumsq == 0
    if zero.any():
        raw[zero, 0] = 1
        sumsq[zero] = 1
    inv = 1.0 / np.sqrt(sumsq.astype(np.float64))
    return (raw.astype(np.float64) * inv[:, None]).astype(np.float32)


def np_synth_rows_f16(seed: int, first_row: int, n: int) -> np.ndarray:
    return np_synth_rows_f32(seed, first_row, n).astype(np.float16)


def np_scores_seq(stored_f32: np.ndarray, query: np.ndarray) -> np.ndarray:
    """score[r] = sequential f32 sum_i q[i]*x[r,i]; one rounding per multiply and per add."""
    x = np.ascontiguousarray(stored_f32, dtype=np.float32)
    q = _f32(query)
    acc = np.zeros(x.shape[0], dtype=np.float32)
    for i in range(x.shape[1]):
        acc = acc + q[i] * x[:, i]
    return acc


def np_search(stored_f32: np.ndarray, labels, query, k: int, row_scale=None):
    """Exact top-k by (distance asc, label asc, row asc); distance = 1 - score (f32).  Rows whose score is NaN
    are not results, so the count is min(k, rows with a non-NaN score)."""
    n = stored_f32.shape[0]
    with np.errstate(invalid="ignore", over="ignore"):
        scores = np_scores_seq(stored_f32, query)
        if row_scale is not None:
            scores = (np.asarray(row_scale, dtype=np.float32) * scores).astype(np.float32)
    dist = (np.float32(1.0) - scores).astype(np.float32)
    lab = np.arange(1, n + 1, dtype=np.uint64) if labels is None else np.asarray(labels, dtype=np.uint64)
    order = np.lexsort((np.arange(n), lab, dist))
    order = order[~np.isnan(dist[order])][:k]
    return lab[order].copy(), dist[order].copy()


def make_queries(corpus_seed: int, query_seed: int, nq: int, n_rows: int,
                 planted_fraction: float = 0.5) -> np.ndarray:
    """Synthetic f32 unit queries.  The first nq*planted_fraction are noisy copies of
    stored rows of the synthetic corpus (so a meaningful nearest neighbour exists), the
    rest are fresh unit vectors drawn from another seed."""
    qs = np_synth_rows_f32(query_seed, 0, nq).astype(np.float64)
    n_pl = int(nq * planted_fraction) if n_rows > 0 else 0
    if n_pl:
        tgt = np_mix64(np.arange(n_pl, dtype=np.uint64) + np.uint64(query_seed + 77)) % np.uint64(n_rows)
        for i, r in enumerate(tgt):
            base = np_synth_rows_f32(corpus_seed, int(r), 1)[0].astype(np.float64)
            qs[i] = base + 0.35 * qs[i]
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    return qs.astype(np.float32)


def planted_rows(query_seed: int, nq: int, n_rows: int, planted_fraction: float = 0.5) -> np.ndarray:
    n_pl = int(nq * planted_fraction) if n_rows > 0 else 0
    return (np_mix64(np.arange(n_pl, dtype=np.uint64) + np.uint64(query_seed + 77)) % np.uint64(max(n_rows, 1))).astype(np.int64)


def np_clustered_rows_f32(seed: int, first_row: int, n: int, centers: int = 1024, intrinsic: int = 24,
                          spread: float = 0.8, iso: float = 0.15) -> np.ndarray:
    """A corpus shaped more like sentence embeddings than i.i.d. noise: a mixture of `centers` unit centres;
    a row = normalize(centre + spread * (low-dimensional offset in a shared `intrinsic`-dim subspace) +
    iso * isotropic noise).  Same-cluster rows have cosine ~ 1/(1+spread^2+iso^2) ~ 0.6, the neighbourhood of
    a row has intrinsic dimension ~`intrinsic` instead of 384.  Row r depends only on (seed, r), so shards
    and chunks agree.  Used for the recall report of the HNSW stand-in (graph indexes are at their worst on
    isotropic noise); NOT a claim about MiniLM's actual distribution."""
    cen = np_synth_rows_f32(seed ^ 0xC3A5C85C, 0, centers).astype(np.float64)                # unit centres
    basis = np_synth_rows_f32(seed ^ 0x5BD1E995, 0, intrinsic).astype(np.float64)            # subspace rows (~orthogonal)
    rows = np.arange(n, dtype=np.uint64) + np.uint64(first_row)
    which = (np_mix64(rows + np.uint64(seed + 1234567)) % np.uint64(centers)).astype(np.int64)
    g_iso = np_synth_rows_f32(seed ^ 0x27D4EB2F, first_row, n).astype(np.float64)            # unit, isotropic
    z = np_synth_rows_f32(seed ^ 0x165667B1, first_row, n).astype(np.float64)[:, :intrinsic]  # ~N(0, 1/384) coords
    z *= np.sqrt(EM_LEN / intrinsic)                                                          # |z| ~ 1
    x = cen[which] + spread * (z @ basis) + iso * g_iso
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x.astype(np.float32)


def np_store_i8(rows: np.ndarray):
    """numpy twin of dawn_oracle_store_i8: scale = absmax/127 (f32 division), q = roundf(x/scale) (half away
    from zero, the reference's rounding at src/search/vector.rs:30-32), clamped to +-127; a NaN quotient (a NaN component,
    or an inf one over an inf scale) stores 0, as Rust's `as` does.  NaN components are left out of absmax."""
    rows = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, EM_LEN)
    amax = np.abs(np.where(np.isnan(rows), np.float32(0), rows)).max(axis=1).astype(np.float32)
    scale = np.where(amax > 0, (amax / np.float32(127.0)).astype(np.float32), np.float32(1.0)).astype(np.float32)
    with np.errstate(invalid="ignore"):
        t64 = (rows / scale[:, None]).astype(np.float32).astype(np.float64)  # the f32 quotient; +-0.5 is exact in f64
        q = np.where(t64 >= 0, np.floor(t64 + 0.5), np.ceil(t64 - 0.5))
    q = np.where(np.isnan(q), 0, np.clip(q, -127, 127))
    return q.astype(np.int8), scale


def np_to24(v: np.ndarray) -> bytes:
    """numpy twin of Vec::<f32>::to24 (src/search/vector.rs:74-86): ((x+1)/2 * 0x7FFFFF) as i32, low 3 bytes LE."""
    v = np.ascontiguousarray(v, dtype=np.float32).reshape(EM_LEN)
    t = (v.astype(np.float64) + 1.0) / 2.0 * float(0x7FFFFF)
    x = np.where(np.isnan(t), 0.0, np.clip(np.trunc(t), -2147483648.0, 2147483647.0)).astype(np.int64)
    x = (x & 0xFFFFFFFF).astype(np.uint32)
    out = np.empty((EM_LEN, 3), dtype=np.uint8)
    out[:, 0] = x & 0xFF
    out[:, 1] = (x >> 8) & 0xFF
    out[:, 2] = (x >> 16) & 0xFF
    return out.tobytes()


def np_from24(data: bytes) -> np.ndarray:
    """numpy twin of Vec::<f32>::from24 (src/search/vector.rs:52-72) including its `v |= 0xFF` quirk."""
    b = np.frombuffer(data, dtype=np.uint8).reshape(EM_LEN, 3).astype(np.int64)
    v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
    v = np.where((b[:, 2] & 0x80) > 0, v | 0xFF, v)
    return (v.astype(np.float64) / float(0x7FFFFF) * 2.0 - 1.0).astype(np.float32)
