"""The streaming-scan search paths' own answers at their stage, chunk, query-group and merge edges.

The scans answer every single query below the shadow's size threshold, every batch below the tensor-core paths' thresholds,
every batch of an index holding an odd row, and every escalation of every other path:
  K2      scan_topk_f16_kernel<QT> (scan_topk.cu), 4, 2 or 1 queries per pass, fp16 rows;
  K2/f32  the same kernel over the fp16 copies of a DAWN_SCALAR_F32 index (eps + kF32StoreSlack, k' >= 64), re-scored from
          the f32 vectors;
  K4      scan_topk_i8_kernel<QT>, 2 or 1 queries per pass over the 8-row blocked int8 arena, per-query eps_q;
  K5/K6   finalize over the 148 per-CTA lists, or over the 2..13 per-chunk lists of the fp16-tile int8 path (K4b,
          "i8_native" = 0): select_lists ranks the survivors above the k'-th best list head, and falls back to the
          tree merge (merge_lists) when more than 1024 survive.
Each has shape-dependent logic: ragged last stages (n mod 8; int8 n mod 16 <= 8 leaves the second block absent), one chunk
per CTA or several, fewer CTAs holding data than k' (finalize's lower bound is then -inf), the QT lane mapping, the prune's
rank count at full width, and counters that outgrow their first allocation.  The sweeps put a case on each side of these
edges; a failing case's id names the path, the corpus rows, the batch and k.

The host API re-runs every query a scan could not certify at k' < 128 through the scan at k' = 128, so a scan or finalize
fault that only costs the certificate is repaired there.  These tests therefore also require, on every call, that the path
answered on its own: the exact number of scan passes, no tensor-core or shadow batch, a selection error within the path's
eps, and no escalation or uncertified query but those the CPU model below predicts.  The device API (search_device), which
cannot escalate, is swept as well, query by query.

The model.  near_ties() names the queries a path may fail to certify whatever its selection scores: those whose exact k-th
and k'-th best scores lie within twice the eps.  certificate() predicts the outcome itself: it recomputes in f64 the
selection scores the path ranks (the fp16 rows, the fp16 copy of an f32 index, the int8 rows against the two-level int8
query split, or the dequantised fp16 rows against the fp16 query), takes the k'-th best as the weakest kept candidate and
evaluates finalize's test, 1 - (weakest + eps) > k-th distance.  Only queries within BAND of that threshold may go either
way.  On a B200 (profiles/r07_pytest_scan_edges.txt) nothing escalates on the fp16 and int8 scans of the synthetic corpora;
a DAWN_SCALAR_F32 index, whose eps (5.4e-4) carries the fp16 copies' worst-case rounding (5.1e-4), leaves 214 of 2049 queries
uncertified at k = 120 (k' = 128 is only 8 deeper), K4b escalates 9 of 33 at k = 57 (k' = 64), and the tied row of the
prune corpus is uncertified everywhere.  The host API reports counts, not queries, so its checks bound the counts by the
predicted sets; the device API's per-query flags are checked one by one.  Run with -s to print each such case's counts.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 0x5CA4ED9E        # the 200,003-row corpora (add_synthetic)
EDGE_SEED = 0x5CA4ED9F   # the edge corpora (add_batch)
PRUNE_SEED = 0x5CA4EDA0  # the prune-heavy corpora
KMAX = 120               # DAWN_MAX_K
KREF = 128               # kMaxCand: the reference is computed once this deep (the near-tie model reads the k'-th score)
N_BIG = 200_003          # 782 chunks of 256 rows (5.3 per CTA), 200,003 mod 16 = 3: a ragged last stage and int8 block
N_K4B = 800_003          # 13 chunks of the fp16-tile int8 path at its smallest chunk (65,536 rows)
N_SORTED = 100_003       # rows in ascending order of their score against one query
N_TIED, N_TIED_RANDOM = 40_000, 20_000

# the eps of the certificates (dawn_index.cu)
SCAN_EPS = 3.0e-5        # kScanEps
F32_STORE_SLACK = 5.1e-4  # kF32StoreSlack
GEMM_ACCUM_SLACK = 6.0e-5  # kGemmAccumSlack
I8_DEQUANT_SLACK = 5.6e-4  # kI8DequantSlack

# Rows of the edge corpora (8-row fp16 stages, 16-row int8 stages of two 8-row blocks, 256-row chunks, 148 CTAs)
EDGE_ROWS = [
    1, 7, 8, 9,         # one stage: short, full, one row into the second
    15, 16, 17,         # int8: second block present but short, both full, one row into the second stage
    255, 256, 257,      # one chunk, a full chunk, a second chunk of one row
    4_096, 4_097,       # 16 chunks = k' = 16 CTAs holding data: finalize's lower bound at k' = 16 is -inf below this
    32_768, 32_769,     # 128 chunks: the same at k' = 128, where up to 128 x 128 candidates survive and the tree merge runs
    37_888, 37_889,     # 148 chunks = one per CTA, and one CTA claiming a second chunk of one row
]
DEV_EDGE = [9, 4_097]   # the edge corpora the device API is swept on
EDGE_QUERIES = {n: 1024 if n in DEV_EDGE else 33 for n in EDGE_ROWS}

# Batches: scan passes of 4, 2 and 1 queries (fp16, greedily) or of 2 and 1 (int8)
BATCHES = [1, 2, 3, 4, 5, 6, 7, 8, 15, 16, 33,  # 33 and 16 are forced past the auto threshold of the tensor-core paths
           1024,  # 256 QT=4 passes
           2049]  # 513 passes: 2050 chunk counters, past their first 1024-word allocation
# k: each side of every choose_kprime class (k' = 16 for k <= 12, 32 to 28, 64 to 57, then 128)
KS = [1, 12, 13, 28, 29, 57, 58, 100, 120]
F32_KS = [1, 57, 58, 120]  # DAWN_SCALAR_F32 lists are at least 64 deep
B_BATCHES = [1, 7]  # the reference's call shape, and 4 + 2 + 1 (int8: 2 + 2 + 2 + 1)
C_BATCHES = [1, 6, 33]
DEV_BATCHES = [1, 3, 4, 7, 16, 1024]

# name -> (storage, options)
PATHS = {
    "k2": ("f16", {"force_path": 1, "shadow_i8": 0}),
    "k2f32": ("f32", {"force_path": 1}),
    "k4": ("i8", {"i8_tensor_min_batch": 0}),
}
SCANS = list(PATHS)
# K4b over N_K4B rows: chunk rows -> gathered lists (finalize's probe takes ceil(k' / lists) > 1 entries of each).
# set_option raises "i8_tensor_chunk_rows" to at least 65,536 rows, so 6 and 13 lists need a corpus of more than
# 12 x 65,536 rows rather than smaller chunks of a 200,003-row one.
K4B_CHUNKS = {524_288: 2, 262_144: 4, 150_000: 6, 65_536: 13}
for _rows, _lists in K4B_CHUNKS.items():
    PATHS[f"k4b{_lists}"] = ("i8", {"i8_native": 0, "i8_tensor_min_batch": 1, "i8_tensor_chunk_rows": _rows})
K4B_LISTS = {f"k4b{lists}": lists for lists in K4B_CHUNKS.values()}
K4B_BATCHES = [1, 33]
K4B_KS = [1, 13, 29, 57, 58, 100]  # K4b serves k <= 100; its lists are at least 64 deep

DEFAULTS = {"force_path": 0, "shadow_i8": 0, "i8_tensor_min_batch": 16, "i8_native": 1, "i8_tensor_chunk_rows": 4 << 20}

# Prune-heavy corpora: named batches are lists of query indices
SORTED_BATCHES = {  # q0 (query 0) sees every new chunk beat its threshold, so its buffer drives every query into the prune
    "4q0first": [0, 1, 2, 3], "4q0last": [1, 2, 3, 0], "2q0first": [0, 1], "2q0last": [1, 0], "6q0last": [1, 2, 3, 4, 5, 0]}
TIED_BATCHES = {  # query 0 is the tied row itself: in a QT=4, a QT=2 and a QT=1 pass (int8: lanes 0 and 1 of QT=2, QT=1)
    "7tiefirst": [0, 1, 2, 3, 0, 4, 0], "7tielast": [1, 0, 2, 3, 4, 0, 0]}
PRUNE_KS = [1, 10, 120]

# |margin| of finalize's certificate test below which the model does not predict the outcome: the f32 scan and tensor-core
# scores differ from the f64 ones the model ranks by a few 1e-6 at most (DESIGN.md section 2: 9.5e-7 and 2.0e-6 observed)
BAND = 1e-5
# which selection scores each path ranks (certificate()), and which its escalations rank
SELECTOR = {"k2": "f16", "k2f32": "f32copy", "k4": "i8scan", **{p: "k4b" for p in K4B_LISTS}}
ESCALATION = {"k2": "k2", "k2f32": "k2f32", "k4": "k4", **{p: "k4" for p in K4B_LISTS}}


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def perm_labels(oracle, n, salt=3, base=1):
    return (np.argsort(oracle.np_mix64(np.arange(n, dtype=np.uint64) + np.uint64(salt)), kind="stable") + base).astype(np.uint64)


def f32_rows(oracle, seed, n):
    return np.concatenate([oracle.np_synth_rows_f32(seed, i, min(20_000, n - i)) for i in range(0, n, 20_000)])


def choose_kprime(k):
    """dawn_index.cu:choose_kprime"""
    want, kp = k + max(k // 8, 4), 16
    while kp < want:
        kp *= 2
    return min(kp, 128)


def path_kprime(path, k):
    return max(64, choose_kprime(k)) if path == "k2f32" or path.startswith("k4b") else choose_kprime(k)


def passes(path, batch):
    if path.startswith("k4b"):
        return 0
    if path == "k4":
        return (batch + 1) // 2
    return batch // 4 + (batch % 4) // 2 + batch % 2


def i8_split(qs):
    """s1 hi + s2 lo of prep_queries_i8_kernel restated, in f64: hi and lo are the kernel's integers (f32 quotients, rintf,
    the residual of one fmaf)."""
    x = np.ascontiguousarray(qs, dtype=np.float32)
    amax = np.abs(x).max(axis=1)
    s1 = np.where(amax > 0, amax / np.float32(127), np.float32(1)).astype(np.float32)[:, None]
    hi = np.clip(np.rint(x / s1), -127, 127)
    r = (x.astype(np.float64) - s1.astype(np.float64) * hi).astype(np.float32)
    rmax = np.abs(r).max(axis=1)
    s2 = np.where(rmax > 0, rmax / np.float32(127), np.float32(1)).astype(np.float32)[:, None]
    lo = np.clip(np.rint(r / s2), -127, 127)
    return s1.astype(np.float64) * hi + s2.astype(np.float64) * lo


def i8_scan_eps(qs):
    """eps_q of the int8 scan (prep_queries_i8_kernel): 1.03 ||q - s1 hi - s2 lo|| + 3e-5."""
    e = np.ascontiguousarray(qs, dtype=np.float64) - i8_split(qs)
    return np.sqrt((e * e).sum(axis=1)) * 1.03 + 3.0e-5


def k3_eps(qs, accum_slack):
    """eps_q of the fp16 tiles (gemm_topk.cu:prep_queries_kernel): 1.02 ||q - fp16(q)|| + the accumulation slack."""
    x = np.ascontiguousarray(qs, dtype=np.float32)
    d = x.astype(np.float64) - x.astype(np.float16).astype(np.float64)
    return np.sqrt((d * d).sum(axis=1)) * 1.02 + accum_slack


def path_eps(path, qs):
    """Per-query eps of the path's certificate (the queries here are unit vectors: no scaling by |q|)."""
    if path == "k2":
        return np.full(len(qs), SCAN_EPS)
    if path == "k2f32":
        return np.full(len(qs), SCAN_EPS + F32_STORE_SLACK)
    if path == "k4":
        return i8_scan_eps(qs)
    return k3_eps(qs, GEMM_ACCUM_SLACK + I8_DEQUANT_SLACK)


def near_ties(want, eps, k, kp):
    """Queries a select-then-re-score path may leave uncertified at k': the certificate holds once the k-th exact score is
    more than eps above the weakest kept selection score, which lies within eps of the k'-th exact score.  So a query whose
    exact k-th and k'-th best scores lie within 2 eps may fail it; any other must pass.  `want` is the oracle's top-KREF
    (distance = 1 - score, rounded once); with fewer than k' rows every row is a candidate and the certificate holds."""
    wl, wd, wc = want
    if kp > wd.shape[1]:
        raise ValueError("the reference is not deep enough")
    full = wc >= kp
    gap = wd[:, kp - 1].astype(np.float64) - wd[:, k - 1].astype(np.float64)
    return np.flatnonzero(full & (gap <= 2.0 * np.asarray(eps) + 1e-6))


def selection_top(selector, rows, stored, qs, want):
    """The KREF best selection scores of every query, descending, in f64 (-inf past the corpus)."""
    if selector == "f16":  # the scan scores the fp16 rows with the f32 query: the exact score to within 1e-6
        return np.where(np.arange(KREF)[None, :] < want[2][:, None], 1.0 - want[1].astype(np.float64), -np.inf)
    if selector == "f32copy":
        x, q = rows.astype(np.float16), np.asarray(qs, dtype=np.float64)
    elif selector == "i8scan":
        x, q = stored[0].astype(np.float64) * stored[1][:, None].astype(np.float64), i8_split(qs)
    else:  # k4b: rows dequantised to fp16 (i8_tensor.cu), the fp16-rounded query on the tensor cores
        x = (stored[0].astype(np.float32) * stored[1][:, None]).astype(np.float32).astype(np.float16)
        q = np.asarray(qs, dtype=np.float32).astype(np.float16).astype(np.float64)
    top = np.full((len(qs), KREF), -np.inf)
    for r0 in range(0, len(x), 25_000):
        s = q @ x[r0:r0 + 25_000].astype(np.float64).T
        s = np.concatenate([top, s], axis=1)
        keep = min(KREF, s.shape[1])
        top[:, :keep] = -np.sort(-np.partition(s, s.shape[1] - keep, axis=1)[:, s.shape[1] - keep:], axis=1)
    return top


def certificate(c, path, batch, k, kp=None):
    """Predicted flag of each query of the batch at k': 1 certified, -1 not, 0 within BAND of finalize's threshold."""
    kp = kp or path_kprime(path, k)
    r = c.rows(batch)
    wl, wd, wc = c.want
    if c.nrows < kp:  # fewer rows than k': every row is a candidate
        return np.ones(len(r), dtype=int)
    weakest = c.sel[SELECTOR[path]][r, kp - 1]
    margin = (1.0 - (weakest + path_eps(path, c.queries[r]))) - wd[r, k - 1].astype(np.float64)
    return np.where(margin > BAND, 1, np.where(margin < -BAND, -1, 0))


class Corpus:
    def __init__(self, kind, n, idx, queries, want, batches=None, nrows=0, sel=None):
        self.kind, self.n, self.idx, self.queries, self.want = kind, n, idx, queries, want
        self.batches, self.nrows, self.sel = batches or {}, nrows, sel or {}

    def rows(self, batch):
        return np.arange(batch) if isinstance(batch, int) else np.asarray(self.batches[batch])

    def reference(self, batch, k, deep=False):
        """The oracle's top-k of the batch's queries: a prefix of the top-KREF under (distance, label, row)."""
        r = self.rows(batch)
        wl, wd, wc = self.want
        if deep:
            return wl[r], wd[r], wc[r]
        return wl[r, :k], wd[r, :k], np.minimum(wc[r], k)

    def qs(self, batch):
        return self.queries[self.rows(batch)]


def reference(oracle, kind, stored, labels, qs):
    """The oracle's top-KREF of every query over the stored rows: (labels, distances, counts)."""
    if kind == "f16":
        wl, wd, wc, certified = oracle.cpu_scan_f16(stored, labels, qs, KREF)
        if certified:  # its own slack held; otherwise (long ties) the oracle answers query by query
            return wl, wd, wc
        one = lambda q: oracle.search_f16(stored, labels, q, KREF)  # noqa: E731
    elif kind == "i8":
        one = lambda q: oracle.search_i8(stored[0], stored[1], labels, q, KREF)  # noqa: E731
    else:
        one = lambda q: oracle.search_f32(stored, labels, q, KREF)  # noqa: E731
    with ThreadPoolExecutor(min(64, os.cpu_count() or 1)) as ex:
        res = list(ex.map(one, qs))
    wl = np.zeros((len(qs), KREF), dtype=np.uint64)
    wd = np.zeros((len(qs), KREF), dtype=np.float32)
    wc = np.zeros(len(qs), dtype=np.int64)
    for i, (l, d) in enumerate(res):
        wc[i] = len(l)
        wl[i, :len(l)], wd[i, :len(l)] = l, d
    return wl, wd, wc


def store(oracle, kind, rows):
    return oracle.store_f16(rows) if kind == "f16" else oracle.store_i8(rows) if kind == "i8" else rows


def stored_scores(kind, stored, q):
    x = stored[0].astype(np.float64) * stored[1][:, None] if kind == "i8" else np.asarray(stored, dtype=np.float64)
    return x @ q.astype(np.float64)


def corpus_data(oracle, kind, name, shared):
    """(rows to add or None for add_synthetic, labels or None, stored rows, queries, named batches) of one corpus."""
    if name in (N_BIG, N_K4B):
        if ("big", name) not in shared:
            shared[("big", name)] = f32_rows(oracle, SEED, name)
        rows = shared[("big", name)]
        qs = oracle.make_queries(SEED, 1, max(BATCHES) if name == N_BIG else max(K4B_BATCHES), name)
        stored = oracle.synth_rows_f16(SEED, 0, name) if kind == "f16" else store(oracle, kind, rows)
        return None, None, stored, qs, {}
    if name == "sorted":
        rows = f32_rows(oracle, PRUNE_SEED, N_SORTED)
        qs = oracle.make_queries(PRUNE_SEED, 5, 6, N_SORTED)
        order = np.argsort(stored_scores(kind, store(oracle, kind, rows), qs[0]), kind="stable")
        rows = np.ascontiguousarray(rows[order])
        labels = perm_labels(oracle, N_SORTED, salt=7)
        return rows, labels, store(oracle, kind, rows), qs, SORTED_BATCHES
    if name == "tied":
        base = oracle.np_synth_rows_f32(PRUNE_SEED + 1, 0, 1)
        rows = np.concatenate([np.repeat(base, N_TIED, axis=0), oracle.np_synth_rows_f32(PRUNE_SEED + 2, 0, N_TIED_RANDOM)])
        n = len(rows)
        rows = np.ascontiguousarray(rows[perm_labels(oracle, n, salt=9, base=0).astype(np.int64)])  # ties spread over all chunks
        labels = perm_labels(oracle, n, salt=11)
        qs = np.concatenate([base, oracle.make_queries(PRUNE_SEED + 2, 6, 4, N_TIED_RANDOM)])
        return rows, labels, store(oracle, kind, rows), qs, TIED_BATCHES
    if "edge" not in shared:
        shared["edge"] = f32_rows(oracle, EDGE_SEED, max(EDGE_ROWS))
    rows = shared["edge"][:name]
    labels = perm_labels(oracle, name)
    return rows, labels, store(oracle, kind, rows), oracle.make_queries(EDGE_SEED, 2, EDGE_QUERIES[name], name), {}


KINDS = {"f16": "F16", "f32": "F32", "i8": "I8"}


def build_corpus(dawn, oracle, kind, name, shared):
    rows, labels, stored, qs, batches = corpus_data(oracle, kind, name, shared)
    n = len(stored[0]) if kind == "i8" else len(stored)
    idx = dawn.new_index(dawn.IndexOptions(quantization=getattr(dawn.ScalarKind, KINDS[kind]), capacity=n))
    if rows is None:
        idx.add_synthetic(SEED, 0, n)  # labels 1..n, as the oracle's when it is given none
    else:
        idx.add_batch(labels, rows)
    want = reference(oracle, kind, stored, labels, qs)
    assert (want[2] == min(KREF, n)).all()
    if rows is None and kind == "f32":
        rows = shared[("big", name)]
    selectors = [SELECTOR[p] for p in PATHS if PATHS[p][0] == kind and (name == N_K4B or not p.startswith("k4b"))]
    sel = {s: selection_top(s, rows, stored, qs, want) for s in set(selectors)}
    return Corpus(kind, name, idx, qs, want, batches, n, sel), stored, labels


@pytest.fixture(scope="module")
def corpora(dawn, oracle):
    """corpora(kind, name) -> Corpus, built on first use and kept for the module: an index and the oracle's top-KREF."""
    cache, shared = {}, {}

    def get(kind, name, with_stored=False):
        if (kind, name) not in cache:
            cache[(kind, name)] = build_corpus(dawn, oracle, kind, name, shared)
        c, stored, labels = cache[(kind, name)]
        return (c, stored, labels) if with_stored else c

    yield get
    for c, _, _ in cache.values():
        c.idx.close()


def use(idx, opts):
    for key, val in {**DEFAULTS, **opts}.items():
        idx.set_option(key, val)


def mismatches(got, want):
    gl, gd, gc = got
    wl, wd, wc = want
    valid = np.arange(wl.shape[1])[None, :] < wc[:, None]
    bad = (gc != wc) | (((gl != wl) | (bits(gd) != bits(wd))) & valid).any(axis=1)
    return np.flatnonzero(bad)


def check(c, what, got, p, flags=None):
    """The oracle's bits, answered by the path alone: no uncertified query (and so no escalation) but those certificate()
    predicts.  what = (path, corpus, batch, k); flags: the device API's per-query flags (it re-runs nothing)."""
    path, _, batch, k = what
    want = c.reference(batch, k)
    nb = len(want[2])
    qs = c.qs(batch)
    pred = certificate(c, path, batch, k)
    model = near_ties(c.reference(batch, k, deep=True), path_eps(path, qs), k, path_kprime(path, k))
    assert set(np.flatnonzero(pred < 1).tolist()) <= set(model.tolist()), (what, "prediction outside the near-tie model")
    assert p["device_status"] == 0, (what, p)
    assert p["gemm_batches"] == K4B_LISTS.get(path, 0) and p["shadow_batches"] == 0, ("another path ran", what, p)
    lo, hi = int((pred < 0).sum()), int((pred < 1).sum())  # uncertified at the path's k'
    certified = np.ones(nb, dtype=bool)
    if flags is not None:
        certified = (flags & 1) == 1
        wrong = np.flatnonzero((certified & (pred < 0)) | (~certified & (pred > 0)))
        assert not len(wrong), (what, "queries whose certificate differs from the prediction", wrong[:8].tolist(),
                                [int(f) for f in flags[wrong[:8]]], p)
        assert p["device_uncertified"] == int((~certified).sum()), (what, p)
        assert p["escalations"] == 0 and p["uncertified"] == 0 and p["scan_launches"] == passes(path, nb), (what, p)
    else:
        if choose_kprime(k) < 128 or path.startswith("k4b"):  # the host API escalates to the scan at k' = 128
            again = certificate(c, ESCALATION[path], batch, k, kp=128)
            esc = p["escalations"]
            assert lo <= esc <= hi, ("the path did not answer on its own", what, f"{lo}..{hi} escalations expected", p)
            assert int(((pred < 0) & (again < 0)).sum()) <= p["uncertified"] <= int(((pred < 1) & (again < 1)).sum()), \
                ("escalations left uncertified", what, p)
        else:
            esc = 0
            assert p["escalations"] == 0 and lo <= p["uncertified"] <= hi, ("unexpected uncertified queries", what, f"{lo}..{hi}", p)
        # every finalize counts what it left uncertified: the batch's (all escalated, if any were), then the escalations'
        assert p["device_uncertified"] == esc + p["uncertified"], (what, p)
        assert p["scan_launches"] == passes(path, nb) + esc, ("scan passes", what, f"{passes(path, nb)} + {esc} expected", p)
    eps = path_eps(path, qs).max()
    if path.startswith("k4b") and p["escalations"]:
        eps = max(eps, i8_scan_eps(qs).max())
    assert p["max_selection_error"] <= eps, ("selection error beyond the path's eps", what, eps, p)
    bad = [int(i) for i in mismatches(got, want) if certified[i]]
    assert not bad, (what, f"{len(bad)} of {nb} certified queries differ from the oracle", bad[:8], p)
    if hi or p["device_uncertified"]:  # the counts behind the figures in DESIGN.md section 2 (visible with pytest -s)
        print(f"\n  {what}: escalations {p['escalations']}, uncertified {p['uncertified']}, device_uncertified "
              f"{p['device_uncertified']}; predicted {lo}, {hi - lo} more within BAND, at k' = {path_kprime(path, k)}")


def search_host(c, path, batch, k):
    use(c.idx, PATHS[path][1])
    try:
        c.idx.profile(reset=True)
        got = c.idx.search_batch(c.qs(batch), k)
        return got, c.idx.profile(reset=True)
    finally:
        use(c.idx, {})


def search_device(idx, qs, k):
    """search_device on a side stream into sentinel-filled buffers -> ((labels, distances, counts), flags)."""
    import torch

    b = len(qs)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dq = torch.from_numpy(np.ascontiguousarray(qs)).to("cuda")
        ol = torch.full((b, k), -1, dtype=torch.int64, device="cuda")
        od = torch.full((b, k), float("nan"), dtype=torch.float32, device="cuda")
        oc = torch.full((b,), -1, dtype=torch.int32, device="cuda")
        of = torch.zeros(b, dtype=torch.int32, device="cuda")
        idx.search_device(dq.data_ptr(), b, k, ol.data_ptr(), od.data_ptr(), oc.data_ptr(), of.data_ptr(), side.cuda_stream)
    side.synchronize()
    got = (ol.cpu().numpy().view(np.uint64), od.cpu().numpy(), oc.cpu().numpy().astype(np.int64))
    return got, of.cpu().numpy()


def cases(paths, names, batches, ks, prefix="", skip=()):
    out = []
    for path in paths:
        for name in names:
            for b in batches:
                for k in (F32_KS if path == "k2f32" and ks is KS else ks):
                    if (path, name, b, k) in skip:
                        continue
                    out.append(pytest.param(path, name, b, k, id=f"{prefix}{path}-n{name}-b{b}-k{k}"))
    return out


A_CASES = cases(SCANS, [N_BIG], BATCHES, [10, KMAX])
B_CASES = cases(SCANS, [N_BIG], B_BATCHES, KS, skip={(p, N_BIG, b, KMAX) for p in SCANS for b in B_BATCHES})
C_CASES = cases(SCANS, EDGE_ROWS, C_BATCHES, [10, KMAX])
D_CASES = cases(list(K4B_LISTS), [N_K4B], K4B_BATCHES, K4B_KS)
E_CASES = cases(["k2", "k4"], ["sorted"], list(SORTED_BATCHES), PRUNE_KS) + \
    cases(["k2", "k4"], ["tied"], list(TIED_BATCHES), PRUNE_KS)


# ---------------------------------------------------------------------------------------------------- the reference
@pytest.mark.parametrize("kind,name", [("f16", N_BIG), ("f32", N_BIG), ("i8", N_BIG), ("i8", N_K4B), ("f16", 4_097),
                                       ("f32", 257), ("i8", 17), ("f16", "tied"), ("i8", "sorted")])
def test_reference_at_smaller_k_is_a_prefix(oracle, corpora, kind, name):
    """Every k is checked against a slice of the top-KREF: the oracle's own top-k must be that slice."""
    c, stored, labels = corpora(kind, name, with_stored=True)
    for k in (1, 13, 58, KMAX):
        sl, sd, sc = c.reference(len(c.queries), k)
        for i in (0, 1, len(c.queries) - 1):
            if kind == "f16":
                wl, wd = oracle.search_f16(stored, labels, c.queries[i], k)
            elif kind == "f32":
                wl, wd = oracle.search_f32(stored, labels, c.queries[i], k)
            else:
                wl, wd = oracle.search_i8(stored[0], stored[1], labels, c.queries[i], k)
            assert len(wl) == sc[i] and (wl == sl[i, :sc[i]]).all() and (bits(wd) == bits(sd[i, :sc[i]])).all(), (kind, name, i, k)


def test_tied_row_is_a_near_tie_everywhere(corpora):
    """The tied row cannot be certified at any k' (its k-th and k'-th scores are equal), and the model says so."""
    c = corpora("f16", "tied")
    for k in PRUNE_KS:
        assert 0 in near_ties(c.reference("7tiefirst", k, deep=True), SCAN_EPS, k, choose_kprime(k)).tolist()
        assert (certificate(c, "k2", "7tiefirst", k)[np.asarray(TIED_BATCHES["7tiefirst"]) == 0] == -1).all()


# ---------------------------------------------------------------------------------------------------- A-E: host API
@pytest.mark.parametrize("path,name,batch,k", A_CASES + B_CASES + C_CASES + D_CASES + E_CASES)
def test_host_api(corpora, path, name, batch, k):
    c = corpora(PATHS[path][0], name)
    got, p = search_host(c, path, batch, k)
    check(c, (path, name, batch, k), got, p)
    if name == "tied":  # the tied row's hits are one run of equal distances, in ascending label order
        for i in np.flatnonzero(c.rows(batch) == 0):
            labels, dist = got[0][i], got[1][i]
            assert (bits(dist) == bits(dist[:1])).all() and (np.diff(labels.astype(np.int64)) > 0).all(), (path, batch, k, i)


# ---------------------------------------------------------------------------------------------------- F: device API
@pytest.mark.parametrize("path,name,batch,k", cases(SCANS, [N_BIG] + DEV_EDGE, DEV_BATCHES, [10, KMAX], "dev-"))
def test_device_api(corpora, path, name, batch, k):
    """search_device cannot escalate: the scan's own answer is what a device-resident caller gets."""
    c = corpora(PATHS[path][0], name)
    qs = c.qs(batch)
    use(c.idx, PATHS[path][1])
    try:
        c.idx.profile(reset=True)
        got, flags = search_device(c.idx, qs, k)
        check(c, (path, name, batch, k), got, c.idx.profile(reset=True), flags=flags)
        host = c.idx.search_batch(qs, k)
        differ = [int(i) for i in mismatches(got, host) if flags[i] & 1]
        assert not differ, ("device and host API differ", path, name, batch, k, differ[:8])
    finally:
        use(c.idx, {})


@pytest.mark.parametrize("path", ["k2", "k4"])
def test_device_workspace_grows_and_is_reused(dawn, corpora, path):
    """One fresh handle: batches of 1, then 2049 (2050 chunk counters), then 1 through search_device, so its scan workspace
    grows and is reused."""
    kind = PATHS[path][0]
    c = corpora(kind, N_BIG)
    with dawn.new_index(dawn.IndexOptions(quantization=getattr(dawn.ScalarKind, KINDS[kind]), capacity=N_BIG)) as idx:
        idx.add_synthetic(SEED, 0, N_BIG)
        use(idx, PATHS[path][1])
        for k in (KMAX, 10):
            for batch in (1, 2049, 1):
                idx.profile(reset=True)
                got, flags = search_device(idx, c.qs(batch), k)
                check(c, (path, N_BIG, batch, k), got, idx.profile(reset=True), flags=flags)
