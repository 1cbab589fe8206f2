"""The tensor-core search paths' own answers at their tile, select and round-schedule edges.

Three tensor-core paths answer batched searches, and a fourth is kept as an A/B partner:
  K3   fp16 tiles (gemm_topk.cu);
  K4d  the int8 kernel (gemm_i8.cu) filtering an fp16 corpus through its int8 shadow, groups of 32 or 1 rows per scale;
  K4c  the same kernel over an int8 corpus;
  K4b  an int8 corpus dequantised to fp16 tiles (i8_tensor.cu, "i8_native" = 0; k <= 100 only).
Each has shape-dependent logic: 128-query tiles or 256-query CTA pairs, a ragged last corpus tile, the int8 select's one-stage
or two-stage form, and a round schedule whose growth depends on k' and on the 2048-entry candidate log.  The sweeps below put a
case on each side of every such boundary; a failing case's id names the path, the corpus rows, the batch and k.

The host API re-runs every query the tensor path could not certify (or whose log overflowed) through the exact scan, so its
answer stays right when the tensor path fails.  These tests therefore also require, on every call, that the path answered on
its own: no escalation, nothing uncertified (on the device either), no scan launched, the intended path in the profile, and on
the int8 kernel's paths, whose rounds rank exact scores, a zero selection error.  The synthetic corpora have no ties, so with
default knobs nothing escalates but the few near ties listed in NEAR_TIES.  The device API (search_device), which cannot
escalate, is swept as well.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 0x7E57ED9E       # the 200,003-row corpora (add_synthetic)
EDGE_SEED = 0x7E57ED9F  # the edge corpora (add_batch)
KMAX = 120              # DAWN_MAX_K: the reference is computed once at this k and sliced
N_BIG = 200_003         # 782 tiles of 256 rows, the last one holding 67 rows; ~9 rounds at x2 growth

# Rows of the edge corpora (256-row tiles, 8-row int8 blocks, 32-row shadow scale groups)
EDGE_ROWS = [
    65_536,  # exactly 256 tiles: the smallest corpus the int8 paths and the shadow serve
    65_537,  # a 1-row last tile, 8-row block and 32-row group
    81_664,  # 319 tiles: 256 + 256 / 4 > 319, so the x2/x4/x8 schedules fold the short last round into the one before
    81_920,  # 320 tiles: 256 + 64 = 320 is not > 320, so a last round of 64 tiles runs on its own
]

# Sweep A: batches
BATCHES = [
    1,     # one query: a 128-query tile with 127 padding queries, the int8 select's one-stage form
    64,    # the last batch with the int8 one-stage select (n_queries <= 64)
    65,    # the first with the two-stage select (prune at tau - 2 eta, then re-score exactly)
    128,   # the last batch on one 128-query tile and one CTA (K3 grows up to x32 there)
    129,   # the first on a CTA pair (256-query tile; K3 back to x4..x16)
    256,   # one full CTA-pair tile
    257,   # two CTA-pair tiles, the second holding one query: the chunk rendezvous of several query tiles
    1024,  # bench.py's batch
    2049,  # above 1024: nine CTA-pair tiles, the last holding one query
]

# Sweep B: k, each value on one side of a boundary.  K3's k' = choose_kprime(k) (16/32/64/128); the int8 kernel's
# k' = k + 4 rounded up to 4, at least 16.  Growth per round: K3 x16/x8/x4 by k' (x32..x8 on one CTA); K4c x8 for
# k' <= 64, else x4; K4d x8, clamped to x4 and x2 so that (growth - 1) * k' * 5.5 + k' fits the 2048-entry log.
KS = [
    1,    # smallest k: k' = 16 (K4b: 64)
    12,   # K3 k' = 16 (x16; x32 on one CTA), the last k with it
    13,   # K3 k' = 32 (x8; x32 on one CTA)
    28,   # K3 k' = 32, the last k with it
    29,   # K3 k' = 64 (x8; x16 on one CTA)
    44,   # K4d k' = 48: x8, the last k with it
    45,   # K4d k' = 52: x4
    57,   # K3 k' = 64, the last k with it
    58,   # K3 k' = 128 (x4; x8 on one CTA)
    60,   # K4c k' = 64: x8, the last k with it
    61,   # K4c k' = 68 > 64: x4
    100,  # the largest k K4b serves (K3 k' = 128)
    112,  # K4d k' = 116: x4, the last k with it
    113,  # K4d k' = 120: x2
    120,  # DAWN_MAX_K: K3 k' = 128 leaves 8 candidates of slack, K4 k' = 124
]
B_BATCHES = [65, 129]  # one 128-query tile (K3 on one CTA, the int8 two-stage select) / a CTA pair

# name -> (storage, options, whether the rounds rank exact scores)
PATHS = {
    "k3": ("f16", {"force_path": 2}, False),
    "k4d32": ("f16", {"force_path": 2, "shadow_i8": 1, "shadow_big_k_rows": 0}, True),
    "k4d1": ("f16", {"force_path": 2, "shadow_i8": 1, "shadow_big_k_rows": 0, "shadow_group_rows": 1}, True),
    "k4c": ("i8", {"i8_tensor_min_batch": 1, "i8_native": 1}, True),
    "k4b": ("i8", {"i8_tensor_min_batch": 1, "i8_native": 0}, False),
}
MAIN = ["k3", "k4d32", "k4d1", "k4c"]
K4B_MAX_K = 100

# (path, rows, batch, k) -> queries that K3 or K4b cannot certify.  Both select on approximate scores (an fp16-rounded query;
# K4b also dequantised rows) and certify a result only when the k'-th candidate's selection score plus the query's eps stays
# below the k-th exact score (DESIGN.md section 2).  These queries have their exact k-th and k'-th best scores within that eps,
# so no round schedule can certify them: the host API re-runs them through the scan and the device API flags them.  K3 at
# k = 120 already has k' = 128, the longest list there is.  A CPU model (the oracle's scores, eps = 1.02 ||q - fp16(q)|| +
# 6e-5) names the same K3 queries: 418, 536, 1165, 1347 and 1945 at k = 120, 61 at k = 12.
NEAR_TIES = {
    ("k3", N_BIG, 1024, 120): 2,
    ("k3", N_BIG, 2049, 120): 5,
    ("k3", N_BIG, 65, 12): 1,
    ("k3", N_BIG, 129, 12): 1,
    ("k4b", N_BIG, 65, 57): 3,
    ("k4b", N_BIG, 129, 57): 6,
}

DEFAULTS = {"force_path": 0, "shadow_i8": 0, "shadow_group_rows": 32, "shadow_big_k_rows": 40_000_000,
            "i8_tensor_min_batch": 16, "i8_native": 1, "gemm_cta_group": 0, "gemm_chunk_tiles": 0,
            "gemm_sequential_tiles": 0, "gemm_growth": 0}

# Sweep D: the tuning knobs tools/ab_gemm.py turns.  Escalations are allowed here, wrong or uncertified answers are not.
KNOBS = {
    "cta1": {"gemm_cta_group": 1},        # one CTA per 128-query tile, with several query tiles
    "cta2": {"gemm_cta_group": 2},        # CTA pairs
    "chunk1": {"gemm_chunk_tiles": 1},    # one tile per work unit
    "chunk7": {"gemm_chunk_tiles": 7},    # 7 tiles per work unit, more than the first round holds
    "seq": {"gemm_sequential_tiles": 1},  # tiles in physical order
    "growth2": {"gemm_growth": 2},
    "growth32": {"gemm_growth": 32},      # clamped to what the log holds
}
KNOB_CASES = [(name, 300) for name in KNOBS] + [("cta2", 40)]  # 40 on a CTA pair: a half-empty 256-query tile


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def perm_labels(oracle, n, salt=3, base=1):
    return (np.argsort(oracle.np_mix64(np.arange(n, dtype=np.uint64) + np.uint64(salt)), kind="stable") + base).astype(np.uint64)


def f32_rows(oracle, seed, n):
    return np.concatenate([oracle.np_synth_rows_f32(seed, i, min(20_000, n - i)) for i in range(0, n, 20_000)])


class Corpus:
    def __init__(self, kind, n, idx, queries, want):
        self.kind, self.n, self.idx, self.queries, self.want = kind, n, idx, queries, want

    def reference(self, batch, k):
        """The oracle's top-k of the first `batch` queries: a prefix of the top-KMAX under (distance, label, row)."""
        wl, wd, wc = self.want
        return wl[:batch, :k], wd[:batch, :k], np.minimum(wc[:batch], k)


def reference_i8(oracle, q8, sc, labels, qs, k):
    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        res = list(ex.map(lambda q: oracle.search_i8(q8, sc, labels, q, k), qs))
    wl = np.zeros((len(qs), k), dtype=np.uint64)
    wd = np.zeros((len(qs), k), dtype=np.float32)
    wc = np.zeros(len(qs), dtype=np.int64)
    for i, (l, d) in enumerate(res):
        wc[i] = len(l)
        wl[i, :len(l)], wd[i, :len(l)] = l, d
    return wl, wd, wc


def build_corpus(dawn, oracle, kind, n, edge_rows):
    quant = dawn.ScalarKind.F16 if kind == "f16" else dawn.ScalarKind.I8
    idx = dawn.new_index(dawn.IndexOptions(quantization=quant, capacity=n))
    if n == N_BIG:
        idx.add_synthetic(SEED, 0, n)  # labels 1..n, as the oracle's when it is given none
        labels = None
        qs = oracle.make_queries(SEED, 1, max(BATCHES), n)
        if kind == "f16":
            stored = oracle.synth_rows_f16(SEED, 0, n)
        else:
            stored = oracle.store_i8(f32_rows(oracle, SEED, n))
    else:
        rows = edge_rows[:n]
        labels = perm_labels(oracle, n)
        idx.add_batch(labels, rows)
        qs = oracle.make_queries(EDGE_SEED, 2, 129, n)
        stored = oracle.store_f16(rows) if kind == "f16" else oracle.store_i8(rows)
    if kind == "f16":
        wl, wd, wc, certified = oracle.cpu_scan_f16(stored, labels, qs, KMAX)
        assert certified
    else:
        wl, wd, wc = reference_i8(oracle, stored[0], stored[1], labels, qs, KMAX)
    assert (wc == KMAX).all()
    return Corpus(kind, n, idx, qs, (wl, wd, wc)), stored, labels


@pytest.fixture(scope="module")
def corpora(dawn, oracle):
    """corpora(kind, n) -> Corpus, built on first use and kept for the module: an index and the oracle's top-KMAX."""
    cache = {}
    edge = {}

    def get(kind, n, with_stored=False):
        if (kind, n) not in cache:
            if n != N_BIG and "rows" not in edge:
                edge["rows"] = f32_rows(oracle, EDGE_SEED, max(EDGE_ROWS))
            cache[(kind, n)] = build_corpus(dawn, oracle, kind, n, edge.get("rows"))
        c, stored, labels = cache[(kind, n)]
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


def check(what, got, want, p, knobs=False, flags=None):
    """The oracle's bits, from the intended path, answered by that path alone (escalations allowed under `knobs`).
    what = (path, rows, batch, k, ...); flags: the device API's per-query flags (it re-runs nothing)."""
    path = what[0]
    near = NEAR_TIES.get(what[:4], 0)
    assert p["device_status"] == 0, (what, p)
    assert p["gemm_batches"] == 1, ("the tensor path did not run once", what, p)
    assert p["shadow_batches"] == (1 if path.startswith("k4d") else 0), ("another path ran", what, p)
    assert p["uncertified"] == 0, (what, p)
    certified = np.ones(len(want[2]), dtype=bool)
    if flags is not None:
        certified = (flags & 1) == 1
        assert int((~certified).sum()) == near and p["device_uncertified"] == near, \
            (what, f"{int((~certified).sum())} queries without a certificate, {near} expected", p)
        assert p["escalations"] == 0 and p["scan_launches"] == 0, (what, p)
    elif not knobs:
        assert p["escalations"] == near and p["device_uncertified"] == near and p["scan_launches"] == near, \
            ("the tensor path did not answer on its own", what, f"{near} near ties expected", p)
    if PATHS[path][2] and p["escalations"] == 0:
        assert p["max_selection_error"] == 0.0, ("the rounds did not rank exact scores", what, p)
    bad = [i for i in mismatches(got, want) if certified[i]]
    assert not bad, (what, f"{len(bad)} of {len(want[2])} certified queries differ from the oracle", [int(i) for i in bad[:8]], p)


def search_host(c, path, batch, k, extra=None):
    use(c.idx, {**PATHS[path][1], **(extra or {})})
    try:
        c.idx.profile(reset=True)
        got = c.idx.search_batch(c.queries[:batch], k)
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


def cases(paths, sizes, batches, ks, prefix="", skip=()):
    out = []
    for path in paths:
        for n in sizes:
            for b in batches:
                for k in ks:
                    if (path == "k4b" and k > K4B_MAX_K) or (path, n, b, k) in skip:
                        continue
                    out.append(pytest.param(path, n, b, k, id=f"{prefix}{path}-n{n}-b{b}-k{k}"))
    return out


ALL = MAIN + ["k4b"]
A_CASES = cases(ALL, [N_BIG], BATCHES, [10, KMAX])
B_CASES = cases(ALL, [N_BIG], B_BATCHES, KS, skip={(p, N_BIG, b, k) for p in ALL for b in B_BATCHES for k in (10, KMAX)})
C_CASES = cases(ALL, EDGE_ROWS, [40, 129], [10, KMAX])


# ---------------------------------------------------------------------------------------------------- the reference
@pytest.mark.parametrize("kind,n", [("f16", N_BIG), ("i8", N_BIG), ("f16", 65_537), ("i8", 65_537)])
def test_reference_at_smaller_k_is_a_prefix(oracle, corpora, kind, n):
    """Every k below KMAX is checked against a slice of the top-KMAX: the oracle's own top-k must be that slice."""
    c, stored, labels = corpora(kind, n, with_stored=True)
    for k in (1, 13, 61, 113):
        sl, sd, _ = c.reference(len(c.queries), k)
        for i in (0, 1, len(c.queries) - 1):
            if kind == "f16":
                wl, wd = oracle.search_f16(stored, labels, c.queries[i], k)
            else:
                wl, wd = oracle.search_i8(stored[0], stored[1], labels, c.queries[i], k)
            assert len(wl) == k and (wl == sl[i]).all() and (bits(wd) == bits(sd[i])).all(), (kind, n, i, k)


# ---------------------------------------------------------------------------------------------------- A, B, C: host API
@pytest.mark.parametrize("path,n,batch,k", A_CASES + B_CASES + C_CASES)
def test_host_api(corpora, path, n, batch, k):
    c = corpora(PATHS[path][0], n)
    got, p = search_host(c, path, batch, k)
    check((path, n, batch, k), got, c.reference(batch, k), p)


# ---------------------------------------------------------------------------------------------------- D: knobs
@pytest.mark.parametrize("path", ["k3", "k4d32", "k4c"])
@pytest.mark.parametrize("knob,batch", [pytest.param(kn, b, id=f"{kn}-b{b}") for kn, b in KNOB_CASES])
@pytest.mark.parametrize("k", [10, KMAX], ids=lambda k: f"k{k}")
def test_knobs(corpora, path, knob, batch, k):
    c = corpora(PATHS[path][0], N_BIG)
    got, p = search_host(c, path, batch, k, KNOBS[knob])
    check((path, N_BIG, batch, k, knob), got, c.reference(batch, k), p, knobs=True)


# ---------------------------------------------------------------------------------------------------- E: device API
@pytest.mark.parametrize("path,n,batch,k", cases(ALL, [N_BIG], BATCHES, [10, KMAX], "dev-") +
                         cases(ALL, EDGE_ROWS, [40, 129], [10, KMAX], "dev-"))
def test_device_api(corpora, path, n, batch, k):
    """search_device cannot escalate: the tensor path's own answer is what a device-resident caller gets."""
    c = corpora(PATHS[path][0], n)
    qs = c.queries[:batch]
    use(c.idx, PATHS[path][1])
    try:
        c.idx.profile(reset=True)
        got, flags = search_device(c.idx, qs, k)
        check((path, n, batch, k), got, c.reference(batch, k), c.idx.profile(reset=True), flags=flags)
        host = c.idx.search_batch(qs, k)
        differ = [i for i in mismatches(got, host) if flags[i] & 1]
        assert not differ, ("device and host API differ", path, n, batch, k, differ[:8])
    finally:
        use(c.idx, {})


@pytest.mark.parametrize("kind", ["f16", "i8"])
def test_device_workspace_grows_and_is_reused(dawn, corpora, kind):
    """One fresh handle: batches of 64, then 2049, then 1 through search_device, so its workspace grows and is reused."""
    c = corpora(kind, N_BIG)
    quant = dawn.ScalarKind.F16 if kind == "f16" else dawn.ScalarKind.I8
    with dawn.new_index(dawn.IndexOptions(quantization=quant, capacity=N_BIG)) as idx:
        idx.add_synthetic(SEED, 0, N_BIG)
        for path in (["k3", "k4d32"] if kind == "f16" else ["k4c"]):
            use(idx, PATHS[path][1])
            for k in (KMAX, 10):
                for batch in (64, 2049, 1):
                    idx.profile(reset=True)
                    got, flags = search_device(idx, c.queries[:batch], k)
                    check((path, N_BIG, batch, k), got, c.reference(batch, k), idx.profile(reset=True), flags=flags)
        use(idx, {})
