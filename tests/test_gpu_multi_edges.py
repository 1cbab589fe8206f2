"""The multi-shard search and its device merge at their shard-count, placement, re-run and merge edges.

Three layers sit above the single-GPU search paths:
  K7        merge_results_kernel (dawn_index.cu, dawn_merge_results_device): merges n_lists sorted per-shard lists per query;
  dawn_multi  one process, one shard per listed device, a peer copy (a device listed twice) or an NCCL all-gather of one
            packed block per shard, K7 on the first device, and an exact re-run of every query a shard did not certify;
  sharded.py  one process per GPU under torch.distributed, the same block plus the shard's certificate flags, the same
            merge, and a second exchange after the re-runs.
Every answer here must come from these layers and equal a plain CPU reference bit for bit: labels, distance bits, counts.

The merge rule (merge_model, checked against a brute-force statement of it in the CPU suite): take each list's first
min(count, k) entries; drop an entry whose (distance, label) also occurs in a list with a smaller index; order the rest by
(distance, label, list index); keep the first k.  With every label stored once this is the whole-corpus answer.  A label
stored on several shards at one distance comes back as often as the lowest-index shard holding it stores it.

dawn_multi places add_batch rows in 4096-row blocks, round-robin over the shards, with a cursor that carries over between
calls and skips full shards; reserve gives each shard ceil(n / G) rows.  Placement restates that in Python, and the tests
check it through size(), capacity errors, the search route of each shard and duplicate labels.

Re-runs.  A shard re-runs a query exactly when its certificate fails.  rerun_bounds() predicts that from the shard's own
oracle scores: a query whose certificate margin (the near-tie band of test_gpu_scan_edges.py) is below -BAND must re-run,
one within BAND may, any other must not.  exact_reruns must lie between the two counts.
"""
import os
import signal
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x3A17ED60        # the add_synthetic sweep corpus
SPLIT_SEED = 0x3A17ED61  # the corpus whose two shards take different paths
PLACE_SEED = 0x3A17ED62  # the placement corpora
TIE_SEED = 0x3A17ED63    # the tied corpora
KMAX = 120               # DAWN_MAX_K
KREF = 128               # references are computed this deep once and sliced (the re-run model reads the k'-th score)
BLOCK = 4096             # dawn_multi_add_batch's block
INVALID, CAPACITY = -1, -3

# certificate eps (dawn_index.cu) and the band of the re-run model (test_gpu_scan_edges.py)
SCAN_EPS = 3.0e-5
F32_STORE_SLACK = 5.1e-4
GEMM_ACCUM_SLACK = 6.0e-5
I8_DEQUANT_SLACK = 5.6e-4
LOOSE_EPS = 1.0e-3  # K4c, K4d and K3 over an f32 index's copies: only the near-tie bound (no re-run outside it)
BAND = 1e-5

N_SWEEP = 100_003
SWEEP_G = [1, 2, 3, 8, 9, 16]
KS = [1, 12, 13, 28, 29, 57, 58, 100, 120]  # each side of every k' class
SWEEP_BATCHES = [1, 33]
N_SPLIT = 31 * BLOCK  # 126,976 rows: with G = 2 and room for 65,536 per shard, 16 blocks land on shard 0 and 15 on shard 1


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------- A. the merge model
def merge_model(lists, counts, k):
    """The documented merge of one query: lists = [(labels, distances)] per list, counts = entries each list claims.
    -> (labels, distances) of the merged answer."""
    keys, seen = [], set()
    for li, ((lab, dst), c) in enumerate(zip(lists, counts)):
        c = int(min(int(c), k))
        own = set()
        for p in range(c):
            key = (float(np.float32(dst[p])), int(lab[p]))
            own.add(key)
            if key not in seen:
                keys.append((key[0], key[1], li))
        seen |= own
    keys.sort()
    keys = keys[:k]
    return (np.array([e[1] for e in keys], dtype=np.uint64), np.array([e[0] for e in keys], dtype=np.float32))


def merge_brute(lists, counts, k):
    """The same rule stated entry by entry, without sets or a sort: the guard of merge_model."""
    kept = []
    for li, ((lab, dst), c) in enumerate(zip(lists, counts)):
        for p in range(min(int(c), k)):
            dup = any(float(lists[o][1][q]) == float(dst[p]) and int(lists[o][0][q]) == int(lab[p])
                      for o in range(li) for q in range(min(int(counts[o]), k)))
            if not dup:
                kept.append((float(dst[p]), int(lab[p]), li))
    out = []
    while kept and len(out) < k:  # selection by repeated minimum
        j = min(range(len(kept)), key=lambda i: kept[i])
        out.append(kept.pop(j))
    return np.array([e[1] for e in out], dtype=np.uint64), np.array([e[0] for e in out], dtype=np.float32)


def random_lists(rng, n_lists, k, n_dist=4, n_lab=6, count_hi=None, extra=()):
    """n_lists sorted lists of k entries from few distances and labels, so that ties and duplicates are common."""
    pool = np.concatenate([rng.choice(np.linspace(-0.5, 1.5, 9).astype(np.float32), n_dist, replace=False),
                           np.array(extra, dtype=np.float32)])
    lists, counts = [], []
    for _ in range(n_lists):
        d = rng.choice(pool, k).astype(np.float32)
        lab = rng.integers(1, n_lab + 1, k).astype(np.uint64)
        o = np.lexsort((lab, d))
        lists.append((lab[o], d[o]))
        counts.append(int(rng.integers(0, (count_hi or k + 3) + 1)))
    return lists, counts


def test_merge_model_matches_the_rule_stated_entry_by_entry():
    rng = np.random.default_rng(7)
    dups = same_shard = 0
    for trial in range(3000):
        n_lists, k = int(rng.integers(1, 6)), int(rng.integers(1, 7))
        lists, counts = random_lists(rng, n_lists, k, extra=(-np.inf, np.inf) if trial % 3 == 0 else (),
                                     count_hi=k + 3 if trial % 2 else max(1, k // 2))  # short lists: nothing cut at k
        ml, md = merge_model(lists, counts, k)
        bl, bd = merge_brute(lists, counts, k)
        assert (ml == bl).all() and (bits(md) == bits(bd)).all(), (trial, lists, counts, k)
        assert len(ml) <= k
        taken = [(float(d), int(l)) for lab, dst in [(ll[:min(c, k)], dd[:min(c, k)]) for (ll, dd), c in zip(lists, counts)]
                 for l, d in zip(lab, dst)]
        dups += len(taken) != len(set(taken))
        # a label keeps the copies it has in the lowest-index list that holds it (when nothing is cut at k)
        if len(ml) < k:
            for key in set(taken):
                first = next(li for li, ((lab, dst), c) in enumerate(zip(lists, counts))
                             if any((float(d), int(l)) == key for l, d in zip(lab[:min(c, k)], dst[:min(c, k)])))
                lab, dst = lists[first]
                c = min(counts[first], k)
                want = sum((float(d), int(l)) == key for l, d in zip(lab[:c], dst[:c]))
                got = sum((float(d), int(l)) == key for l, d in zip(ml, md))
                assert got == want, (trial, key)
                same_shard += want > 1
    assert dups > 500 and same_shard > 25  # the inputs exercise the rule (1,067 and 59 with this seed)


# ---------------------------------------------------------------------------------------------------- B. K7 alone
SENT_LABEL = 0xA5A5A5A5A5A5A5A5
SENT_DIST = 0x7FC0DEAD  # a NaN no input holds
SENT_COUNT = 0xFFFFFFFF


def block_stride(layout, batch, k):
    if layout == "dense":
        return 0
    if layout == "multi":  # dawn_multi.cu:block_bytes
        return (batch * k * 12 + batch * 4 + 15) // 16 * 16
    if layout == "sharded":  # sharded.py:ResultBlock, which also carries the flags
        return (batch * k * 12 + batch * 8 + 15) // 16 * 16
    return (batch * k * 12 + batch * 4 + 15) // 16 * 16 + 16  # "padded"


def run_merge(dawn, labels, dists, counts, k, layout, n_lists=None):
    """labels [L,B,k] u64, dists [L,B,k] f32, counts [L,B] u32 -> K7's (labels, distances, counts) on a side stream, read
    back with the sentinels left where it wrote nothing."""
    import torch

    L, B = counts.shape
    n_lists = n_lists or L
    side = torch.cuda.Stream()
    stride = block_stride(layout, B, k)
    with torch.cuda.stream(side):
        if stride == 0:
            tl = torch.from_numpy(labels.view(np.int64).copy()).cuda()
            td = torch.from_numpy(dists.copy()).cuda()
            tc = torch.from_numpy(counts.view(np.int32).copy()).cuda()
            pl, pd, pc = tl.data_ptr(), td.data_ptr(), tc.data_ptr()
        else:
            host = np.full((L, stride), 0x5A, dtype=np.uint8)
            for li in range(L):
                host[li, :B * k * 8] = labels[li].reshape(-1).view(np.uint8)
                host[li, B * k * 8:B * k * 12] = dists[li].reshape(-1).view(np.uint8)
                host[li, B * k * 12:B * k * 12 + B * 4] = counts[li].view(np.uint8)
            buf = torch.from_numpy(host).cuda()
            pl = buf.data_ptr()
            pd, pc = pl + B * k * 8, pl + B * k * 12
        ol = torch.full((B, k), SENT_LABEL - (1 << 64), dtype=torch.int64, device="cuda")
        od = torch.from_numpy(np.full((B, k), SENT_DIST, dtype=np.uint32).view(np.float32)).cuda()
        oc = torch.from_numpy(np.full(B, SENT_COUNT, dtype=np.uint32).view(np.int32)).cuda()
        dawn.merge_results_device(0, pl, pd, pc, n_lists, B, k, ol.data_ptr(), od.data_ptr(), oc.data_ptr(),
                                  side.cuda_stream, list_stride_bytes=stride)
    side.synchronize()
    return ol.cpu().numpy().view(np.uint64), od.cpu().numpy(), oc.cpu().numpy().view(np.uint32)


def check_merge(dawn, labels, dists, counts, k, layout, what):
    gl, gd, gc = run_merge(dawn, labels, dists, counts, k, layout)
    L, B = counts.shape
    for b in range(B):
        wl, wd = merge_model([(labels[li, b], dists[li, b]) for li in range(L)], counts[:, b], k)
        c = int(gc[b])
        assert c == len(wl), (what, b, c, len(wl))
        assert (gl[b, :c] == wl).all() and (bits(gd[b, :c]) == bits(wd)).all(), (what, b, gl[b, :c], wl, gd[b, :c], wd)
        assert (gl[b, c:] == SENT_LABEL).all() and (bits(gd[b, c:]) == SENT_DIST).all(), (what, b, "written past the count")


def make_merge_input(rng, n_lists, k, batch, mode):
    """[L,B,k] labels / distances and [L,B] counts of one K7 case."""
    labels = np.zeros((n_lists, batch, k), dtype=np.uint64)
    dists = np.zeros((n_lists, batch, k), dtype=np.float32)
    counts = np.zeros((n_lists, batch), dtype=np.uint32)
    for b in range(batch):
        if mode == "mixed":
            lists, cnt = random_lists(rng, n_lists, k, n_dist=6, n_lab=3 * k, count_hi=k)
        elif mode == "unique":  # distinct labels everywhere: the whole-corpus case
            perm = rng.permutation(n_lists * k * 2)[:n_lists * k] + 1
            lists, cnt = [], []
            for li in range(n_lists):
                d = np.sort(rng.random(k).astype(np.float32))
                lab = perm[li * k:(li + 1) * k].astype(np.uint64)
                o = np.lexsort((lab, d))
                lists.append((lab[o], d[o]))
                cnt.append(k)
        elif mode == "one_distance":  # the whole order rests on labels, across and within lists
            lists, cnt = random_lists(rng, n_lists, k, n_dist=1, n_lab=4 * k, count_hi=k)
        elif mode == "infinities":
            lists, cnt = random_lists(rng, n_lists, k, n_dist=2, n_lab=2 * k, count_hi=k, extra=(-np.inf, np.inf))
        elif mode == "duplicates":  # every list repeats its predecessor's entries: the compaction runs in every list
            lists, cnt = random_lists(rng, 1, k, n_dist=3, n_lab=2 * k, count_hi=k)
            for li in range(1, n_lists):
                lab, d = lists[-1]
                lab, d = lab.copy(), d.copy()
                j = int(rng.integers(0, k))
                d[j:] = np.float32(d[j] + np.float32(0.25)) if rng.random() < 0.5 else d[j:]  # same label, other distance
                o = np.lexsort((lab, d))
                lists.append((lab[o], d[o]))
                cnt.append(int(rng.integers(1, k + 1)))
            cnt[0] = k
        elif mode == "twice":  # a label twice in one list and once in another, in both orders
            lists, cnt = [], []
            for li in range(n_lists):
                d = np.full(k, np.float32(0.5))
                lab = np.arange(1, k + 1, dtype=np.uint64)
                if (li + b) % 2 == 0 and k >= 2:
                    lab[1] = lab[0]
                lists.append((lab, d))
                cnt.append(k)
        elif mode == "clamp":  # counts above k
            lists, cnt = random_lists(rng, n_lists, k, n_dist=5, n_lab=3 * k, count_hi=k)
            cnt = [[k + 1, k + 7, 1000, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF][(li + b) % 6] for li in range(n_lists)]
        elif mode == "junk":  # past each short count: entries that would rank first
            lists, cnt = random_lists(rng, n_lists, k, n_dist=5, n_lab=3 * k, count_hi=k)
            lists = [(lab.copy(), d.copy()) for lab, d in lists]
            cnt = [int(rng.integers(0, k)) if k > 1 else 0 for _ in range(n_lists)]
            for li, c in enumerate(cnt):
                lab, d = lists[li]
                d[c:] = np.array([-np.inf, np.nan], dtype=np.float32)[np.arange(k - c) % 2]
                lab[c:] = 0
        elif mode == "zero":
            lists, cnt = random_lists(rng, n_lists, k, count_hi=k)
            cnt = [0] * n_lists
        elif mode == "some_zero":
            lists, cnt = random_lists(rng, n_lists, k, n_dist=5, n_lab=3 * k, count_hi=k)
            cnt = [0 if (li + b) % 3 else c for li, c in enumerate(cnt)]
        else:
            raise ValueError(mode)
        for li, ((lab, d), c) in enumerate(zip(lists, cnt)):
            labels[li, b], dists[li, b], counts[li, b] = lab, d, c
    return labels, dists, counts


SHAPES = [(n, k) for n in (1, 2, 3, 7, 8, 9, 63, 64) for k in (1, 2, 16, 113, 120) if n * k <= 1024] + [(8, 120), (9, 113)]
MODES = ["unique", "mixed", "one_distance", "infinities", "duplicates", "twice", "clamp", "junk", "zero", "some_zero"]
MERGE_CASES = [pytest.param(n, k, 3, "mixed", "dense", id=f"L{n}-k{k}-b3-mixed-dense") for n, k in sorted(set(SHAPES))]
MERGE_CASES += [pytest.param(n, k, 3, m, "dense", id=f"L{n}-k{k}-b3-{m}-dense")
                for n, k in ((2, 16), (9, 113), (64, 16), (8, 120)) for m in MODES if m != "mixed"]
MERGE_CASES += [pytest.param(n, k, 3, m, lay, id=f"L{n}-k{k}-b3-{m}-{lay}")
                for n, k in ((3, 16), (9, 113)) for m in ("mixed", "junk", "clamp") for lay in ("multi", "sharded", "padded")]
MERGE_CASES += [pytest.param(n, k, b, "mixed", lay, id=f"L{n}-k{k}-b{b}-mixed-{lay}")
                for n, k in ((2, 10), (64, 16)) for b in (1, 2049) for lay in ("dense", "multi")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_lists,k,batch,mode,layout", MERGE_CASES)
def test_merge_kernel_against_the_model(dawn, n_lists, k, batch, mode, layout):
    rng = np.random.default_rng(n_lists * 100_000 + k * 100 + batch + MODES.index(mode) * 7)
    labels, dists, counts = make_merge_input(rng, n_lists, k, batch, mode)
    check_merge(dawn, labels, dists, counts, k, layout, (n_lists, k, batch, mode, layout))


@pytest.mark.gpu
@pytest.mark.parametrize("n_lists,k", [(25, 41), (65, 1), (1025, 1), (1, 121), (2, 0)])
def test_merge_kernel_rejects_bad_shapes(dawn, n_lists, k):
    """n_lists x k = 1025, more than 64 lists, k past DAWN_MAX_K and k = 0 are bad arguments, not device failures."""
    import torch

    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    with pytest.raises(dawn.DawnError) as e:
        dawn.merge_results_device(0, p, p, p, n_lists, 1, k, p, p, p, torch.cuda.current_stream().cuda_stream or 1)
    assert e.value.code == INVALID, str(e.value)
    labels, dists, counts = make_merge_input(np.random.default_rng(1), 2, 4, 1, "mixed")
    check_merge(dawn, labels, dists, counts, 4, "dense", "after a rejected shape")


# ---------------------------------------------------------------------------------------------------- references
def pool_map(fn, items):
    with ThreadPoolExecutor(min(64, os.cpu_count() or 1)) as ex:
        return list(ex.map(fn, items))


def f32_rows(oracle, seed, n):
    return np.concatenate([oracle.np_synth_rows_f32(seed, i, min(20_000, n - i)) for i in range(0, n, 20_000)])


def perm_labels(oracle, n, salt, base=1):
    return (np.argsort(oracle.np_mix64(np.arange(n, dtype=np.uint64) + np.uint64(salt)), kind="stable") + base).astype(np.uint64)


def reference(oracle, kind, stored, labels, qs, depth=KREF):
    """The oracle's top-`depth` of every query over the stored rows -> (labels, distances, counts)."""
    nq = len(qs)
    n = len(stored[0]) if kind == "i8" else len(stored)
    wl = np.zeros((nq, depth), dtype=np.uint64)
    wd = np.zeros((nq, depth), dtype=np.float32)
    wc = np.zeros(nq, dtype=np.int64)
    if n == 0:
        return wl, wd, wc
    if kind == "f16":
        l, d, c, certified = oracle.cpu_scan_f16(stored, labels, qs, depth)
        if certified:
            return l, d, c
        one = lambda q: oracle.search_f16(stored, labels, q, depth)  # noqa: E731
    elif kind == "i8":
        one = lambda q: oracle.search_i8(stored[0], stored[1], labels, q, depth)  # noqa: E731
    else:
        one = lambda q: oracle.search_f32(stored, labels, q, depth)  # noqa: E731
    for i, (l, d) in enumerate(pool_map(one, qs)):
        wc[i] = len(l)
        wl[i, :len(l)], wd[i, :len(l)] = l, d
    return wl, wd, wc


def store(oracle, kind, rows):
    return oracle.store_f16(rows) if kind == "f16" else oracle.store_i8(rows) if kind == "i8" else np.ascontiguousarray(rows)


def take(kind, stored, idx):
    return (stored[0][idx], stored[1][idx]) if kind == "i8" else stored[idx]


def check_answer(got, want, k, what, limit=None):
    """got = (labels, distances, counts) of the batch; want = a top-KREF reference; limit: only hits with d < limit."""
    gl, gd, gc = got
    wl, wd, wc = want
    for i in range(len(gc)):
        keep = int(min(wc[i], k))
        if limit is not None and not np.isnan(limit):
            keep = int((wd[i, :keep] < np.float32(limit)).sum())
        assert gc[i] == keep, (what, limit, i, int(gc[i]), keep)
        assert (gl[i, :keep] == wl[i, :keep]).all(), (what, limit, i, gl[i, :keep][:8], wl[i, :keep][:8])
        assert (bits(gd[i, :keep]) == bits(wd[i, :keep])).all(), (what, limit, i)


# ---------------------------------------------------------------------------------------------------- the re-run model
def choose_kprime(k):
    """dawn_index.cu:choose_kprime"""
    want, kp = k + max(k // 8, 4), 16
    while kp < want:
        kp *= 2
    return min(kp, 128)


def path_kprime(path, k):
    return max(64, choose_kprime(k)) if path in ("k2f32", "k3f32", "k4b") else choose_kprime(k)


def i8_split(qs):
    """s1 hi + s2 lo of prep_queries_i8_kernel, in f64."""
    x = np.ascontiguousarray(qs, dtype=np.float32)
    amax = np.abs(x).max(axis=1)
    s1 = np.where(amax > 0, amax / np.float32(127), np.float32(1)).astype(np.float32)[:, None]
    hi = np.clip(np.rint(x / s1), -127, 127)
    r = (x.astype(np.float64) - s1.astype(np.float64) * hi).astype(np.float32)
    rmax = np.abs(r).max(axis=1)
    s2 = np.where(rmax > 0, rmax / np.float32(127), np.float32(1)).astype(np.float32)[:, None]
    lo = np.clip(np.rint(r / s2), -127, 127)
    return s1.astype(np.float64) * hi + s2.astype(np.float64) * lo


def k3_eps(qs, slack):
    x = np.ascontiguousarray(qs, dtype=np.float32)
    d = x.astype(np.float64) - x.astype(np.float16).astype(np.float64)
    return np.sqrt((d * d).sum(axis=1)) * 1.02 + slack


def path_eps(path, qs):
    n = len(qs)
    if path == "k2":
        return np.full(n, SCAN_EPS)
    if path == "k2f32":
        return np.full(n, SCAN_EPS + F32_STORE_SLACK)
    if path == "k3":
        return k3_eps(qs, GEMM_ACCUM_SLACK)
    if path == "k4":
        e = np.ascontiguousarray(qs, dtype=np.float64) - i8_split(qs)
        return np.sqrt((e * e).sum(axis=1)) * 1.03 + 3.0e-5
    if path == "k4b":
        return k3_eps(qs, GEMM_ACCUM_SLACK + I8_DEQUANT_SLACK)
    return np.full(n, LOOSE_EPS)


def selection_top(path, kind, rows, stored, qs, want):
    """The KREF best selection scores the path ranks, descending, in f64; None for the paths held to the near-tie bound."""
    if path == "k2" and kind == "f16":
        return np.where(np.arange(KREF)[None, :] < want[2][:, None], 1.0 - want[1].astype(np.float64), -np.inf)
    if path == "k3":
        x, q = np.asarray(stored, dtype=np.float64), np.asarray(qs, dtype=np.float32).astype(np.float16).astype(np.float64)
    elif path == "k2f32":
        x, q = rows.astype(np.float16).astype(np.float64), np.asarray(qs, dtype=np.float64)
    elif path == "k4":
        x, q = stored[0].astype(np.float64) * stored[1][:, None].astype(np.float64), i8_split(qs)
    elif path == "k4b":
        x = (stored[0].astype(np.float32) * stored[1][:, None]).astype(np.float32).astype(np.float16).astype(np.float64)
        q = np.asarray(qs, dtype=np.float32).astype(np.float16).astype(np.float64)
    else:
        return None
    top = np.full((len(qs), KREF), -np.inf)
    for r0 in range(0, len(x), 25_000):
        s = np.concatenate([top, q @ x[r0:r0 + 25_000].T], axis=1)
        keep = min(KREF, s.shape[1])
        top[:, :keep] = -np.sort(-np.partition(s, s.shape[1] - keep, axis=1)[:, s.shape[1] - keep:], axis=1)
    return top


class Shard:
    """One shard's rows (indices into the corpus), its oracle top-KREF and the selection scores of the paths it may take."""

    def __init__(self, oracle, kind, rows, stored, labels, qs, idx):
        self.n = len(idx)
        self.kind, self.qs = kind, qs
        self.stored = take(kind, stored, idx)
        self.labels = labels[idx]
        self.rows = rows[idx] if rows is not None else None
        self.want = reference(oracle, kind, self.stored, self.labels, qs)
        self._sel = {}

    def sel(self, path):
        if path not in self._sel:
            self._sel[path] = selection_top(path, self.kind, self.rows, self.stored, self.qs, self.want) if self.n else None
        return self._sel[path]


def rerun_bounds(shards, paths, q_rows, k):
    """(must, may) re-runs of a batch (query indices q_rows) at k, summed over the shards; paths[g] is shard g's path."""
    lo = hi = 0
    for sh, path in zip(shards, paths):
        kp = path_kprime(path, k)
        if sh.n < kp:  # every row is a candidate: the certificate holds
            continue
        wd = sh.want[1][q_rows].astype(np.float64)
        eps = path_eps(path, sh.qs[q_rows])
        sel = sh.sel(path)
        if sel is None:  # near-tie bound only: the exact k-th and k'-th scores within 2 eps
            hi += int((wd[:, kp - 1] - wd[:, k - 1] <= 2.0 * eps + 1e-6).sum())
            continue
        margin = (1.0 - (sel[q_rows, kp - 1] + eps)) - wd[:, k - 1]
        lo += int((margin < -BAND).sum())
        hi += int((margin <= BAND).sum())
    return lo, hi


# ---------------------------------------------------------------------------------------------------- C. placement model
class Placement:
    """dawn_multi_reserve / dawn_multi_add_batch restated: which shard each added row lands on."""

    def __init__(self, G):
        self.G, self.cap, self.rows, self.cursor = G, [0] * G, [[] for _ in range(G)], 0

    def reserve(self, n):
        per = -(-n // self.G)
        self.cap = [max(c, per) for c in self.cap]

    def add_batch(self, idx):
        """Adds the rows idx in order; returns False where the C call fails for capacity (after the rows placed so far)."""
        done = 0
        while done < len(idx):
            for _ in range(self.G):
                g = self.cursor % self.G
                room = self.cap[g] - len(self.rows[g])
                if room > 0:
                    break
                self.cursor += 1
            else:
                return False
            n = min(BLOCK, len(idx) - done, room)
            self.rows[g].extend(int(i) for i in idx[done:done + n])
            done += n
            self.cursor += 1
        return True

    def add_synthetic(self, first, n):
        per = -(-n // self.G)
        for g in range(self.G):
            a = min(g * per, n)
            self.rows[g].extend(range(first + a, first + min(a + per, n)))

    def sizes(self):
        return [len(r) for r in self.rows]


def multi_search(m, qs, k, limit=None):
    """search through a MultiIndex; -> (answer, stats before, stats after)."""
    before = m.stats()
    got = m.search_batch(qs, k) if limit is None else m.search_batch_limit(qs, k, limit)
    return got, before, m.stats()


def check_stats(before, after, lo, hi, what, searches=1):
    assert after["peer_exchanges"] - before["peer_exchanges"] == searches, (what, before, after)
    assert after["nccl_exchanges"] == before["nccl_exchanges"], (what, after)
    reruns = after["exact_reruns"] - before["exact_reruns"]
    assert lo <= reruns <= hi, ("exact re-runs outside the model", what, f"{lo}..{hi}", reruns)
    return reruns


# ---------------------------------------------------------------------------------------------------- C. the G sweep
@pytest.fixture(scope="module")
def sweep(dawn, oracle):
    """G -> (MultiIndex over the add_synthetic corpus, its shards); plus the queries and the whole-corpus reference."""
    stored = oracle.synth_rows_f16(SEED, 0, N_SWEEP)
    labels = np.arange(1, N_SWEEP + 1, dtype=np.uint64)
    qs = oracle.make_queries(SEED, 1, max(SWEEP_BATCHES), N_SWEEP)
    want = reference(oracle, "f16", stored, labels, qs)
    handles = {}

    def get(G):
        if G not in handles:
            m = dawn.MultiIndex([0] * G)
            m.reserve(N_SWEEP)
            m.add_synthetic(SEED, 0, N_SWEEP)
            pl = Placement(G)
            pl.add_synthetic(0, N_SWEEP)
            assert m.size() == N_SWEEP and m.shards() == G
            shards = [Shard(oracle, "f16", None, stored, labels, qs, np.array(r, dtype=np.int64)) for r in pl.rows]
            handles[G] = (m, shards)
        return handles[G]

    yield get, qs, want
    for m, _ in handles.values():
        m.close()


def f16_route(n, batch, force=0):
    """The path an fp16 shard of n rows takes for a batch under the default options (dawn_index.cu:search_enqueue)."""
    if force == 1 or n < 1024:
        return "k2"
    return "k3" if force == 2 or (batch >= 16 and n >= 65536) or (batch >= 2 and n >= 2_000_000) else "k2"


SWEEP_CASES = [pytest.param(G, b, k, id=f"G{G}-b{b}-k{k}") for G in SWEEP_G for b in SWEEP_BATCHES
               for k in sorted({kk for kk in KS if G * kk <= 1024} | {min(KMAX, 1024 // G)})]


@pytest.mark.gpu
@pytest.mark.parametrize("G,batch,k", SWEEP_CASES)
def test_shard_count_and_k(sweep, G, batch, k):
    get, qs, want = sweep
    m, shards = get(G)
    r = np.arange(batch)
    got, before, after = multi_search(m, qs[:batch], k)
    check_answer(got, tuple(w[r] for w in want), k, (G, batch, k))
    lo, hi = rerun_bounds(shards, [f16_route(s.n, batch) for s in shards], r, k)
    reruns = check_stats(before, after, lo, hi, (G, batch, k))
    if reruns or hi:
        print(f"\n  G{G} b{batch} k{k}: exact_reruns {reruns}, model {lo}..{hi}")


@pytest.mark.gpu
@pytest.mark.parametrize("G,k", [(9, 114), (16, 65), (2, 121)])
def test_k_past_the_merge_width_is_rejected(dawn, sweep, G, k):
    """shards x k > 1024 (or k > DAWN_MAX_K) is a bad argument; the handle answers the next call."""
    get, qs, want = sweep
    m, _ = get(G)
    before = m.stats()
    with pytest.raises(dawn.DawnError) as e:
        m.search_batch(qs[:3], k)
    assert e.value.code == INVALID, str(e.value)
    kk = min(KMAX, 1024 // G)
    got, _, after = multi_search(m, qs[:3], kk)
    check_answer(got, tuple(w[:3] for w in want), kk, (G, k, "after the rejected call"))
    assert after["searches"] == before["searches"] + 1


@pytest.mark.gpu
def test_k0_and_batch0_return_ok(sweep):
    get, qs, want = sweep
    m, _ = get(3)
    before = m.stats()
    gl, gd, gc = m.search_batch(qs[:4], 0)
    assert (gc == 0).all() and len(gc) == 4
    gl, gd, gc = m.search_batch(np.zeros((0, 384), dtype=np.float32), 10)
    assert len(gc) == 0
    assert m.stats()["peer_exchanges"] == before["peer_exchanges"]


# ---------------------------------------------------------------------------------------------------- C. placement
def place_pool(oracle, n):
    rows = f32_rows(oracle, PLACE_SEED, n)
    return rows, perm_labels(oracle, n, salt=5)


PLACEMENTS = {
    # name: (G, [ops]); op = ("reserve", n) | ("batch", first, n) | ("single", first, n) | ("synthetic", n)
    "G3-reserve-cuts-blocks": (3, [("reserve", 10_000), ("batch", 0, 10_000), ("batch", 10_000, 3)]),
    "G2-cursor-carries": (2, [("reserve", 20_000), ("batch", 0, 5_000), ("single", 5_000, 5), ("batch", 5_005, 9_000),
                              ("single", 14_005, 3), ("batch", 14_008, 5_992), ("single", 20_000, 1)]),
    "G8-below-one-block": (8, [("reserve", 8 * BLOCK), ("batch", 0, 3_000)]),
    "G3-singles-skip-full": (3, [("reserve", 7), ("single", 0, 7), ("reserve", 12), ("batch", 7, 5), ("single", 12, 1)]),
    "G16-synthetic-below-G": (16, [("reserve", 16), ("synthetic", 5)]),
    "G9-synthetic-short-last": (9, [("reserve", 20_000), ("synthetic", 20_000)]),
}
PLACE_POOL = 20_001


@pytest.fixture(scope="module")
def place_data(oracle):
    rows, labels = place_pool(oracle, PLACE_POOL)
    qs = np.concatenate([oracle.make_queries(PLACE_SEED, 3, 6, PLACE_POOL), rows[[0, 4_095, 4_096, 9_999]]])
    return rows, labels, qs


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PLACEMENTS))
def test_placement(dawn, oracle, place_data, name):
    """size() after every step, capacity errors exactly where the model runs out of room, and answers equal to the oracle
    over the rows the model placed; then a duplicate of a row sent to its own shard or to another by the next add."""
    G, ops = PLACEMENTS[name]
    rows, labels, qs = place_data
    syn = {}
    with dawn.MultiIndex([0] * G) as m:
        pl = Placement(G)
        for op in ops:
            if op[0] == "reserve":
                m.reserve(op[1])
                pl.reserve(op[1])
            elif op[0] == "synthetic":
                m.add_synthetic(PLACE_SEED, 0, op[1])
                pl.add_synthetic(0, op[1])
                syn = {"n": op[1]}
            else:
                _, first, n = op
                if op[0] == "batch":
                    calls = [(pl.add_batch(np.arange(first, first + n)),
                              lambda: m.add_batch(labels[first:first + n], rows[first:first + n]))]
                else:  # one add per row: the model places each before the call is made
                    calls = [(pl.add_batch(np.array([i])), lambda i=i: m.add(int(labels[i]), rows[i]))
                             for i in range(first, first + n)]
                for fits, call in calls:
                    if fits:
                        call()
                    else:
                        with pytest.raises(dawn.DawnError) as e:
                            call()
                        assert e.value.code == CAPACITY, str(e.value)
            assert m.size() == sum(pl.sizes()), (name, op, m.size(), pl.sizes())
        if syn:
            src_rows = f32_rows(oracle, PLACE_SEED, syn["n"])  # add_synthetic's rows; labels first_row + i + 1
            src_labels = np.arange(1, syn["n"] + 1, dtype=np.uint64)
            src_stored = oracle.synth_rows_f16(PLACE_SEED, 0, syn["n"])
            q = np.concatenate([qs[:6], src_rows[:1]])
        else:
            src_rows, src_labels, src_stored, q = rows, labels, None, qs
        stored = src_stored if src_stored is not None else oracle.store_f16(src_rows)
        sizes = pl.sizes()
        placed = np.array(sorted(i for r in pl.rows for i in r), dtype=np.int64)
        want = reference(oracle, "f16", stored[placed], src_labels[placed], q)
        shards = [Shard(oracle, "f16", None, stored, src_labels, q, np.array(r, dtype=np.int64)) for r in pl.rows]
        for k in sorted({1, 10, min(KMAX, 1024 // G)}):
            got, before, after = multi_search(m, q, k)
            check_answer(got, want, k, (name, sizes, k))
            lo, hi = rerun_bounds(shards, [f16_route(s.n, len(q)) for s in shards], np.arange(len(q)), k)
            check_stats(before, after, lo, hi, (name, k))
        if syn or G < 2:
            return
        # duplicates: the next add_batch call goes to shard pl.cursor % G (skipping full shards); re-add a row of that shard
        # and a row of another one, and compare with merge_model over the shards' own oracle lists
        m.reserve(sum(pl.cap) + 2 * G)
        pl.reserve(sum(pl.cap) + 2 * G)
        target = next(g for g in [(pl.cursor + j) % G for j in range(G)] if pl.cap[g] > len(pl.rows[g]))
        other = next(g for g in range(G) if g != target and pl.rows[g])
        same_row, cross_row = pl.rows[target][0] if pl.rows[target] else None, pl.rows[other][-1]
        dup = [r for r in (same_row, cross_row) if r is not None]
        assert pl.add_batch(np.array(dup))
        assert all(r in pl.rows[target] for r in dup)
        m.add_batch(labels[dup], rows[dup])
        assert m.size() == sum(pl.sizes())
        qd = rows[dup]
        shards = [Shard(oracle, "f16", None, stored, labels, qd, np.array(r, dtype=np.int64)) for r in pl.rows]
        k = min(KMAX, 1024 // G)
        (gl, gd, gc), _, _ = multi_search(m, qd, k)
        for i, r in enumerate(dup):
            wl, wd = merge_model([(s.want[0][i], s.want[1][i]) for s in shards], [s.want[2][i] for s in shards], k)
            assert gc[i] == len(wl) and (gl[i, :gc[i]] == wl).all() and (bits(gd[i, :gc[i]]) == bits(wd)).all(), (name, r)
            copies = int((gl[i, :gc[i]] == labels[r]).sum())
            assert copies == (2 if r == same_row else 1), (name, "same shard" if r == same_row else "two shards", copies)


# ---------------------------------------------------------------------------------------------------- C. paths in one call
SPLITS = {
    # name: (storage, G, options, route(shard rows, batch, k) -> path)
    "f16-k3|k2": ("f16", 2, {}, lambda n, b, k: f16_route(n, b)),
    "shadow-k4d|k2": ("f16", 2, {"shadow_i8": 1},
                      lambda n, b, k: ("k4d" if not (b >= 128 and k > 32) else "k3") if b >= 16 and n >= 65536 else "k2"),
    "i8-k4c|k4": ("i8", 2, {}, lambda n, b, k: "k4c" if b >= 16 and n >= 65536 else "k4"),
    "i8-k4b|k4": ("i8", 2, {"i8_native": 0}, lambda n, b, k: "k4b" if b >= 16 and n >= 65536 and k <= 100 else "k4"),
    "f32-k3|k2": ("f32", 2, {}, lambda n, b, k: "k3f32" if b >= 16 and n >= 65536 else "k2f32"),
    "f16x3-tensor": ("f16", 3, {"force_path": 2}, lambda n, b, k: "k3"),
    "f16x2-tensor": ("f16", 2, {"force_path": 2}, lambda n, b, k: "k3"),
}
SPLIT_QUERIES = {"f16": 700, "i8": 33, "f32": 33}
KINDS = {"f16": "F16", "f32": "F32", "i8": "I8"}


@pytest.fixture(scope="module")
def split(dawn, oracle):
    """name -> (MultiIndex, Placement, shards, queries, whole-corpus reference) over the same N_SPLIT rows."""
    rows = f32_rows(oracle, SPLIT_SEED, N_SPLIT)
    labels = perm_labels(oracle, N_SPLIT, salt=13)
    cache, per_kind = {}, {}

    def get(name):
        if name in cache:
            return cache[name]
        kind, G, opts, route = SPLITS[name]
        if kind not in per_kind:
            qs = oracle.make_queries(SPLIT_SEED, 2, SPLIT_QUERIES[kind], N_SPLIT)
            stored = store(oracle, kind, rows)
            per_kind[kind] = (qs, stored, reference(oracle, kind, stored, labels, qs))
        qs, stored, want = per_kind[kind]
        m = dawn.MultiIndex([0] * G, quantization=getattr(dawn.ScalarKind, KINDS[kind]))
        pl = Placement(G)
        cap = 2 * 65_536 if G == 2 else N_SPLIT
        m.reserve(cap)
        pl.reserve(cap)
        m.add_batch(labels, rows)
        assert pl.add_batch(np.arange(N_SPLIT))
        assert m.size() == N_SPLIT
        if G == 2:
            assert pl.sizes() == [65_536, 61_440]
        for key, val in opts.items():
            m.set_option(key, val)
        shards = [Shard(oracle, kind, rows, stored, labels, qs, np.array(r, dtype=np.int64)) for r in pl.rows]
        cache[name] = (m, pl, shards, qs, want, (kind, opts, route, rows, labels))
        return cache[name]

    yield get
    for v in cache.values():
        v[0].close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["f16-k3|k2", "shadow-k4d|k2", "i8-k4c|k4", "i8-k4b|k4", "f32-k3|k2"])
def test_split_route_of_each_shard(dawn, split, name):
    """A standalone index holding a shard's rows takes the path the model names for it at batch 16 (and the scan below)."""
    m, pl, shards, qs, want, (kind, opts, route, rows, labels) = split(name)
    for g, r in enumerate(pl.rows):
        r = np.array(r, dtype=np.int64)
        with dawn.new_index(dawn.IndexOptions(quantization=getattr(dawn.ScalarKind, KINDS[kind]), capacity=len(r))) as idx:
            idx.add_batch(labels[r], rows[r])
            for key, val in opts.items():
                idx.set_option(key, val)
            for b in (15, 16):
                idx.profile(reset=True)
                idx.search_batch(qs[:b], 10)
                p = idx.profile(reset=True)
                path = route(len(r), b, 10)
                tensor = p["gemm_batches"] > 0 or p["shadow_batches"] > 0
                assert tensor == (path not in ("k2", "k4", "k2f32")), (name, g, b, path, p)
                assert (p["shadow_batches"] > 0) == (path == "k4d"), (name, g, b, path, p)


SPLIT_CASES = [pytest.param(name, b, k, id=f"{name}-b{b}-k{k}")
               for name in ("f16-k3|k2", "shadow-k4d|k2", "i8-k4c|k4", "i8-k4b|k4", "f32-k3|k2")
               for b in (1, 15, 16, 33) for k in (10, 29, 100, 120)
               if not (b in (1, 15) and k in (29, 100))]
SPLIT_CASES += [pytest.param(name, b, k, id=f"{name}-b{b}-k{k}") for name in ("f16x2-tensor", "f16x3-tensor")
                for b in (300, 700) for k in (10, 120)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,batch,k", SPLIT_CASES)
def test_split_paths_in_one_call(split, name, batch, k):
    """Shards on different paths in one call, and (force_path = 2, 2 or 3 query tiles) several tensor-core launches of the
    shards sharing one GPU: the chunk rendezvous times out, the answers stay exact."""
    m, pl, shards, qs, want, (kind, opts, route, rows, labels) = split(name)
    r = np.arange(batch)
    got, before, after = multi_search(m, qs[:batch], k)
    check_answer(got, tuple(w[r] for w in want), k, (name, batch, k))
    paths = [route(s.n, batch, k) for s in shards]
    lo, hi = rerun_bounds(shards, paths, r, k)
    reruns = check_stats(before, after, lo, hi, (name, batch, k, paths))
    if reruns or hi:
        print(f"\n  {name} b{batch} k{k} {paths}: exact_reruns {reruns}, model {lo}..{hi}")


def limit_values(want, k):
    wd = want[1]
    limits = [-np.inf, np.inf, np.nan]
    for i in range(min(2, len(wd))):
        for j in (0, k // 2, k - 1):
            d = np.float32(wd[i, j])
            limits += [d, np.nextafter(d, np.float32(-np.inf)), np.nextafter(d, np.float32(np.inf))]
    return limits


@pytest.mark.gpu
@pytest.mark.parametrize("name,batch,k", [pytest.param(n, b, k, id=f"{n}-b{b}-k{k}") for n in ("f16-k3|k2", "i8-k4c|k4")
                                          for b, k in ((1, 10), (7, 120), (33, 10), (33, 120))])
def test_split_distance_limit_edges(split, name, batch, k):
    """The limit is an emitted distance, one ulp either side of it, -inf, +inf or NaN (none): exactly the oracle's hits
    with d < L."""
    m, pl, shards, qs, want, _ = split(name)
    w = tuple(x[:batch] for x in want)
    for lim in limit_values(w, k):
        got, _, after = multi_search(m, qs[:batch], k, limit=float(lim))
        check_answer(got, w, k, (name, batch, k), limit=float(lim))


# ---------------------------------------------------------------------------------------------------- D. tied shards
N_TIE, N_TIE_RANDOM = 3_000, 5_000


@pytest.fixture(scope="module")
def tied(dawn, oracle):
    base = oracle.np_synth_rows_f32(TIE_SEED, 0, 1)
    rows = np.concatenate([np.repeat(base, N_TIE, axis=0), oracle.np_synth_rows_f32(TIE_SEED + 1, 0, N_TIE_RANDOM)])
    n = len(rows)
    order = perm_labels(oracle, n, salt=17, base=0).astype(np.int64)
    rows = np.ascontiguousarray(rows[order])
    labels = perm_labels(oracle, n, salt=19)
    qs = np.concatenate([base, oracle.make_queries(TIE_SEED + 1, 4, 23, N_TIE_RANDOM)])
    stored = oracle.store_f16(rows)
    want = reference(oracle, "f16", stored, labels, qs)
    tie = np.zeros(n, dtype=bool)
    tie[np.flatnonzero(order < N_TIE)] = True
    return rows, labels, qs, stored, want, tie


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3])
def test_tied_shards_rerun_and_stay_exact(dawn, oracle, tied, G):
    """Every shard holding a run of k' or more ties re-runs the tied query exactly; the merged answer stays the oracle's,
    with and without a distance limit, on the scan and on the tensor-core path."""
    rows, labels, qs, stored, want, tie = tied
    n = len(rows)
    with dawn.MultiIndex([0] * G) as m:
        m.reserve(n)
        pl = Placement(G)
        pl.reserve(n)
        m.add_batch(labels, rows)
        assert pl.add_batch(np.arange(n))
        shards = [Shard(oracle, "f16", None, stored, labels, qs, np.array(r, dtype=np.int64)) for r in pl.rows]
        tied_rows = [int(tie[r].sum()) for r in pl.rows]
        d_tie = np.float32(want[1][0, 0])
        for force in (0, 2):
            m.set_option("force_path", force)
            for batch, k in ((1, 10), (24, 20), (24, 100)):
                r = np.arange(batch)
                what = (G, force, batch, k)
                got, before, after = multi_search(m, qs[:batch], k)
                check_answer(got, tuple(w[r] for w in want), k, what)
                lo, hi = rerun_bounds(shards, [f16_route(s.n, batch, force) for s in shards], r, k)
                reruns = check_stats(before, after, lo, hi, what)
                holding = sum(t >= choose_kprime(k) for t in tied_rows)
                assert reruns >= holding, (what, "a shard full of ties did not re-run", tied_rows, reruns)
                assert (got[0][0, :k] == want[0][0, :k]).all() and (bits(got[1][0, :k]) == bits(d_tie)).all()
                for lim in (d_tie, np.nextafter(d_tie, np.float32(np.inf)), 0.9):
                    got, before, after = multi_search(m, qs[:batch], k, limit=float(lim))
                    check_answer(got, tuple(w[r] for w in want), k, what, limit=float(lim))
        m.set_option("force_path", 0)


# ---------------------------------------------------------------------------------------------------- D. a wrong first pass
# An f32 index selects its candidates on fp16 copies.  HIDDEN rows are one vector plus f32 perturbations below half an
# fp16 ulp: their copies are identical, so the selection ties them all, while their exact f32 distances differ.  They are
# stored worst first, with labels rising in that order, so whatever tie-break the selection uses keeps the wrong k' of
# them: at k' = 64 (k <= 57) the first pass answers wrongly and cannot certify, and the re-run at k' = 128, which holds
# all 100 of them, gives the oracle's answer.  More tied copies than 128 cannot be repaired by a re-run: the host API then
# reports the query uncertified (test_hidden_corpus_past_the_deepest_list_is_reported).
N_HIDDEN, N_HIDDEN_RANDOM = 100, 4_000
HIDDEN_KS = [10, 57]


def hidden_corpus(oracle, seed, n_hidden=N_HIDDEN):
    """(rows, labels, the query) of the wrong-first-pass corpus: n_hidden rows first, worst first, then random rows."""
    base = oracle.np_synth_rows_f32(seed, 0, 1)[0]
    b16 = base.astype(np.float16)
    step = np.spacing(np.abs(b16)).astype(np.float32)  # fp16 ulp above |b16|; the one below is at least half of it
    rng = np.random.default_rng(seed)
    hid = (b16.astype(np.float32)[None, :] + rng.uniform(-0.2, 0.2, (n_hidden, 384)).astype(np.float32) * step).astype(np.float32)
    q = base.astype(np.float32)
    hid = hid[np.argsort(hid.astype(np.float64) @ q.astype(np.float64), kind="stable")]  # lowest score (worst) first
    rows = np.ascontiguousarray(np.concatenate([hid, oracle.np_synth_rows_f32(seed + 1, 0, N_HIDDEN_RANDOM)]))
    labels = np.arange(1, len(rows) + 1, dtype=np.uint64)
    return rows, labels, q


@pytest.fixture(scope="module")
def hidden(oracle):
    rows, labels, q = hidden_corpus(oracle, TIE_SEED + 7)
    copies = oracle.store_f16(rows[:N_HIDDEN]).view(np.uint16)
    assert (copies == copies[:1]).all(), "the hidden rows' fp16 copies differ"
    qs = np.concatenate([q[None, :], oracle.make_queries(TIE_SEED + 8, 9, 15, N_HIDDEN_RANDOM)])
    want = reference(oracle, "f32", rows, labels, qs)
    assert len(set(bits(want[1][0, :N_HIDDEN]).tolist())) > 10  # the hidden rows' exact distances differ
    return rows, labels, qs, want


@pytest.mark.gpu
@pytest.mark.parametrize("force", [1, 2], ids=["k2f32", "k3f32"])
def test_hidden_corpus_first_pass_is_wrong(dawn, hidden, force):
    """The premise of the re-run cases below: without its re-run an f32 index answers the hidden query wrongly and flags
    it uncertified (search_device cannot re-run); the host API, which re-runs, answers it exactly."""
    import torch

    rows, labels, qs, want = hidden
    with dawn.new_index(dawn.IndexOptions(quantization=dawn.ScalarKind.F32, capacity=len(rows))) as idx:
        idx.add_batch(labels, rows)
        idx.set_option("force_path", force)
        for k in HIDDEN_KS:
            b = 2
            dq = torch.from_numpy(np.ascontiguousarray(qs[:b])).cuda()
            ol = torch.zeros((b, k), dtype=torch.int64, device="cuda")
            od = torch.zeros((b, k), dtype=torch.float32, device="cuda")
            oc = torch.zeros(b, dtype=torch.int32, device="cuda")
            of = torch.zeros(b, dtype=torch.int32, device="cuda")
            idx.search_device(dq.data_ptr(), b, k, ol.data_ptr(), od.data_ptr(), oc.data_ptr(), of.data_ptr(),
                              torch.cuda.current_stream().cuda_stream or 1)
            torch.cuda.synchronize()
            assert int(of.cpu()[0]) & 1 == 0, (force, k, "the hidden query was certified")
            first = ol.cpu().numpy().view(np.uint64)[0]
            assert not (first == want[0][0, :k]).all(), (force, k, "the first pass was already right")
            check_answer(idx.search_batch(qs[:b], k), tuple(w[:b] for w in want), k, (force, k, "host API"))


@pytest.mark.gpu
def test_hidden_corpus_past_the_deepest_list_is_reported(dawn, oracle):
    """With more tied fp16 copies than the deepest candidate list (k' = 128) the re-run selects on the same copies and
    cannot repair the answer; the host API must then count the query as uncertified rather than pass it as exact."""
    rows, labels, q = hidden_corpus(oracle, TIE_SEED + 9, n_hidden=1_500)
    with dawn.new_index(dawn.IndexOptions(quantization=dawn.ScalarKind.F32, capacity=len(rows))) as idx:
        idx.add_batch(labels, rows)
        for force in (1, 2):
            idx.set_option("force_path", force)
            idx.profile(reset=True)
            idx.search_batch(q[None, :], KMAX)
            p = idx.profile(reset=True)
            # k' = 128 already: the scan has nothing deeper to run; K3 re-runs on the scan, which ties the copies the same way
            assert p["escalations"] == (force == 2) and p["uncertified"] == 1, (force, p)
            idx.search_batch(q[None, :], 10)
            p = idx.profile(reset=True)
            assert p["escalations"] == 1 and p["uncertified"] == 1, (force, p)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3])
def test_rerun_repairs_a_wrong_first_pass(dawn, hidden, G):
    """dawn_multi on the hidden corpus: the shard holding the hidden rows must re-run the query and patch labels,
    distances and counts into its block before the merge; the merged answer is the oracle's, with and without a limit."""
    rows, labels, qs, want = hidden
    with dawn.MultiIndex([0] * G, quantization=dawn.ScalarKind.F32) as m:
        m.reserve(len(rows))
        m.add_batch(labels, rows)
        for force in (1, 2):
            m.set_option("force_path", force)
            for batch, k in ((1, 10), (16, 10), (16, 57)):
                what = (G, force, batch, k)
                w = tuple(x[:batch] for x in want)
                got, before, after = multi_search(m, qs[:batch], k)
                check_answer(got, w, k, what)
                assert after["exact_reruns"] - before["exact_reruns"] >= 1, (what, "the hidden query was not re-run")
                lim = float(w[1][0, k // 2])
                got, _, _ = multi_search(m, qs[:batch], k, limit=lim)
                check_answer(got, w, k, what, limit=lim)


# ---------------------------------------------------------------------------------------------------- E. sharded.py
SHARD_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["DAWN_ROOT"])
import numpy as np, torch, torch.distributed as dist
from dawnsearch_b200.sharded import ResultBlock, ShardedIndex, shard_range
from oracle import oracle as O
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["DAWN_TEST_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) if backend == "nccl" else 0
if backend == "nccl":
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
else:
    dist.init_process_group("gloo")
torch.cuda.set_device(local)
SEED = 0x3A17ED64
ok = True

def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)

def report(what, got, want, k, limit=None):
    global ok
    gl, gd, gc = got
    wl, wd, wc = want
    same = True
    for i in range(len(gc)):
        keep = int(min(wc[i], k))
        if limit is not None:
            keep = int((wd[i, :keep] < np.float32(limit)).sum())
        same &= bool(gc[i] == keep and (gl[i, :keep] == wl[i, :keep]).all() and (bits(gd[i, :keep]) == bits(wd[i, :keep])).all())
    if rank == 0:
        print(what, "ok" if same else "MISMATCH", flush=True)
    ok &= same

def reruns_per_rank(sh):
    mine = torch.tensor([sh.last_search_escalated], dtype=torch.int64)
    if backend == "nccl":
        mine = mine.cuda()
    got = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(got, mine)
    return [int(t.item()) for t in got]

def check_reruns(what, per_rank, others_too):
    global ok
    if rank == 0:
        good = per_rank[0] >= 1 and (others_too or all(e == 0 for e in per_rank[1:]))
        print(f"{what} re-runs {per_rank}", "ok" if good else "MISMATCH", flush=True)
        ok &= good

def reference(stored, labels, qs, k):
    l, d, c, cert = O.cpu_scan_f16(stored, labels, qs, k)
    if cert:
        return l, d, c
    l = np.zeros((len(qs), k), dtype=np.uint64); d = np.zeros((len(qs), k), dtype=np.float32); c = np.zeros(len(qs), dtype=np.int64)
    for i, q in enumerate(qs):
        a, b = O.search_f16(stored, labels, q, k)
        l[i, :len(a)], d[i, :len(a)], c[i] = a, b, len(a)
    return l, d, c

# small corpora: the last rank empty (per * (world - 1) >= rows), and ranks with fewer than k rows
for rows in (world - 1, 2 * world - 2, 7):
    first, n = shard_range(rank, world, rows)
    sh = ShardedIndex(local, n)
    if n:
        sh.index.add_synthetic(SEED, first, n)
    stored = O.synth_rows_f16(SEED, 0, rows)
    qs = O.make_queries(SEED, 3, 5, max(rows, 1))
    for k in (1, 10):
        report(f"rows {rows} k {k}", sh.search(qs, k), reference(stored, None, qs, k), k)
    sh.close()
# a synthetic corpus: k up to the widest merge of the world, limits, and the pipelined path
rows = 150_001
first, n = shard_range(rank, world, rows)
sh = ShardedIndex(local, n)
sh.index.add_synthetic(SEED, first, n)
stored = O.synth_rows_f16(SEED, 0, rows)
for batch, k in ((1, 120), (33, 120), (33, 57), (300, 10)):
    qs = O.make_queries(SEED, 10 + batch, batch, rows)
    want = reference(stored, None, qs, k)
    report(f"synthetic batch {batch} k {k}", sh.search(qs, k), want, k)
    if batch == 33:
        for lim in (float(want[1][0, k // 2]), float(np.nextafter(want[1][0, k // 2], np.float32(np.inf))), float("-inf"), float("inf")):
            report(f"limit {lim} batch {batch} k {k}", sh.search(qs, k, distance_limit=lim), want, k, limit=lim)
qsets = [O.make_queries(SEED, 40 + i, 32, rows) for i in range(5)]
dq = [torch.from_numpy(q).cuda() for q in qsets]
outs = []
for i in range(5):
    blk = sh.search_device(dq[i], 20, pipelined=True)
    sh.wait_results()
    outs.append(blk.clone())
torch.cuda.synchronize()
rb = ResultBlock(32, 20)
for i in range(5):
    L, D, Cn = rb.views(outs[i].cpu())
    got = (L.numpy().astype(np.uint64), D.numpy(), Cn.numpy().astype(np.int64))
    report(f"pipelined step {i}", got, reference(stored, None, qsets[i], 20), 20)
sh.close()
# ties on rank 0's rows only: rank 0 re-runs, the others do not, and the second exchange carries the patch
base = O.np_synth_rows_f32(SEED + 1, 0, 1)
rows_t = np.concatenate([np.repeat(base, 2_000, axis=0), O.np_synth_rows_f32(SEED + 2, 0, 4_000 * world)])
labels = O.np_mix64(np.arange(len(rows_t), dtype=np.uint64) + np.uint64(23)) >> np.uint64(8)
first, n = shard_range(rank, world, len(rows_t))
sh = ShardedIndex(local, n)
sh.index.add_batch(labels[first:first + n], rows_t[first:first + n])
stored = O.store_f16(rows_t)
qs = np.concatenate([base, O.make_queries(SEED + 2, 5, 15, 4_000)])
for k in (10, 100):
    want = reference(stored, labels, qs, k)
    report(f"tied k {k}", sh.search(qs, k), want, k)
    check_reruns(f"tied k {k}", reruns_per_rank(sh), others_too=False)
    lim = float(np.nextafter(want[1][0, 0], np.float32(np.inf)))
    report(f"tied limit k {k}", sh.search(qs, k, distance_limit=lim), want, k, limit=lim)
sh.close()
# a wrong first pass on rank 0 (test_rerun_repairs_a_wrong_first_pass): 100 f32 rows whose fp16 copies are one vector, stored
# worst first, so the selection keeps the wrong candidates; only the re-run and the second exchange give the oracle's answer
from dawnsearch_b200.index import ScalarKind
base = O.np_synth_rows_f32(SEED + 3, 0, 1)[0]
b16 = base.astype(np.float16)
step = np.spacing(np.abs(b16)).astype(np.float32)
rng = np.random.default_rng(SEED + 3)
hid = (b16.astype(np.float32)[None, :] + rng.uniform(-0.2, 0.2, (100, 384)).astype(np.float32) * step).astype(np.float32)
hid = hid[np.argsort(hid.astype(np.float64) @ base.astype(np.float64), kind="stable")]
rows_h = np.ascontiguousarray(np.concatenate([hid, O.np_synth_rows_f32(SEED + 4, 0, 3_000 * world)]))
labels_h = np.arange(1, len(rows_h) + 1, dtype=np.uint64)
first, n = shard_range(rank, world, len(rows_h))
sh = ShardedIndex(local, n, quantization=ScalarKind.F32)
sh.index.add_batch(labels_h[first:first + n], rows_h[first:first + n])
qs = np.concatenate([base[None, :], O.make_queries(SEED + 4, 6, 7, 3_000)])
for force in (1, 2):
    sh.index.set_option("force_path", force)
    for k in (10, 57):
        res = [O.search_f32(rows_h, labels_h, q, k) for q in qs]
        want = (np.array([r[0] for r in res]), np.array([r[1] for r in res]), np.array([len(r[0]) for r in res]))
        report(f"hidden force {force} k {k}", sh.search(qs, k), want, k)
        check_reruns(f"hidden force {force} k {k}", reruns_per_rank(sh), others_too=True)
sh.close()
flag = torch.tensor([1 if ok else 0])
if backend == "nccl":
    flag = flag.cuda()
dist.broadcast(flag, 0)
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
'''
# lines rank 0 prints per run: 3 small corpora x 2 k, 4 synthetic + 2 x 4 limits, 5 pipelined, 2 x 3 tied, 2 x 2 x 2 hidden
WORKER_LINES = 6 + 4 + 8 + 5 + 6 + 8


def run_shard_worker(tmp_path, backend, world, port):
    script = tmp_path / f"multi_edges_worker_{world}.py"
    script.write_text(SHARD_WORKER)
    env = dict(os.environ, DAWN_ROOT=ROOT, DAWN_TEST_BACKEND=backend)
    # a session of its own, so that on a timeout torchrun and every worker it started are killed together, well before
    # pytest's own timeout could end the test and leave them running
    p = subprocess.Popen([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                         env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = p.communicate(timeout=600)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        out, err = p.communicate()
        pytest.fail("the sharded worker timed out: " + out[-2000:] + err[-2000:])
    assert p.returncode == 0, out[-4000:] + err[-4000:]
    assert "MISMATCH" not in out, out
    assert out.count(" ok") == WORKER_LINES, out


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_worlds_on_one_gpu(tmp_path, world):
    """Every rank on GPU 0, the exchange staged through the host over gloo."""
    run_shard_worker(tmp_path, "gloo", world, 29641 + world)


@pytest.mark.gpu
def test_sharded_world_2_over_nccl(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    run_shard_worker(tmp_path, "nccl", 2, 29651)
