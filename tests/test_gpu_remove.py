"""dawn_index_remove_batch / dawn_multi_remove_batch: rows are compacted out of the device corpus, and every search path must
answer exactly what the oracle answers over the surviving rows -- bit for bit, for every storage layout."""
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 0x5EED0F1D
MAX_LABEL = 2**64 - 1


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def same(got, want):
    gl, gd, gc = got[:3]
    wl, wd, wc = want[:3]
    assert (gc == wc).all()
    for b in range(len(gc)):
        c = int(gc[b])
        assert (gl[b, :c] == wl[b, :c]).all(), b
        assert (bits(gd[b, :c]) == bits(wd[b, :c])).all(), b


def synth(oracle, seed, n):
    return np.concatenate([oracle.np_synth_rows_f32(seed, i, min(20000, n - i)) for i in range(0, n, 20000)])


def oracle_batch(fn, qs, k):
    """Per-query oracle over a thread pool (the C oracle drops the GIL) -> (labels[B,k], distances[B,k], counts[B])."""
    with ThreadPoolExecutor(16) as ex:
        res = list(ex.map(lambda q: fn(q, k), qs))
    lab = np.zeros((len(qs), k), dtype=np.uint64)
    dist = np.zeros((len(qs), k), dtype=np.float32)
    cnt = np.zeros(len(qs), dtype=np.int64)
    for i, (l, d) in enumerate(res):
        lab[i, :len(l)], dist[i, :len(d)], cnt[i] = l, d, len(l)
    return lab, dist, cnt


class Corpus:
    """Rows as the oracle sees them for one storage layout; `want(keep, qs, k)` answers over rows[keep] only."""

    def __init__(self, oracle, scalar, rows, labels):
        self.oracle, self.scalar, self.rows, self.labels = oracle, scalar, rows, labels
        if scalar == 0:
            self.f16 = oracle.store_f16(rows)
        elif scalar == 1:
            self.q8, self.sc = oracle.store_i8(rows)

    def want(self, keep, qs, k):
        O, lab = self.oracle, self.labels[keep]
        if self.scalar == 0:
            return O.cpu_scan_f16(self.f16[keep], lab, qs, k)[:3]
        if self.scalar == 1:
            q8, sc = np.ascontiguousarray(self.q8[keep]), np.ascontiguousarray(self.sc[keep])
            return oracle_batch(lambda q, kk: O.search_i8(q8, sc, lab, q, kk), qs, k)
        rows = np.ascontiguousarray(self.rows[keep])
        return oracle_batch(lambda q, kk: O.search_f32(rows, lab, q, kk), qs, k)


def labelled_corpus(oracle, n, seed):
    """Permuted labels, some owned by several rows (at the head, in the middle and in the tail)."""
    rows = synth(oracle, seed, n)
    labels = (np.argsort(oracle.np_mix64(np.arange(n, dtype=np.uint64) + np.uint64(seed)), kind="stable") + 1).astype(np.uint64)
    rng = np.random.default_rng(seed)
    for r in np.concatenate([[1, 2, n - 3, n - 1], rng.choice(np.arange(10, n - 10), 300, replace=False)]):
        labels[r] = labels[rng.integers(0, n)]
    return rows, labels


def removal_set(labels, rng):
    n = len(labels)
    counts = {}
    for l in labels.tolist():
        counts[l] = counts.get(l, 0) + 1
    multi = np.array([l for l, c in counts.items() if c > 1], dtype=np.uint64)
    req = np.concatenate([
        np.array([n + 1000, n + 2000, MAX_LABEL], dtype=np.uint64),  # absent (including the label ~0)
        labels[:5],                                                  # rows at the head
        labels[n - 257:],                                            # the whole tail
        multi[:40],                                                  # labels that own several rows
        labels[rng.choice(n, 3000, replace=False)],                  # anywhere, some already in the tail
    ])
    req = np.concatenate([req, req[::7]])                            # repeated in the request
    return rng.permutation(req)


LAYOUTS = {"f16": 0, "i8": 1, "f32": 2}


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_remove_every_layout_and_path(dawn, oracle, layout, tmp_path):
    scalar = LAYOUTS[layout]
    n = 200_000
    rows, labels = labelled_corpus(oracle, n, SEED + scalar)
    C = Corpus(oracle, scalar, rows, labels)
    rng = np.random.default_rng(7 + scalar)
    req = removal_set(labels, rng)
    keep = ~np.isin(labels, req)
    qs = np.concatenate([rows[[0, 3, n - 1, n - 300, 77_777]] + 0.01, oracle.make_queries(SEED, 5 + scalar, 1019, n)]).astype(np.float32)
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)

    def build():
        idx = dawn.new_index(dawn.IndexOptions(quantization=scalar, capacity=n))
        if scalar == 0:
            idx.set_option("shadow_i8", 1)
        idx.add_batch(labels, rows)
        return idx

    idx = build()
    uniq, cnt = np.unique(labels, return_counts=True)
    single = keep & np.isin(labels, uniq[cnt == 1])  # rows whose label owns no other row: get() must not change
    probe = np.concatenate([labels[single][:20], labels[n - 400:n - 257][single[n - 400:n - 257]][:20]])  # and moved tail rows
    before = {int(l): idx.get(int(l)) for l in probe}
    idx.search_batch(qs[:64], 10)  # builds the shadow before the removal (F16)
    removed = idx.remove_batch(req)
    assert removed == n - keep.sum() and idx.size() == keep.sum() and idx.capacity() == n
    assert idx.remove_batch(req) == 0
    for l in probe:
        assert (idx.get(int(l)) == before[int(l)]).all()
    gone = set(req.tolist())
    for l in list(gone)[:10]:
        with pytest.raises(dawn.DawnError):
            idx.get(l)

    def paths():
        if scalar == 1:
            yield "native int8", {"i8_tensor_min_batch": 1}, "gemm"
            yield "int8 scan", {"i8_tensor_min_batch": 0}, "scan"
        else:
            yield "scan", {"force_path": 1, "shadow_i8": 0}, "scan"
            yield "fp16 tensor", {"force_path": 2, "shadow_i8": 0}, "gemm"
            if scalar == 0:
                yield "shadow", {"force_path": 0, "shadow_i8": 1, "shadow_single_rows": 0, "shadow_big_k_rows": 0}, "shadow"

    for k in (10, 100):
        want = C.want(keep, qs, k)
        for name, opts, kind in paths():
            for key, v in opts.items():
                idx.set_option(key, v)
            for b in (1, 64, 1024):
                if kind == "scan" and b == 1024 and k == 100:
                    continue  # 1024 single-query scan passes over the corpus add nothing the other batches do not cover
                idx.profile(reset=True)
                got = idx.search_batch(qs[:b], k)
                p = idx.profile(reset=True)
                assert p["uncertified"] == 0 and p["device_status"] == 0, (name, b, k, p)
                if kind == "shadow":
                    assert p["shadow_batches"] == 1 and p["escalations"] == 0, (name, b, k, p)
                if kind == "gemm":
                    assert p["gemm_batches"] >= 1, (name, b, k, p)
                same(got, tuple(a[:b] for a in want))
                assert not np.isin(got[0][:, :k][np.arange(k)[None, :] < got[2][:, None]], req).any()

    # persistence: the compacted corpus saves and loads; the same calls give byte-identical files
    path_a, path_b = str(tmp_path / "a.dawn"), str(tmp_path / "b.dawn")
    idx.save(path_a)
    twin = build()
    twin.search_batch(qs[:64], 10)
    assert twin.remove_batch(req) == removed
    twin.save(path_b)
    twin.close()
    assert open(path_a, "rb").read() == open(path_b, "rb").read()
    fresh = dawn.new_index(dawn.IndexOptions(quantization=scalar))
    fresh.load(path_a)
    assert fresh.size() == keep.sum()
    for k in (10, 100):
        same(fresh.search_batch(qs[:64], k), idx.search_batch(qs[:64], k))
    fresh.close()
    idx.close()


def shadow_index(dawn, n_cap):
    idx = dawn.new_index(dawn.IndexOptions(capacity=n_cap))
    idx.set_option("shadow_i8", 1)
    idx.set_option("shadow_single_rows", 0)
    idx.set_option("shadow_big_k_rows", 0)
    return idx


def search_shadow(idx, qs, k, shadow=True):
    idx.profile(reset=True)
    got = idx.search_batch(qs, k)
    p = idx.profile(reset=True)
    assert p["uncertified"] == 0 and p["shadow_batches"] == (1 if shadow else 0), p
    if shadow:
        assert p["escalations"] == 0 and p["device_uncertified"] == 0, p
    return got


def test_remove_moves_rows_the_shadow_has_not_quantised(dawn, oracle):
    n0, n1 = 100_000, 120_000
    rows = synth(oracle, SEED + 11, n1)
    labels = np.arange(n1, dtype=np.uint64) * 3 + 2
    stored = oracle.store_f16(rows)
    qs = oracle.make_queries(SEED + 11, 3, 256, n1)
    with shadow_index(dawn, n1 + 1000) as idx:
        idx.add_batch(labels[:n0], rows[:n0])
        search_shadow(idx, qs, 10)  # the shadow now covers [0, n0)
        idx.add_batch(labels[n0:n1], rows[n0:n1])  # not searched: the shadow lags
        req = labels[:2000:3]  # head rows, whose donors are the new rows
        assert idx.remove_batch(req) == len(req)
        keep = ~np.isin(labels, req)
        for k in (10, 50):
            same(search_shadow(idx, qs, k), oracle.cpu_scan_f16(stored[keep], labels[keep], qs, k))
        # a shadow left behind while the option is off: the remove drops it, the next search rebuilds it
        idx.set_option("shadow_i8", 0)
        extra = synth(oracle, SEED + 12, 1000)
        extra_labels = np.arange(1000, dtype=np.uint64) * 3 + 10**9
        idx.add_batch(extra_labels, extra)
        search_shadow(idx, qs, 10, shadow=False)
        req2 = labels[5000:7000:2]
        assert idx.remove_batch(req2) == len(req2)
        idx.set_option("shadow_i8", 1)
        keep &= ~np.isin(labels, req2)
        all_stored = np.concatenate([stored[keep], oracle.store_f16(extra)])
        all_labels = np.concatenate([labels[keep], extra_labels])
        same(search_shadow(idx, qs, 10), oracle.cpu_scan_f16(all_stored, all_labels, qs, 10))


def test_update_is_remove_then_add(dawn, oracle):
    n = 80_000
    rows = synth(oracle, SEED + 21, n)
    labels = np.arange(1, n + 1, dtype=np.uint64)
    with dawn.new_index(dawn.IndexOptions(capacity=n + 10)) as idx:
        idx.add_batch(labels, rows)
        target = 4242
        new_vec = rows[70_000] + 0.05 * rows[123]
        new_vec = (new_vec / np.linalg.norm(new_vec)).astype(np.float32)
        assert idx.remove(target) == 1
        idx.add(target, new_vec)
        assert idx.size() == n
        m = idx.search(new_vec, 20)
        assert (m.labels == target).sum() == 1
        stored = oracle.store_f16(np.concatenate([np.delete(rows, target - 1, axis=0), new_vec[None]]))
        lab = np.concatenate([np.delete(labels, target - 1), [target]]).astype(np.uint64)
        wl, wd = oracle.search_f16(stored, lab, new_vec, 20)
        assert (m.labels == wl).all() and (bits(m.distances) == bits(wd)).all()
        assert (idx.get(target) == oracle.store_f16(new_vec[None])[0].astype(np.float32)).all()


def test_remove_covers_staged_adds_and_empties_the_index(dawn, oracle):
    n = 5_000
    rows = synth(oracle, SEED + 31, n + 1)
    labels = np.arange(10, n + 10, dtype=np.uint64)
    with dawn.new_index(dawn.IndexOptions(capacity=2 * n)) as idx:
        idx.add_batch(labels, rows[:n])
        idx.search(rows[0], 5)
        idx.add(99_999, rows[n])  # staged, not yet on the device
        assert idx.size() == n + 1
        assert idx.remove(99_999) == 1 and idx.size() == n
        with pytest.raises(dawn.DawnError):
            idx.get(99_999)
        m = idx.search(rows[n], 10)
        assert 99_999 not in m.labels.tolist()
        # remove everything: nothing is left to find; then the index fills and searches exactly again
        assert idx.remove_batch(np.concatenate([labels, labels[:10]])) == n
        assert idx.size() == 0 and idx.capacity() == 2 * n
        gl, gd, cnt = idx.search_batch(rows[:8], 10)
        assert (cnt == 0).all()
        assert idx.remove_batch(labels) == 0
        idx.add_batch(labels[::-1].copy(), rows[:n])
        stored = oracle.store_f16(rows[:n])
        qs = oracle.make_queries(SEED + 31, 2, 16, n)
        same(idx.search_batch(qs, 10), oracle.cpu_scan_f16(stored, labels[::-1].copy(), qs, 10))


def test_remove_of_a_long_row_keeps_results_exact_and_verify_restores_the_shadow(dawn, oracle):
    n = 70_000
    rows = synth(oracle, SEED + 41, n)
    labels = np.arange(1, n + 1, dtype=np.uint64)
    stored = oracle.store_f16(rows)
    qs = oracle.make_queries(SEED + 41, 2, 64, n)
    want = oracle.cpu_scan_f16(stored, labels, qs, 10)
    with shadow_index(dawn, n + 1) as idx:
        idx.add_batch(labels, rows)
        same(search_shadow(idx, qs, 10), want)
        long_row = (rows[5] * 1.5).astype(np.float32)
        idx.add(n + 1, long_row)
        # a stored row longer than the norm gate widens every bound: exact, but not through the shadow
        long_stored = np.concatenate([stored, oracle.store_f16(long_row[None])])
        same(search_shadow(idx, qs, 10, shadow=False), oracle.cpu_scan_f16(long_stored, np.append(labels, n + 1), qs, 10))
        assert idx.remove(n + 1) == 1
        same(search_shadow(idx, qs, 10, shadow=False), want)  # the norm statistics still bound the removed row
        v = idx.verify()
        assert v["bad_rows"] == 0 and v["max_norm"] < 1.01
        same(search_shadow(idx, qs, 10), want)


def test_searches_during_removals_see_one_corpus_state(dawn, oracle):
    n = 100_000
    rows = synth(oracle, SEED + 51, n)
    labels = (np.argsort(oracle.np_mix64(np.arange(n, dtype=np.uint64) + np.uint64(51)), kind="stable") + 1).astype(np.uint64)
    stored = oracle.store_f16(rows)
    qs = oracle.make_queries(SEED + 51, 2, 64, n)
    rng = np.random.default_rng(51)
    batches = np.array_split(rng.permutation(labels)[:20_000], 10)
    keep = np.ones(n, dtype=bool)
    states = [oracle.cpu_scan_f16(stored, labels, qs, 10)]
    for b in batches:
        keep &= ~np.isin(labels, b)
        states.append(oracle.cpu_scan_f16(stored[keep], labels[keep], qs, 10))

    def state_of(got):
        for i, w in enumerate(states):
            if (got[2] == w[2]).all() and (got[0] == w[0]).all() and (bits(got[1]) == bits(w[1])).all():
                return i
        return -1

    with dawn.new_index(dawn.IndexOptions(capacity=n)) as idx:
        idx.add_batch(labels, rows)
        stop = threading.Event()
        seen, errors = [], []

        def searcher():
            try:
                while not stop.is_set():
                    seen.append(state_of(idx.search_batch(qs, 10)))
            except Exception as e:  # reported below
                errors.append(e)

        threads = [threading.Thread(target=searcher) for _ in range(4)]
        for t in threads:
            t.start()
        for b in batches:
            idx.remove_batch(b)
        stop.set()
        for t in threads:
            t.join()
        assert not errors, errors
        assert seen and -1 not in seen, seen
        assert state_of(idx.search_batch(qs, 10)) == 10


def test_multi_remove_over_two_shards(dawn, oracle):
    n = 120_000
    rows = synth(oracle, SEED + 61, n)
    labels = (np.arange(n, dtype=np.uint64) * 7 + 3)
    stored = oracle.store_f16(rows)
    qs = oracle.make_queries(SEED + 61, 2, 64, n)
    with dawn.MultiIndex([0, 0]) as m:
        m.reserve(n)
        m.add_batch(labels, rows)  # 4096-row blocks alternate between the shards
        req = np.concatenate([labels[::13], labels[:100], np.array([5, 6, MAX_LABEL], dtype=np.uint64)])
        keep = ~np.isin(labels, req)
        assert m.remove_batch(req) == n - keep.sum()
        assert m.size() == keep.sum()
        assert m.remove(int(labels[1])) == 0 and m.remove(int(labels[1 + 13 * 1000 + 1])) == 1
        keep[1 + 13 * 1000 + 1] = False
        for k in (10, 100):
            same(m.search_batch(qs, k), oracle.cpu_scan_f16(stored[keep], labels[keep], qs, k))
