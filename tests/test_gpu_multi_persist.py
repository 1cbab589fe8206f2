"""Persistence and read-back of the multi-shard handle: dawn_multi_save / _load / _get / _get_i24 / _verify / _search_i24.

A save writes one file: a 4096-byte header (magic DAWNMULT, version, scalar, dims, G, add cursor, rows[G]) and one
page-aligned section per shard (labels, then the stored rows as dawn_index_save writes them).  read_multi() below is a
reader of that layout written from include/dawn_index.h; every file a test writes goes through it, and it checks the
header fields, the section starts, the zero padding and the exact length.

Every handle lists device 0 G times, as test_gpu_multi_edges.py does, and its Placement model says which rows each shard
was given.  Answers are compared bit for bit (labels, distance bits, counts) with the CPU oracle over every stored row and
with the handle the file came from.
"""
import os
import threading

import numpy as np
import pytest

from test_gpu_multi_edges import Placement, check_answer, f32_rows, perm_labels, reference, store

INVALID, IO = -1, -4
KINDS = {"f16": "F16", "i8": "I8", "f32": "F32"}
SCALAR = {"f16": 0, "i8": 1, "f32": 2}
ROW_BYTES = {"f16": 768, "f32": 1536}
I8_BLOCK = 3104
PAGE = 4096
SEED = 0x3A17ED70
N_EDGE = 4 * 4096 + 1237    # shards end in partial 4096-row and 8-row blocks; with G = 8 four shards stay empty
N_BIG = 36 * 4096 + 1237    # G = 2: both shards >= 65,536 rows, so K4c, K4d and K3 run
FIRST_ADD = 10_000          # two add_batch calls: the cursor carries over
KS = [1, 20, 120]
NQ = 33


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------- the file layout
def payload_bytes(kind, rows):
    return -(-rows // 8) * I8_BLOCK if kind == "i8" else rows * ROW_BYTES[kind]


def read_multi(path, kind):
    """Parse a DAWNMULT file and check its layout -> (G, cursor, [(labels, payload bytes)] per section)."""
    raw = open(path, "rb").read()
    assert raw[:8] == b"DAWNMULT"
    version, scalar, dims, G = np.frombuffer(raw[8:24], dtype="<u4")
    cursor = int(np.frombuffer(raw[24:32], dtype="<u8")[0])
    assert (version, scalar, dims) == (1, SCALAR[kind], 384) and 1 <= G <= 64 and cursor < G
    rows = np.frombuffer(raw[32:32 + 8 * G], dtype="<u8").astype(np.int64)
    assert not any(raw[32 + 8 * G:PAGE]), "header padding is not zero"
    end, sections = PAGE, []
    for g in range(G):
        start = -(-end // PAGE) * PAGE
        assert not any(raw[end:start]), f"padding before section {g} is not zero"
        n = int(rows[g])
        labels = np.frombuffer(raw[start:start + 8 * n], dtype="<u8")
        body = raw[start + 8 * n:start + 8 * n + payload_bytes(kind, n)]
        assert len(body) == payload_bytes(kind, n)
        sections.append((labels, body))
        end = start + 8 * n + payload_bytes(kind, n)
    assert len(raw) == end, ("file length", len(raw), end)
    return int(G), cursor, sections


def expected_payload(kind, rows, stored, idx):
    """The stored-row bytes a section holding corpus rows idx must carry."""
    if kind == "f16":
        return np.ascontiguousarray(stored[idx]).view(np.uint16).tobytes()
    if kind == "f32":
        return np.ascontiguousarray(rows[idx], dtype=np.float32).tobytes()
    q8, sc = stored[0][idx], stored[1][idx]
    n = len(idx)
    blocks = np.zeros((-(-n // 8), I8_BLOCK), dtype=np.uint8)
    for r in range(n):
        blocks[r // 8, (r % 8) * 384:(r % 8 + 1) * 384] = q8[r].view(np.uint8)
        blocks[r // 8, 3072 + (r % 8) * 4:3072 + (r % 8 + 1) * 4] = np.frombuffer(sc[r:r + 1].tobytes(), dtype=np.uint8)
    return blocks.tobytes()


def row_units(kind, body, n):
    """Split a section's payload into per-row byte strings (int8: the row's 384 bytes and its scale)."""
    if kind != "i8":
        w = ROW_BYTES[kind]
        return [body[r * w:(r + 1) * w] for r in range(n)]
    out = []
    for r in range(n):
        b = (r // 8) * I8_BLOCK
        out.append(body[b + (r % 8) * 384:b + (r % 8 + 1) * 384] + body[b + 3072 + (r % 8) * 4:b + 3072 + (r % 8 + 1) * 4])
    return out


# ---------------------------------------------------------------------------------------------------- corpora
class Corpus:
    def __init__(self, oracle, kind, n, salt):
        self.kind, self.n = kind, n
        self.rows = f32_rows(oracle, SEED + salt, n)
        self.labels = perm_labels(oracle, n, salt)
        self.stored = store(oracle, kind, self.rows)
        self.qs = oracle.make_queries(SEED + salt, 5, NQ, n)
        self.want = reference(oracle, kind, self.stored, self.labels, self.qs)
        self.limit = float(np.median(self.want[1][:, 10]))


def build(dawn, c, G, reserve=None):
    """A MultiIndex over corpus c, added in two add_batch calls; -> (handle, Placement)."""
    m = dawn.MultiIndex([0] * G, quantization=getattr(dawn.ScalarKind, KINDS[c.kind]))
    pl = Placement(G)
    m.reserve(reserve or c.n)
    pl.reserve(reserve or c.n)
    for a, b in ((0, FIRST_ADD), (FIRST_ADD, c.n)):
        m.add_batch(c.labels[a:b], c.rows[a:b])
        assert pl.add_batch(np.arange(a, b))
    assert m.size() == c.n
    return m, pl


ROUTES = {"f16": [("scan", {"force_path": 1}), ("tiles", {"force_path": 2}), ("shadow", {"force_path": 0, "shadow_i8": 1})],
          "i8": [("scan", {"force_path": 1}), ("tiles", {"force_path": 0})],
          "f32": [("scan", {"force_path": 1}), ("tiles", {"force_path": 2})]}


def answers(m, c):
    """Every route x k x (no limit, limit) -> {key: (labels, distances, counts)}."""
    out = {}
    for route, opts in ROUTES[c.kind]:
        for key, v in opts.items():
            m.set_option(key, v)
        for k in KS:
            out[(route, k, None)] = m.search_batch(c.qs, k)
            out[(route, k, c.limit)] = m.search_batch_limit(c.qs, k, c.limit)
    m.set_option("force_path", 0)
    if c.kind == "f16":
        m.set_option("shadow_i8", 0)
    return out


def check_answers(got, c, before=None, what=""):
    for (route, k, limit), a in got.items():
        check_answer(a, c.want, k, (what, route, k), limit=limit)
        if before is not None:
            b = before[(route, k, limit)]
            for x, y in zip(a, b):
                assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), (what, route, k, limit)


def gets(m, labels):
    return np.stack([m.get(int(x)) for x in labels])


# ---------------------------------------------------------------------------------------------------- 1-3. round trip
ROUND_TRIP = [("edge", 1), ("edge", 2), ("edge", 3), ("edge", 8), ("big", 2)]


@pytest.fixture(scope="module")
def saved(dawn, oracle, tmp_path_factory):
    """(kind, corpus name, G) -> (corpus, placement, answers, gets of every label, verify, file path)."""
    d = tmp_path_factory.mktemp("multi_persist")
    corpora, cache = {}, {}

    def get(kind, name, G):
        if (kind, name) not in corpora:
            corpora[(kind, name)] = Corpus(oracle, kind, N_EDGE if name == "edge" else N_BIG, 1 + list(KINDS).index(kind))
        c = corpora[(kind, name)]
        if (kind, name, G) not in cache:
            m, pl = build(dawn, c, G)
            path = str(d / f"{kind}-{name}-G{G}.dawn")
            before = answers(m, c)
            g_all = gets(m, c.labels) if name == "edge" else gets(m, c.labels[::97])
            ver = m.verify()
            m.save(path)
            m.close()
            cache[(kind, name, G)] = (c, pl, before, g_all, ver, path)
        return cache[(kind, name, G)]

    return get


def check_sections(path, c, pl, G, cursor):
    """A same-G file: the header and every section's labels and rows against the rows placement gave each shard."""
    g_file, cur, secs = read_multi(path, c.kind)
    assert g_file == G and cur == cursor
    for g, (labels, body) in enumerate(secs):
        idx = np.array(pl.rows[g], dtype=np.int64)
        assert np.array_equal(labels, c.labels[idx]), g
        assert body == expected_payload(c.kind, c.rows, c.stored, idx), ("section rows", g)


@pytest.mark.gpu
@pytest.mark.parametrize("target", ["fresh", "reserved", "nonempty"])
@pytest.mark.parametrize("name,G", ROUND_TRIP, ids=[f"{n}-G{g}" for n, g in ROUND_TRIP])
@pytest.mark.parametrize("kind", list(KINDS))
def test_round_trip_same_shard_count(dawn, oracle, saved, kind, name, G, target):
    c, pl, before, g_all, ver, path = saved(kind, name, G)
    check_sections(path, c, pl, G, pl.cursor % G)
    m = dawn.MultiIndex([0] * G, quantization=getattr(dawn.ScalarKind, KINDS[kind]))
    try:
        if target == "reserved":
            m.reserve(c.n)
            cap = m.capacity()
        elif target == "nonempty":
            other = Corpus(oracle, kind, 3000, 40)
            m.reserve(3000)
            m.add_batch(other.labels, other.rows)
        m.load(path)
        assert m.size() == c.n
        if target == "reserved":
            assert m.capacity() == cap  # filled in place: no second arena
        check_answers(answers(m, c), c, before, (kind, name, G, target))
        probe = c.labels if (name == "edge" and target == "fresh") else c.labels[::97]
        want = g_all if (name == "edge" and target == "fresh") else (g_all[::97] if name == "edge" else g_all)
        assert np.array_equal(bits(gets(m, probe)), bits(want))
        assert m.verify() == ver
    finally:
        m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_saves_are_deterministic(dawn, oracle, saved, kind, tmp_path):
    c, pl, _, _, _, path = saved(kind, "edge", 3)
    extra = Corpus(oracle, kind, 5000, 50)
    extra.labels = extra.labels + np.uint64(10 * N_EDGE)
    ref = open(path, "rb").read()
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    m, _ = build(dawn, c, 3)
    try:
        m.save(a)
        m.save(b)
        assert open(a, "rb").read() == open(b, "rb").read() == ref
        m.reserve(c.n + extra.n + 30_000)
        m.add_batch(extra.labels, extra.rows)
        m.save(a)
    finally:
        m.close()
    m2 = dawn.MultiIndex([0] * 3, quantization=getattr(dawn.ScalarKind, KINDS[kind]))
    try:
        m2.load(path)
        m2.save(b)
        assert open(b, "rb").read() == ref  # save -> load -> save
        m2.reserve(c.n + extra.n + 30_000)
        m2.add_batch(extra.labels, extra.rows)
        m2.save(b)
        assert open(a, "rb").read() == open(b, "rb").read()  # ... -> add X -> save equals add X -> save
        read_multi(b, kind)
    finally:
        m2.close()


# ---------------------------------------------------------------------------------------------------- 4. other shard counts
RESHARD = [(3, 1), (3, 2), (3, 5), (8, 3), (1, 4), ("single", 1), ("single", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("src,G2", RESHARD, ids=[f"{s}to{g}" for s, g in RESHARD])
@pytest.mark.parametrize("kind", list(KINDS))
def test_load_into_another_shard_count(dawn, saved, kind, src, G2, tmp_path):
    c, pl, _, g_all, _, path = saved(kind, "edge", 3 if src == "single" else src)
    if src == "single":
        path = str(tmp_path / "single.dawn")
        with dawn.Index(dawn.IndexOptions(device=0, quantization=getattr(dawn.ScalarKind, KINDS[kind]))) as one:
            one.reserve(c.n)
            one.add_batch(c.labels, c.rows)
            one.save(path)
        order = np.arange(c.n)
    else:
        order = np.concatenate([np.array(r, dtype=np.int64) for r in pl.rows])  # the sections, concatenated
    m = dawn.MultiIndex([0] * G2, quantization=getattr(dawn.ScalarKind, KINDS[kind]))
    try:
        m.load(path)
        assert m.size() == c.n
        again = str(tmp_path / "again.dawn")
        m.save(again)
        g_file, cursor, secs = read_multi(again, kind)
        assert g_file == G2 and cursor == 0
        per = -(-c.n // G2)
        units = row_units(kind, expected_payload(kind, c.rows, c.stored, order), c.n)
        for g, (labels, body) in enumerate(secs):
            a, b = min(g * per, c.n), min((g + 1) * per, c.n)
            assert np.array_equal(labels, c.labels[order[a:b]]), g
            assert row_units(kind, body, b - a) == units[a:b], ("rows moved or re-quantised", g)
        check_answers(answers(m, c), c, None, (kind, src, G2))
        assert np.array_equal(bits(gets(m, c.labels)), bits(g_all))
    finally:
        m.close()


# ---------------------------------------------------------------------------------------------------- 5. failures
def corrupt(raw, what):
    b = bytearray(raw)
    put = lambda off, v, dt: b.__setitem__(slice(off, off + np.dtype(dt).itemsize), np.array([v], dtype=dt).tobytes())  # noqa
    if what == "magic":
        b[0:8] = b"DAWNMULX"
    elif what == "version":
        put(8, 2, "<u4")
    elif what == "scalar":
        put(12, 3, "<u4")
    elif what == "dims":
        put(16, 768, "<u4")
    elif what == "G0":
        put(20, 0, "<u4")
    elif what == "G65":
        put(20, 65, "<u4")
    elif what == "cursor":
        put(24, 3, "<u8")
    elif what == "short":
        del b[-1]
    elif what == "long":
        b.append(0)
    return bytes(b)


BAD = ["missing", "magic", "version", "scalar", "dims", "G0", "G65", "cursor", "short", "long", "other-scalar"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_failed_load_leaves_the_handle_unchanged(dawn, oracle, saved, kind, tmp_path):
    c, _, _, _, _, path = saved(kind, "edge", 3)
    raw = open(path, "rb").read()
    live = Corpus(oracle, kind, 6000, 60)
    m = dawn.MultiIndex([0] * 2, quantization=getattr(dawn.ScalarKind, KINDS[kind]))
    try:
        m.reserve(6000)
        m.add_batch(live.labels, live.rows)
        ref_file = str(tmp_path / "ref")
        m.save(ref_file)
        ref_ans = m.search_batch(live.qs, 20)
        for what in BAD:
            bad = str(tmp_path / f"bad-{what}")
            if what == "other-scalar":
                other = [k for k in KINDS if k != kind][0]
                with dawn.Index(dawn.IndexOptions(device=0, quantization=getattr(dawn.ScalarKind, KINDS[other]))) as one:
                    one.reserve(100)
                    one.add_batch(live.labels[:100], live.rows[:100])
                    one.save(bad)
            elif what != "missing":
                open(bad, "wb").write(corrupt(raw, what))
            with pytest.raises(dawn.DawnError) as e:
                m.load(bad)
            assert e.value.code == IO, what
            assert m.size() == 6000, what
            got = m.search_batch(live.qs, 20)
            assert all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(got, ref_ans)), what
            again = str(tmp_path / "again")
            m.save(again)
            assert open(again, "rb").read() == open(ref_file, "rb").read(), what
        check_answer(m.search_batch(live.qs, 20), live.want, 20, "after the failures")
    finally:
        m.close()
    L = dawn.index.load_library()
    assert L.dawn_multi_save(None, b"x") == INVALID and L.dawn_multi_load(None, b"x") == INVALID
    with dawn.MultiIndex([0] * 2, quantization=getattr(dawn.ScalarKind, KINDS[kind])) as e:
        assert L.dawn_multi_save(e._h, None) == INVALID and L.dawn_multi_load(e._h, None) == INVALID
        empty = str(tmp_path / "empty")
        e.save(empty)
        g, cursor, secs = read_multi(empty, kind)
        assert g == 2 and cursor == 0 and all(len(lab) == 0 for lab, _ in secs) and os.path.getsize(empty) == PAGE
    with dawn.MultiIndex([0] * 3, quantization=getattr(dawn.ScalarKind, KINDS[kind])) as e3:
        e3.load(empty)
        assert e3.size() == 0 and e3.search_batch(live.qs[:2], 5)[2].tolist() == [0, 0]


# ---------------------------------------------------------------------------------------------------- 6. concurrent use
@pytest.mark.gpu
def test_searches_and_gets_run_through_a_save_and_a_load(dawn, oracle, saved, tmp_path):
    old = Corpus(oracle, "f16", N_BIG, 70)
    c, _, _, _, _, new_path = saved("f16", "big", 2)
    k = 20
    old_get = {int(x): None for x in old.labels[:64]}
    m, _ = build(dawn, old, 2)
    try:
        for x in old_get:
            old_get[x] = m.get(x)
        new_rows = {int(l): c.stored[i].astype(np.float32) for i, l in enumerate(c.labels) if int(l) in old_get}
        old_on_old = old.want
        new_on_old = reference(oracle, "f16", c.stored, c.labels, old.qs)  # the old queries against the new corpus
        stop, seen, errors = threading.Event(), {"old": 0, "new": 0}, []

        def same(got, want):
            return all(got[2][q] == min(want[2][q], k) and (got[0][q, :got[2][q]] == want[0][q, :got[2][q]]).all() and
                       (bits(got[1][q, :got[2][q]]) == bits(want[1][q, :got[2][q]])).all() for q in range(NQ))

        def worker():
            i = 0
            while not stop.is_set():
                try:
                    got = m.search_batch(old.qs, k)
                    which = "old" if same(got, old_on_old) else "new" if same(got, new_on_old) else None
                    assert which, "an answer of neither corpus"
                    seen[which] += 1
                    lab = list(old_get)[i % len(old_get)]
                    v = bits(m.get(lab))
                    assert np.array_equal(v, bits(old_get[lab])) or np.array_equal(v, bits(new_rows[lab])), lab
                    i += 1
                except (dawn.DawnError, AssertionError) as e:
                    errors.append(e)

        th = threading.Thread(target=worker)
        th.start()
        try:
            m.save(str(tmp_path / "during.dawn"))
            m.load(new_path)
        finally:
            stop.set()
            th.join()
        assert not errors, errors[:3]
        assert seen["old"] > 0
        check_answer(m.search_batch(c.qs, k), c.want, k, "after the load")
        read_multi(str(tmp_path / "during.dawn"), "f16")
    finally:
        m.close()


# ---------------------------------------------------------------------------------------------------- 7. read-back calls
@pytest.mark.gpu
def test_get_verify_and_i24_search(dawn, oracle):
    rows = f32_rows(oracle, SEED + 80, 30)
    rows[12] *= np.float32(1.05)  # off the gate on shard 1
    rows[25] *= np.float32(0.9)   # and on shard 2
    labels = np.arange(1, 31, dtype=np.uint64)
    labels[20] = labels[12] = 500  # label 500 on shard 1 (row 12) and shard 2 (row 20)
    labels[13] = 500               # twice on shard 1: its lowest row there answers
    with dawn.MultiIndex([0] * 3) as m:
        m.reserve(3000)
        for a, b in ((0, 10), (10, 20), (20, 30)):  # one add_batch per shard
            m.add_batch(labels[a:b], rows[a:b])
        stored = oracle.store_f16(rows).astype(np.float32)
        assert np.array_equal(bits(m.get(500)), bits(stored[12]))
        assert np.array_equal(bits(m.get(3)), bits(stored[2]))
        with pytest.raises(dawn.DawnError) as e:
            m.get(999)
        assert e.value.code == INVALID
        assert m.get_i24(500) == dawn.encode_i24(m.get(500))
        with dawn.Index(dawn.IndexOptions(device=0)) as one:  # one index holding every row has the same norms
            one.reserve(30)
            one.add_batch(labels, rows)
            want = one.verify()
        got = m.verify()
        assert got == want and got["bad_rows"] == 2, (got, want)
        for q in oracle.make_queries(SEED + 80, 3, 4, 30):
            wire = dawn.encode_i24(q)
            qd = dawn.decode_i24(wire)
            for lim in (None, 0.9):
                a = m.search_i24(wire, 10, lim)
                bl, bd, bc = m.search_batch_limit(qd[None, :], 10, float("nan") if lim is None else lim)
                assert np.array_equal(a.labels, bl[0, :bc[0]]) and np.array_equal(bits(a.distances), bits(bd[0, :bc[0]]))
        with pytest.raises(dawn.DawnError) as e:
            m.search_i24(bytes(1152), 10)
        assert e.value.code == INVALID
    with dawn.MultiIndex([0] * 2) as e:
        assert e.verify() == {"bad_rows": 0, "min_norm": 0.0, "max_norm": 0.0}
