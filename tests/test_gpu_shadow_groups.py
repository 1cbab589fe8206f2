"""Option "shadow_group_rows": the int8 shadow of an fp16 corpus stores one scale per group of 32 rows (the default) or one per
row.  The shadow only filters, so answers must be bit-identical to the oracle, to the fp16 tensor-core path and to each
other -- also when appends split a group, so that its old rows keep their scale and its new rows get another."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 0xDA5EA2C4


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def same(a, b):
    assert (a[2] == b[2]).all()
    assert (a[0] == b[0]).all()
    assert (bits(a[1]) == bits(b[1])).all()


def corpus(oracle):
    """Synthetic rows with a spiky row (one large component) and a zero row in the groups that the appends below split."""
    n = 65536 + 5 + 27 + 100_003
    rows = oracle.np_synth_rows_f32(SEED + 9, 0, n)
    rng = np.random.default_rng(3)
    spiky = rng.normal(size=384).astype(np.float32) * 0.02
    spiky[7] = 0.95
    for r in (65_550, 165_569):  # the second group split by an append; the last, partial group
        rows[r] = spiky / np.linalg.norm(spiky)
    rows[65_545] = 0.0
    labels = np.arange(n, dtype=np.uint64) * 5 + 11
    near = rows[[65_537, 65_550, 65_560, 65_600, 165_569]] + rng.normal(size=(5, 384)).astype(np.float32) * 0.05
    qs = np.concatenate([near / np.linalg.norm(near, axis=1, keepdims=True),
                         oracle.make_queries(SEED + 9, 4, 1024 - 5, n)]).astype(np.float32)
    return rows, labels, qs


def search_shadow(idx, qs, k):
    idx.profile(reset=True)
    got = idx.search_batch(qs, k)
    p = idx.profile(reset=True)
    assert p["shadow_batches"] == 1, p
    assert p["uncertified"] == 0 and p["escalations"] == 0 and p["device_uncertified"] == 0 and p["device_status"] == 0, p
    return got


def test_grouped_shadow_over_uneven_appends(dawn, oracle):
    rows, labels, qs = corpus(oracle)
    stored = oracle.store_f16(rows)
    n = len(rows)
    with dawn.new_index(dawn.IndexOptions(capacity=n)) as idx:
        idx.set_option("shadow_i8", 1)
        idx.set_option("shadow_single_rows", 0)  # a single query takes the shadow too
        with pytest.raises(dawn.DawnError):
            idx.set_option("shadow_group_rows", 16)
        start = 0
        for end in (65_541, 65_568, n):  # each search in between extends the shadow from the previous end
            idx.add_batch(labels[start:end], rows[start:end])
            start = end
            for k in (10, 20):
                wl, wd, wc, _ = oracle.cpu_scan_f16(stored[:end], labels[:end], qs, k)
                for b in (1, 64, 1024):
                    got = search_shadow(idx, qs[:b], k)
                    same(got, (wl[:b], wd[:b], wc[:b]))
                    idx.set_option("shadow_i8", 0)
                    plain = idx.search_batch(qs[:b], k)
                    idx.set_option("shadow_i8", 1)
                    same(got, plain)
        # per-row scales (the shadow is rebuilt in one piece), then groups again: the same answers
        for k in (10, 20):
            for b in (64, 1024):
                grouped = search_shadow(idx, qs[:b], k)
                idx.set_option("shadow_group_rows", 1)
                per_row = search_shadow(idx, qs[:b], k)
                idx.set_option("shadow_group_rows", 32)
                regrouped = search_shadow(idx, qs[:b], k)
                same(grouped, per_row)
                same(grouped, regrouped)
