"""The oracle's rules for stored vectors and scores outside the finite, unit-norm world (no GPU needed).

The raw ABI accepts any f32 vector, so the oracle has to say what an index holds and returns for NaN, +-inf and huge
components.  int8 storage: a NaN quotient stores 0 (Rust's `as`), any other quotient is clamped to +-127.  Search: a
row whose exact score is NaN is not a result; +-inf scores keep their order (distance -inf is the best)."""
import numpy as np
import pytest

EM = 384


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def odd_rows(oracle):
    rows = oracle.np_synth_rows_f32(41, 0, 12).copy()
    rows[0, 3] = np.nan
    rows[1, 5] = np.inf
    rows[2, 7] = -np.inf
    rows[3, :2] = (np.inf, -np.inf)
    rows[4, 9] = 1e30
    rows[5, 11] = -1e30
    rows[6] = np.float32(1e-40)           # f32 subnormals only
    rows[6, ::2] = -np.float32(1e-40)
    rows[7] = -0.0                          # negative zeros only: scale 1
    rows[8, 1] = np.nan
    rows[8, 2] = np.inf                     # NaN and inf together
    rows[9] = np.nan                        # nothing but NaN
    rows[10, 20] = np.float32(3.0e38)       # finite, near the f32 maximum
    return rows


def test_i8_store_of_non_finite_components(oracle):
    rows = odd_rows(oracle)
    q, s = oracle.store_i8(rows)
    qn, sn = oracle.np_store_i8(rows)
    assert (q == qn).all()
    assert (bits(s) == bits(sn)).all()
    # a NaN component stores 0 and stays out of absmax
    assert q[0, 3] == 0 and np.isfinite(s[0]) and np.abs(q[0]).max() == 127
    # an inf component makes the scale inf: inf / inf is NaN -> 0, every finite component / inf -> 0
    for r in (1, 2, 3, 8):
        assert np.isinf(s[r]) and (q[r] == 0).all(), r
    assert s[9] == 1.0 and (q[9] == 0).all()
    # huge finite components keep a finite scale and the row's shape
    assert np.isfinite(s[4]) and q[4, 9] == 127 and np.isfinite(s[5]) and q[5, 11] == -127
    assert np.isfinite(s[10]) and q[10, 20] == 127
    # subnormal rows quantise like any other row; -0 rows have scale 1
    assert s[6] > 0 and np.abs(q[6]).max() == 127
    assert s[7] == 1.0 and (q[7] == 0).all()


def nan_corpus(oracle, n=3000):
    rows = oracle.np_synth_rows_f32(42, 0, n).copy()
    rng = np.random.default_rng(5)
    nan_rows = rng.choice(n, 40, replace=False)
    rows[nan_rows, rng.integers(0, EM, 40)] = np.nan
    inf_rows = rng.choice(np.setdiff1d(np.arange(n), nan_rows), 6, replace=False)
    rows[inf_rows[:3], 0] = np.inf   # score +inf for q[0] > 0: distance -inf, the best
    rows[inf_rows[3:], 0] = -np.inf  # score -inf: distance +inf, the worst
    return rows, np.sort(nan_rows), inf_rows


@pytest.mark.parametrize("k", [1, 10, 64])
def test_nan_scores_are_not_results(oracle, k):
    rows, nan_rows, inf_rows = nan_corpus(oracle)
    n = len(rows)
    labels = np.arange(n, dtype=np.uint64) * 3 + 1
    stored = oracle.store_f16(rows)
    q = oracle.make_queries(42, 43, 1, n)[0].copy()
    q[0] = abs(q[0]) + 0.01
    for search, corpus in ((oracle.search_f16, stored), (oracle.search_f32, rows)):
        wl, wd = search(corpus, labels, q, k)
        nl, nd = oracle.np_search(corpus.astype(np.float32), labels, q, k)
        assert len(wl) == min(k, n - len(nan_rows))
        assert (wl == nl).all() and (bits(wd) == bits(nd)).all()
        assert not np.isin(wl, labels[nan_rows]).any()
        assert not np.isnan(wd).any()
        best = np.sort(labels[inf_rows[:3]])[:k]  # ties at -inf break on the label
        assert (wd[:len(best)] == -np.inf).all() and (wl[:len(best)] == best).all()
    cl, cd, cc, _ = oracle.cpu_scan_f16(stored, labels, q[None], k)
    wl, wd = oracle.search_f16(stored, labels, q, k)
    assert cc[0] == len(wl) and (cl[0, :cc[0]] == wl).all() and (bits(cd[0, :cc[0]]) == bits(wd)).all()


def test_nan_rows_make_the_count_short(oracle):
    """Fewer non-NaN rows than k: the count is the number of non-NaN rows, on every oracle."""
    rows = oracle.np_synth_rows_f32(44, 0, 20).copy()
    rows[::3, 7] = np.nan
    q = oracle.make_queries(44, 45, 1, 20)[0]
    keep = 20 - len(range(0, 20, 3))
    for wl, wd in (oracle.search_f16(oracle.store_f16(rows), None, q, 30), oracle.search_f32(rows, None, q, 30),
                   oracle.np_search(rows, None, q, 30)):
        assert len(wl) == keep and not np.isin(wl, np.arange(1, 21, 3)).any()
    # int8 storage keeps such rows: their NaN component is stored as 0
    q8, sc = oracle.store_i8(rows)
    assert len(oracle.search_i8(q8, sc, None, q, 30)[0]) == 20


def test_output_does_not_depend_on_row_order_with_nan_rows(oracle):
    rows, nan_rows, _ = nan_corpus(oracle)
    n = len(rows)
    labels = np.arange(n, dtype=np.uint64) + 1
    qs = oracle.make_queries(42, 46, 4, n)
    perm = np.random.default_rng(6).permutation(n)
    q8, sc = oracle.store_i8(rows)
    for q in qs:
        for k in (5, 50):
            a = oracle.search_f16(oracle.store_f16(rows), labels, q, k)
            b = oracle.search_f16(oracle.store_f16(rows[perm]), labels[perm], q, k)
            c = oracle.search_i8(q8, sc, labels, q, k)
            d = oracle.search_i8(q8[perm], sc[perm], labels[perm], q, k)
            for x, y in ((a, b), (c, d)):
                assert (x[0] == y[0]).all() and (bits(x[1]) == bits(y[1])).all()
