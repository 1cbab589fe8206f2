"""CPU model of the grouped int8 shadow (shadow_quantize_kernel with option "shadow_group_rows" = 32): numpy restatements of
the kernel's arithmetic, not of the kernel.

A call quantises rows [first, first + n).  Rows share the scale s = fl(max absmax / 127) of the rows of their 32-row group
(aligned to the row index) that the same call quantises; rows below `first` keep what an earlier call gave them.  Zero and
non-finite rows are stored as zeros under the group's scale and do not enter its maximum.  x8 = clamp(rint(fl(x / s))) and
kappa = max ||x / s - x8|| over the rows, with the stored s.  Then, as in gemm_i8_topk_kernel's epilogue:
1. the filter s (HI + cq) >= thr never drops a row whose exact score reaches T, whatever mix of scales a chunk holds;
2. the first level's chunk test (max HI + cq) * max s >= thr is implied by any element of the chunk passing (thr > 0);
3. a full group carries one scale, at least as large as each of its rows' own absmax / 127."""
import numpy as np
import pytest

from oracle import oracle as O

DIM = 384
G = 32


class Shadow:
    """The stored scales and int8 rows of an index's shadow, built by appends like ensure_shadow."""

    def __init__(self, n):
        self.s = np.zeros(n, np.float32)
        self.x8 = np.zeros((n, DIM), np.int32)
        self.kappa_raw = 0.0
        self.rows = 0

    def append(self, x16, group=G):
        first, end = self.rows, len(x16)
        x = x16[first:end].astype(np.float32)
        with np.errstate(invalid="ignore"):
            amax = np.abs(x).max(axis=1)
        amax = np.where(amax < np.inf, amax, np.float32(0)).astype(np.float32)  # inf -> stored as zeros
        m = amax.copy()
        if group > 1:
            gid = np.arange(first, end) // group
            for g in np.unique(gid):
                m[gid == g] = amax[gid == g].max()
        s = np.where(m > 0, m / np.float32(127.0), np.float32(1.0)).astype(np.float32)
        v = np.where(amax[:, None] > 0, x, np.float32(0)).astype(np.float32)
        t = (v / s[:, None]).astype(np.float32)
        x8 = np.clip(np.rint(t), -127, 127).astype(np.int32)
        err = np.sqrt(((t - x8).astype(np.float64) ** 2).sum(axis=1)) * 1.00001
        self.kappa_raw = max(self.kappa_raw, float(err.max()))
        self.s[first:end], self.x8[first:end] = s, x8
        self.rows = end

    @property
    def kappa(self):
        return self.kappa_raw * 1.0001 + 1e-4  # what ensure_shadow publishes


def quantize_query(q):
    """prep_queries_i8_gemm_kernel in shadow mode."""
    s1 = np.float32(np.abs(q).max() / np.float32(127.0))
    hi = np.clip(np.rint(q / s1), -127, 127).astype(np.int32)
    delta = float(np.sqrt(((q.astype(np.float64) - float(s1) * hi) ** 2).sum()))
    qn = float(np.sqrt((q.astype(np.float64) ** 2).sum())) * 1.00001
    return s1, hi, delta * 1.10 + 3.0e-5, qn


def corpus(kind, n, rng):
    rows = O.np_synth_rows_f32(91, 0, n)
    if kind == "one_large_component":  # every 7th row: one component carries most of the norm -> groups of mixed scales
        big = rows[::7]
        big[np.arange(len(big)), rng.integers(0, DIM, len(big))] = 8.0
    elif kind == "near_duplicates":
        rows = np.repeat(rows[:1], n, axis=0) + rng.normal(size=(n, DIM)).astype(np.float32) * 3e-4
        rows[::5] *= rng.uniform(0.3, 1.0, size=(len(rows[::5]), 1)).astype(np.float32)  # same direction, smaller absmax
    rows /= np.linalg.norm(rows, axis=1, keepdims=True)
    rows[37] = 0.0  # a zero row inside a group
    return O.store_f16(rows)


# appends that split groups: 45 = 32 + 13, 100 = 96 + 4, ...
BOUNDS = (45, 100, 101, 130, 2000, 4000)


@pytest.mark.parametrize("kind", ["gaussian", "one_large_component", "near_duplicates"])
def test_grouped_filter_never_drops_a_hit(kind):
    rng = np.random.default_rng(17)
    x16 = corpus(kind, BOUNDS[-1], rng)
    sh = Shadow(len(x16))
    for b in BOUNDS:
        sh.append(x16[:b])
    assert sh.kappa <= np.sqrt(DIM) / 2 * 1.001 + 2e-4
    x64 = x16.astype(np.float64)
    queries = [O.np_synth_rows_f32(92, i, 1)[0] for i in range(5)]
    queries += [x16[i].astype(np.float32) for i in (44, 45, 99, 100, 7 * 20)]  # rows next to the append boundaries
    mixed = 0
    for q in queries:
        q = (q / np.linalg.norm(q)).astype(np.float32)
        s1, hi, e1, qn = quantize_query(q)
        HI = sh.x8 @ hi
        exact = x64 @ q.astype(np.float64)
        a = float(s1) * sh.s.astype(np.float64) * HI
        assert (np.abs(exact - a) <= e1 - 2.4e-5 + qn * sh.kappa * sh.s.astype(np.float64)).all(), kind
        cq = np.float32(qn * sh.kappa / float(s1))
        f = (HI.astype(np.float32) + cq) * sh.s
        for rank in (1, 10, 200):
            T = np.sort(exact)[-rank]
            thr = np.float32((np.float32(T) - np.float32(e1)) / s1)
            thr = np.float32(thr - abs(thr) * np.float32(4.0e-7))
            assert (f[exact >= T] >= thr).all(), (kind, rank)
            if not thr > 0:
                continue  # the kernel skips the chunk bound below a positive threshold
            # level 1 over every 32-column chunk (tiles start at multiples of 256 rows: chunks are the groups)
            n = len(f) // G * G
            hmax = HI[:n].reshape(-1, G).max(axis=1).astype(np.float32)
            smax = sh.s[:n].reshape(-1, G).max(axis=1)
            l1 = (hmax + cq) * smax >= thr
            any_elem = (f[:n].reshape(-1, G) >= thr).any(axis=1)
            assert l1[any_elem].all(), (kind, rank)
        mixed = int((sh.s[:n].reshape(-1, G).min(axis=1) < sh.s[:n].reshape(-1, G).max(axis=1)).sum())
    assert mixed >= 2  # the groups split at 45 and 100 carry two scales each


def test_group_scales():
    rng = np.random.default_rng(23)
    x16 = corpus("one_large_component", 4000, rng)
    x16[200] = np.float16(np.inf)  # a non-finite row: zeros under its group's scale, not part of the group's maximum
    finite = np.isfinite(x16.astype(np.float32)).all(axis=1)
    own = np.where(finite, np.abs(x16.astype(np.float32)).max(axis=1) / np.float32(127.0), np.float32(0)).astype(np.float32)
    whole = Shadow(len(x16))
    whole.append(x16)  # one call: every group full
    for g in range(len(x16) // G):
        grp = whole.s[g * G:(g + 1) * G]
        assert (grp == own[g * G:(g + 1) * G].max()).all()  # one scale: fl(max absmax / 127) = max fl(absmax / 127)
        assert (grp >= own[g * G:(g + 1) * G]).all()
    assert (whole.x8[200] == 0).all() and (whole.x8[37] == 0).all()  # the inf row and the zero row
    appended = Shadow(len(x16))
    for b in BOUNDS:
        before = appended.s[:appended.rows].copy()
        appended.append(x16[:b])
        assert (appended.s[:len(before)] == before).all()  # rows already published keep their scales
    for g in range(len(x16) // G):
        grp = appended.s[g * G:(g + 1) * G]
        assert (grp >= own[g * G:(g + 1) * G]).all()
        cuts = [0] + [b - g * G for b in BOUNDS if g * G < b < (g + 1) * G] + [G]  # a scale for each append's part of the group
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            assert (grp[lo:hi] == grp[lo]).all()
    per_row = Shadow(len(x16))  # shadow_group_rows = 1
    per_row.append(x16, group=1)
    assert (per_row.s[own > 0] == own[own > 0]).all() and (per_row.s[own == 0] == 1.0).all()
