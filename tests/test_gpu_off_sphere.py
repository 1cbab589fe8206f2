"""Every search path on rows and queries off the unit sphere (DESIGN.md section 2, "Rows outside the reference's norm gate").

The raw ABI accepts any vector, and every search must still return the oracle's top-k bit for bit.  The kernels' error
bounds are derived for |q| ~ 1 and finite rows, so these tests feed them scaled queries, limits that are exactly an emitted
distance, rows with inf / NaN / fp16-overflowing components and rows far inside and outside the gate.

Each call is checked against two invariants (`profile(reset=True)` per call):
  I1  if no result is reported uncertified, labels, distance bits and counts equal the oracle's;
  I2  for finite rows and 2^-2 <= |q| <= 2^14 they equal the oracle's whatever the certificate says (escalations allowed).
Tiny queries collapse many scores onto one f32 distance and a one-hot query ties thousands of rows: only I1 holds there.
Each path is forced with the existing options, and the profile shows that it (or the path the index must fall back to)
really ran."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 0x0FF5FE2E
N = 70_000                      # >= 65,536: the shadow and the int8 tensor-core paths serve this corpus
ODD = (31, 32, 255, 256, N - 1)  # group / tile edges and the last row
K = 10

DEFAULTS = {"force_path": 0, "shadow_i8": 0, "shadow_group_rows": 32, "shadow_big_k_rows": 40_000_000,
            "i8_tensor_min_batch": 16, "i8_native": 1}


def scan_ran(p):
    return p["gemm_batches"] == 0 and p["shadow_batches"] == 0 and p["scan_launches"] > 0


def k3_ran(p):
    return p["gemm_batches"] >= 1 and p["shadow_batches"] == 0


def shadow_ran(p):
    return p["shadow_batches"] >= 1


# name -> (options, the profile of that path)
F16_PATHS = {
    "scan": ({"force_path": 1}, scan_ran),
    "k3": ({"force_path": 2}, k3_ran),
    "shadow32": ({"force_path": 2, "shadow_i8": 1, "shadow_group_rows": 32, "shadow_big_k_rows": 0}, shadow_ran),
    "shadow1": ({"force_path": 2, "shadow_i8": 1, "shadow_group_rows": 1, "shadow_big_k_rows": 0}, shadow_ran),
}
I8_PATHS = {
    "i8scan": ({"i8_tensor_min_batch": 0}, lambda p: p["gemm_batches"] == 0 and p["scan_launches"] > 0),
    "i8native": ({"i8_tensor_min_batch": 1, "i8_native": 1}, lambda p: p["gemm_batches"] >= 1),
    "i8tiles": ({"i8_tensor_min_batch": 1, "i8_native": 0}, lambda p: p["gemm_batches"] >= 1),
}
F32_PATHS = {"f32scan": ({"force_path": 1}, scan_ran), "f32k3": ({"force_path": 2}, k3_ran)}


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def use_path(idx, opts):
    for key, val in {**DEFAULTS, **opts}.items():
        idx.set_option(key, val)


def reference(oracle, kind, stored, labels, qs, k):
    """The scalar oracle per query (the threaded SIMD scan's slack assumes |q| <= 1)."""
    def one(q):
        if kind == "i8":
            return oracle.search_i8(stored[0], stored[1], labels, q, k)
        return (oracle.search_f32 if kind == "f32" else oracle.search_f16)(stored, labels, q, k)

    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        res = list(ex.map(one, qs))
    wl = np.zeros((len(qs), k), dtype=np.uint64)
    wd = np.zeros((len(qs), k), dtype=np.float32)
    wc = np.zeros(len(qs), dtype=np.int64)
    for i, (l, d) in enumerate(res):
        wc[i] = len(l)
        wl[i, :len(l)], wd[i, :len(l)] = l, d
    return wl, wd, wc


def differing(got, want):
    gl, gd, gc = got
    wl, wd, wc = want
    out = []
    for i in range(len(wc)):
        c = int(wc[i])
        if gc[i] != c or not (gl[i, :c] == wl[i, :c]).all() or not (bits(gd[i, :c]) == bits(wd[i, :c])).all():
            out.append(i)
    return out


def check(idx, got, want, strict, ran, what):
    """I1, then I2 on the queries flagged strict, then which path served the call."""
    p = idx.profile(reset=True)
    bad = differing(got, want)
    assert p["device_status"] == 0, (what, p)
    if p["uncertified"] == 0:
        assert not bad, ("I1: certified yet not the oracle's", what, bad[:8], p)
    strict_bad = [i for i in bad if strict[i]]
    assert not strict_bad, ("I2", what, strict_bad[:8], p)
    if ran is not None:
        assert ran(p), ("path", what, p)


def run_paths(idx, paths, qs, k, want, strict, route=None, small_batch=True):
    """Every path on the whole batch (>= 129 queries: K3's CTA-pair form) and K3 on 64 queries (one CTA)."""
    for name, (opts, ran) in paths.items():
        use_path(idx, opts)
        idx.profile(reset=True)
        expect = route(name, ran) if route else ran
        check(idx, idx.search_batch(qs, k), want, strict, expect, name)
        if small_batch and name in ("k3", "f32k3"):
            idx.profile(reset=True)
            sub = tuple(w[:64] for w in want)
            check(idx, idx.search_batch(qs[:64], k), sub, strict[:64], expect, name + "/64")
    use_path(idx, {})


def make_index(dawn, kind, rows, labels):
    quant = {"f16": dawn.ScalarKind.F16, "i8": dawn.ScalarKind.I8, "f32": dawn.ScalarKind.F32}[kind]
    idx = dawn.new_index(dawn.IndexOptions(quantization=quant, capacity=len(rows)))
    idx.add_batch(labels, rows)
    return idx


def store(oracle, kind, rows):
    return {"f16": oracle.store_f16, "i8": oracle.store_i8, "f32": lambda r: r}[kind](rows)


@pytest.fixture(scope="module")
def base_rows(oracle):
    return np.concatenate([oracle.np_synth_rows_f32(SEED, i, min(20_000, N - i)) for i in range(0, N, 20_000)])


@pytest.fixture(scope="module")
def labels():
    return np.arange(N, dtype=np.uint64) * 7 + 3


# ---------------------------------------------------------------------------------------------------- A. query scale
SCALES = [2.0 ** -24, 2.0 ** -12, 2.0 ** -6, 2.0 ** -2, 1.0, 4.0, 64.0, 4096.0, 16384.0, 3.7]


def scaled_queries(oracle):
    base = oracle.make_queries(SEED, 1, 13, N)
    qs = [base * np.float32(s) for s in SCALES]
    one_hot = np.zeros((1, 384), dtype=np.float32)
    one_hot[0, 7] = 1.0
    qs = np.concatenate(qs + [np.zeros((1, 384), dtype=np.float32), one_hot]).astype(np.float32)
    strict = np.array([2.0 ** -2 <= s <= 2.0 ** 14 for s in SCALES for _ in range(13)] + [False, False])
    return qs, strict


@pytest.mark.parametrize("kind", ["f16", "i8", "f32"])
def test_a_query_scale(dawn, oracle, base_rows, labels, kind):
    qs, strict = scaled_queries(oracle)
    want = reference(oracle, kind, store(oracle, kind, base_rows), labels, qs, K)
    with make_index(dawn, kind, base_rows, labels) as idx:
        run_paths(idx, {"f16": F16_PATHS, "i8": I8_PATHS, "f32": F32_PATHS}[kind], qs, K, want, strict)


# ---------------------------------------------------------------------------------------------------- B. limit edges
def limit_cases(oracle, kind, stored, labels):
    base = oracle.make_queries(SEED, 2, 4, N)
    qs = np.concatenate([base * np.float32(s) for s in (1.0, 64.0, 4096.0)]).astype(np.float32)
    want = reference(oracle, kind, stored, labels, qs, K)
    limits = [-np.inf]
    for g in range(3):
        for j in (0, K // 2, K - 1):
            d = np.float32(want[1][4 * g, j])
            limits += [d, np.nextafter(d, np.float32(-np.inf)), np.nextafter(d, np.float32(np.inf))]
    return qs, want, limits


def check_limit(got, want, limit, what):
    gl, gd, gc = got
    wl, wd, wc = want
    for i in range(len(wc)):
        keep = int((wd[i, :wc[i]] < np.float32(limit)).sum())
        assert gc[i] == keep, (what, limit, i, gc[i], keep)
        assert (gl[i, :keep] == wl[i, :keep]).all() and (bits(gd[i, :keep]) == bits(wd[i, :keep])).all(), (what, limit, i)


@pytest.mark.parametrize("kind", ["f16", "i8"])
def test_b_limit_edges(dawn, oracle, base_rows, labels, kind):
    """The limit is exactly an emitted distance, one ulp either side of it, or -inf: the hits are exactly those with d < L."""
    qs, want, limits = limit_cases(oracle, kind, store(oracle, kind, base_rows), labels)
    paths = {"f16": {n: F16_PATHS[n] for n in ("scan", "k3", "shadow32")}, "i8": I8_PATHS}[kind]
    with make_index(dawn, kind, base_rows, labels) as idx:
        for name, (opts, ran) in paths.items():
            use_path(idx, opts)
            for lim in limits:
                idx.profile(reset=True)
                check_limit(idx.search_batch_limit(qs, K, float(lim)), want, lim, name)
                p = idx.profile(reset=True)
                assert p["device_status"] == 0 and (lim == -np.inf or ran(p)), (name, lim, p)


def test_b_limit_edges_on_the_device_api(dawn, oracle, base_rows, labels):
    """search_device_limit cuts the counts on the device, with no host round trip to escalate through."""
    import torch

    qs, want, limits = limit_cases(oracle, "f16", oracle.store_f16(base_rows), labels)
    b = len(qs)
    with make_index(dawn, "f16", base_rows, labels) as idx:
        for force in (1, 2):
            idx.set_option("force_path", force)
            for lim in limits:
                dq = torch.from_numpy(qs).cuda()
                ol = torch.zeros((b, K), dtype=torch.int64, device="cuda")
                od = torch.zeros((b, K), dtype=torch.float32, device="cuda")
                oc = torch.zeros(b, dtype=torch.int32, device="cuda")
                of = torch.zeros(b, dtype=torch.int32, device="cuda")
                idx.profile(reset=True)
                idx.search_device(dq.data_ptr(), b, K, ol.data_ptr(), od.data_ptr(), oc.data_ptr(), of.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream or 1, distance_limit=float(lim))
                torch.cuda.synchronize()
                got = (ol.cpu().numpy().view(np.uint64), od.cpu().numpy(), oc.cpu().numpy().astype(np.int64))
                flags = of.cpu().numpy()
                for i in range(b):
                    if flags[i]:  # certified on the device: the hits must be the oracle's
                        check_limit(tuple(g[i:i + 1] for g in got), tuple(w[i:i + 1] for w in want), lim, force)


# ---------------------------------------------------------------------------------------------------- C. infinite fp16 rows
def inf_rows(base_rows):
    rows = base_rows.copy()
    rows[31, 0] = np.inf
    rows[32, 0] = 7e4        # rounds to +inf in fp16
    rows[255, 1] = -np.inf
    rows[256, 1] = -1e5      # rounds to -inf in fp16
    rows[N - 1, 2] = np.inf
    return rows


def weighted_queries(oracle, cols, seed):
    """Four queries per base query: positive, negative, zero and fp16-flushed (|q_i| < 2^-25) weight on `cols`."""
    base = oracle.make_queries(SEED, seed, 33, N)
    out = []
    for w in (0.05, -0.05, 0.0, 2.0 ** -26):
        q = base.copy()
        q[:, cols] = np.float32(w)
        out.append(q)
    return np.concatenate(out).astype(np.float32)


def test_c_infinite_fp16_rows(dawn, oracle, base_rows, labels):
    rows = inf_rows(base_rows)
    qs = weighted_queries(oracle, [0, 1, 2], 3)
    strict = np.ones(len(qs), dtype=bool)
    want = reference(oracle, "f16", oracle.store_f16(rows), labels, qs, K)
    assert (want[1][:33, 0] == -np.inf).all()  # +inf scores lead every positive-weight query
    with make_index(dawn, "f16", rows, labels) as idx:
        v = idx.verify()
        assert v["bad_rows"] == len(ODD), v
        run_paths(idx, F16_PATHS, qs, K, want, strict, route=lambda name, ran: scan_ran)
        # without them (and after verify() has rescanned the rows) the fast paths come back
        assert idx.remove_batch(labels[list(ODD)]) == len(ODD)
        assert idx.verify()["bad_rows"] == 0
        keep = np.setdiff1d(np.arange(N), ODD)
        want = reference(oracle, "f16", oracle.store_f16(rows[keep]), labels[keep], qs, K)
        run_paths(idx, F16_PATHS, qs, K, want, strict)


def test_c_infinite_rows_across_two_shards(dawn, oracle, base_rows, labels):
    """-inf distances go through merge_results_device."""
    rows = inf_rows(base_rows)
    qs = weighted_queries(oracle, [0, 1, 2], 4)[:66]
    want = reference(oracle, "f16", oracle.store_f16(rows), labels, qs, K)
    with dawn.MultiIndex([0, 0]) as m:
        m.reserve(N)
        m.add_batch(labels, rows)
        for force in (1, 2):
            m.set_option("force_path", force)
            got = m.search_batch(qs, K)
            assert not differing(got, want), force


# ---------------------------------------------------------------------------------------------------- D. NaN fp16 rows
def test_d_nan_fp16_rows(dawn, oracle, base_rows, labels):
    rows = base_rows.copy()
    for r, c in zip(ODD, (5, 100, 0, 383, 7)):
        rows[r, c] = np.nan
    qs = weighted_queries(oracle, [0, 5], 5)
    want = reference(oracle, "f16", oracle.store_f16(rows), labels, qs, K)
    assert not np.isin(want[0], labels[list(ODD)]).any()
    with make_index(dawn, "f16", rows, labels) as idx:
        assert idx.verify()["bad_rows"] == len(ODD)
        run_paths(idx, F16_PATHS, qs, K, want, np.ones(len(qs), dtype=bool), route=lambda name, ran: scan_ran)


# ---------------------------------------------------------------------------------------------------- E. int8 storage
def test_e_int8_rows_with_nan_inf_and_huge_components(dawn, oracle, base_rows, labels):
    rows = base_rows.copy()
    rows[31, 5] = np.nan
    rows[32, 0] = np.inf
    rows[255, 1] = -np.inf
    rows[256, 2] = 1e30
    rows[N - 1, 0], rows[N - 1, 3] = 1e30, np.nan
    q8, sc = oracle.store_i8(rows)
    qs = weighted_queries(oracle, [0, 1, 2, 3, 5], 6)
    want = reference(oracle, "i8", (q8, sc), labels, qs, K)
    with make_index(dawn, "i8", rows, labels) as idx:
        for r in ODD + (0, 1000):
            got = idx.get(int(labels[r]))
            exp = q8[r].astype(np.float32) * sc[r]
            assert np.array_equal(got, exp, equal_nan=True), (r, got[:6], exp[:6])
        # rows with an infinite scale are odd rows of the norm gate: the int8 scan answers
        run_paths(idx, I8_PATHS, qs, K, want, np.zeros(len(qs), dtype=bool), route=lambda name, ran: I8_PATHS["i8scan"][1])


# ---------------------------------------------------------------------------------------------------- F. f32 beyond fp16
def test_f_f32_rows_beyond_the_fp16_range(dawn, oracle, base_rows, labels):
    rows = base_rows.copy()
    rows[31] = 0.0
    rows[31, :2] = (7e4, -7e4)     # fp16 copy inf - inf; exact score 0.6 * 7e4 - 0.5 * 7e4 = 7000
    rows[255, 0] = 1e5
    rows[N - 1, 2] = -7e4
    q = oracle.make_queries(SEED, 7, 130, N)
    q[:, :3] = (0.6, 0.5, -0.02)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    qs = q.astype(np.float32)
    want = reference(oracle, "f32", rows, labels, qs, K)
    assert (want[0][0, :3] == labels[[255, 31, N - 1]]).all()  # 1e5 * q0 first, then the row the fp16 copy would lose
    with make_index(dawn, "f32", rows, labels) as idx:
        run_paths(idx, F32_PATHS, qs, K, want, np.ones(len(qs), dtype=bool), route=lambda name, ran: None)


# ---------------------------------------------------------------------------------------------------- G. short and long rows
@pytest.mark.parametrize("kind", ["f16", "i8", "f32"])
def test_g_rows_scaled_in_and_out_of_the_gate(dawn, oracle, base_rows, labels, kind):
    """Rows times 2^-10 (fp16 subnormal components) and times 2^4: the certificate's eps is scaled by the longest row."""
    rows = base_rows.copy()
    rows[::7] *= np.float32(2.0 ** -10)
    rows[3::11] *= np.float32(16.0)
    base = oracle.make_queries(SEED, 8, 65, N)
    qs = np.concatenate([base, base * np.float32(64.0)]).astype(np.float32)
    want = reference(oracle, kind, store(oracle, kind, rows), labels, qs, K)
    paths = {"f16": F16_PATHS, "i8": I8_PATHS, "f32": F32_PATHS}[kind]
    # rows beyond the gate turn the shadow off (its filter band is derived for the gate); K3 answers instead
    route = lambda name, ran: k3_ran if name.startswith("shadow") else ran  # noqa: E731
    with make_index(dawn, kind, rows, labels) as idx:
        assert idx.verify()["bad_rows"] == len(range(0, N, 7)) + len(range(3, N, 11)) - len(range(14, N, 77))
        run_paths(idx, paths, qs, K, want, np.ones(len(qs), dtype=bool), route=route)
