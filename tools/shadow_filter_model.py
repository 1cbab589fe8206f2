"""CPU model of the int8-shadow filter in gemm_i8_topk_kernel's epilogue: how often its first level sends a warp down the
slow path (examine(): levels 2 and 3), with per-row scales and with one scale per group of 32 rows.

    python tools/shadow_filter_model.py [--rows 1000000] [--queries 128] [--ranks 1,2,8]

Rows are the synthetic corpus (synth.rows_f32) stored as fp16; queries are unplanted make_queries queries.  The quantiser's
arithmetic is shadow_quantize_kernel's (f32 scale = absmax / 127 of the row or of its 32-row group, x8 = rint(x16 / s)
clamped, kappa measured on the stored scales), the query's is prep_queries_i8_gemm_kernel's.  For each query the threshold
T is its rank-r exact score over the sample, so r / rows is the share of rows above T; thr = (T - e1) / s1 as the select
publishes it.  One epilogue thread is one query: a warp holds 32 queries and runs examine() for a 32-column chunk when any
of them passes level 1, (max HI + cq) * max s >= thr over the chunk.

Columns: filter survivors per exact survivor (rows with s (HI + cq) >= thr over rows with exact >= T), level-1 passes per
(query, chunk), and the share of warp-chunks sent to examine().  The "int8 corpus" line is the same filter with the narrow
band of an int8-stored corpus (per-row scales, e1 = 1.03 delta + 3e-6, no cq), its survivors counted against the fp16 top.
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dawnsearch_b200 import synth  # noqa: E402

SEED = 0xDA5EA2C4
CHUNK = 1 << 16  # rows per block of work (a multiple of 32)


def quantize(x, group):
    """shadow_quantize_kernel on whole groups: (scales f32, x8 as f32, max ||x / s - x8||)."""
    amax = np.abs(x).max(axis=1)
    if group > 1:
        amax = np.repeat(amax.reshape(-1, group).max(axis=1), group)
    s = np.where(amax > 0, amax / np.float32(127.0), np.float32(1.0)).astype(np.float32)
    t = (x / s[:, None]).astype(np.float32)
    x8 = np.clip(np.rint(t), -127, 127)
    return s, x8, float(np.sqrt(((t - x8).astype(np.float64) ** 2).sum(axis=1)).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=128)
    ap.add_argument("--ranks", default="1,2,8")
    args = ap.parse_args()
    n = args.rows // 32 * 32
    nq = args.queries // 32 * 32
    ranks = [int(r) for r in args.ranks.split(",")]
    t0 = time.time()
    x16 = np.concatenate([synth.rows_f32(SEED, f, min(CHUNK, n - f)).astype(np.float16) for f in range(0, n, CHUNK)])
    qs = synth.make_queries(SEED, SEED + 1, nq, 100_000_000, planted_fraction=0.0).astype(np.float32)
    amax_q = np.abs(qs).max(axis=1)
    s1 = (amax_q / np.float32(127.0)).astype(np.float32)
    hi = np.clip(np.rint(qs / s1[:, None]), -127, 127).astype(np.float32)
    delta = np.sqrt(((qs.astype(np.float64) - s1[:, None].astype(np.float64) * hi) ** 2).sum(axis=1))
    qn = np.sqrt((qs.astype(np.float64) ** 2).sum(axis=1)) * 1.00001

    # pass 1: exact top scores per query, kappa of each quantiser
    top = np.full((max(ranks), nq), -np.inf)
    kappa = {1: 0.0, 32: 0.0}
    for f in range(0, n, CHUNK):
        x = x16[f:f + CHUNK].astype(np.float32)
        ex = x.astype(np.float64) @ qs.T.astype(np.float64)
        top = -np.sort(-np.concatenate([top, ex]), axis=0)[:max(ranks)]
        for g in kappa:
            kappa[g] = max(kappa[g], quantize(x, g)[2])
    kappa = {g: k * 1.00001 * 1.0001 + 1e-4 for g, k in kappa.items()}  # as the kernel and ensure_shadow store it
    print(f"{n} rows, {nq} queries, kappa per row {kappa[1]:.3f}, per 32-row group {kappa[32]:.3f} ({time.time() - t0:.0f} s)")

    modes = [("per row", 1, True), ("per 32-row group", 32, True), ("int8 corpus (per row, narrow band)", 1, False)]
    print("share above T | scales | survivors / exact | level-1 passes per (query, chunk) | warp-chunks to examine()")
    for r in ranks:
        T = top[r - 1]
        for name, g, shadow in modes:
            e1 = delta * 1.10 + 3e-5 if shadow else delta * 1.03 + 3e-6
            cq = (qn * kappa[g] / s1).astype(np.float32) if shadow else np.zeros(nq, np.float32)
            thr = ((T - e1) / s1).astype(np.float32)
            n_exact = n_filter = n_l1 = n_warp = 0
            for f in range(0, n, CHUNK):
                x = x16[f:f + CHUNK].astype(np.float32)
                s, x8, _ = quantize(x, g)
                HI = x8 @ hi.T  # exact integers (|HI| <= 384 * 127 * 127 < 2^24)
                n_exact += int((x.astype(np.float64) @ qs.T.astype(np.float64) >= T).sum())
                n_filter += int(((HI + cq) * s[:, None] >= thr).sum())
                hmax = HI.reshape(-1, 32, nq).max(axis=1)
                smax = s.reshape(-1, 32).max(axis=1)
                l1 = (hmax + cq) * smax[:, None] >= thr
                n_l1 += int(l1.sum())
                n_warp += int(l1.reshape(l1.shape[0], nq // 32, 32).any(axis=2).sum())
            chunks = n // 32
            print(f"{r / n:.1e} | {name} | {n_filter / max(n_exact, 1):.2f}x | {n_l1 / (chunks * nq):.2e} | "
                  f"{100.0 * n_warp / (chunks * nq // 32):.1f} %", flush=True)


if __name__ == "__main__":
    main()
