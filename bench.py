#!/usr/bin/env python
"""bench.py -- exact top-k over a synthetic N x 384 fp16 corpus on 1..8 B200 (BASELINE.json metric:
queries/sec and p50 latency, exact top-10 over 100M x 384 fp16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--rows R] [--batch B] [--k 10]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU arm (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's results as DIR/<name>.npy

A step = one batch of B queries (default 1024: the throughput configuration) answered against the
whole corpus (R rows, sharded by id range over the N GPUs: strong scaling).
  value  = queries/s with queries and corpus resident in HBM (CUDA events on the launching
           stream, max over ranks)
  e2e    = the same through the public API with HOST buffers (dawn_index_search_batch at N=1,
           ShardedIndex.search at N>1): H2D of the queries and D2H of the results inside the
           timed region
  batch1 = the latency configuration (one query per step): device and end-to-end p50/p99 and the
           HBM roofline of the streaming-scan kernel
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

SEED = 0xDA5EA2C4
DIM = 384
ROW_BYTES = 768
METRIC = "queries/sec, exact top-k over N x 384 fp16"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="total corpus rows (all GPUs)")
    ap.add_argument("--batch", type=int, default=1024, help="queries per step")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--scalar", default="f16", choices=["f16", "i8"], help="stored precision of the corpus")
    ap.add_argument("--no-shadow", action="store_true",
                    help="fp16 corpus: do not keep the int8 shadow copy (option shadow_i8); batches then run on the fp16 tensor-core tiles")
    ap.add_argument("--latency-steps", type=int, default=200, help="batch-1 steps for the latency section (0 = skip)")
    ap.add_argument("--cpu-sample-rows", type=int, default=2_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweep", default="", help="extra device-resident points: 'batch[:k],...' e.g. 1,4,16:100")
    ap.add_argument("--front", default="sharded", choices=["sharded", "multi"],
                    help="sharded: one process per GPU (torch.distributed / NCCL, the driver's launch); multi: ONE process "
                         "drives all --gpus through the C ABI's dawn_multi_* (NCCL all-gather inside the library)")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the pre-timing comparison with the CPU oracle")
    ap.add_argument("--parity-rows", type=int, default=2_000_000)
    ap.add_argument("--no-hnsw", action="store_true", help="reference arm: skip the HNSW stand-in (build takes ~1 min)")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="reference arm: wall-clock budget of the exact-scan steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the timed path returned in its last step (labels, distances, "
                         "counts; float64 / float32) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


DUMP_LIMIT_BYTES = 64_000_000
NPY_HEADER_BYTES = 1024  # room left per file for the .npy header


def dump_outputs(out_dir, labels, distances, counts):
    """The results of one batch as DIR/{labels,distances,counts}.npy (labels and counts as float64: exact below 2^53).
    A batch whose results exceed DUMP_LIMIT_BYTES is cut to a fixed, seeded sample of its queries, listed in query_rows.npy."""
    labels = np.asarray(labels).astype(np.float64)
    distances = np.asarray(distances).astype(np.float32)
    counts = np.asarray(counts).astype(np.float64)
    nq = labels.shape[0]
    per_query = labels[0].nbytes + distances[0].nbytes + counts[0].nbytes + 8 if nq else 1
    budget = DUMP_LIMIT_BYTES - 4 * NPY_HEADER_BYTES
    out = {"labels": labels, "distances": distances, "counts": counts}
    if nq * per_query > budget:
        rows = np.sort(np.random.default_rng(SEED).choice(nq, budget // per_query, replace=False))
        out = {name: a[rows] for name, a in out.items()}
        out["query_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def ncu_traffic_ratio(kernel_key: str):
    """DRAM bytes / algorithmic bytes of a kernel from the committed ncu captures (profiles/ncu_summary.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            return float(json.load(f)[kernel_key]["traffic_over_algorithmic"])
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tf_burst": float(d["bf16_tflops"]),
                "tf_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0,
                "source": "fallback (B200_PROFILING.md: 6.65 TB/s, 1.59 PF burst, ~1.4 PF sustained)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def cpu_arm(args, steps, warmup, rows_total, budget_s):
    """The reference arm / cpu_baseline: the oracle port (threaded SIMD exact scan, oracle/cpu_scan.c)
    on the host cores.  Every step scans a bounded SAMPLE of the corpus for the whole query batch; the
    sample is sized from a probe step so that warmup + steps fit `budget_s`, and the time is scaled
    linearly to the full corpus (a scan is O(rows))."""
    from oracle import oracle as O

    threads = O.cpu_threads()
    qs = O.make_queries(SEED, SEED + 1, args.batch, rows_total)
    probe_rows = min(200_000, rows_total)
    stored = O.synth_rows_f16(SEED, 0, probe_rows)
    O.cpu_scan_f16(stored, None, qs, args.k, threads=threads)  # page in, spin up the threads
    t0 = time.perf_counter()
    O.cpu_scan_f16(stored, None, qs, args.k, threads=threads)
    per_row = (time.perf_counter() - t0) / probe_rows
    sample = int(min(rows_total, args.cpu_sample_rows, max(50_000, budget_s / ((steps + warmup) * per_row))))
    if sample > probe_rows:
        stored = O.synth_rows_f16(SEED, 0, sample)
    else:
        sample = probe_rows
    times = []
    for s_ in range(warmup + steps):
        t0 = time.perf_counter()
        last = O.cpu_scan_f16(stored, None, qs, args.k, threads=threads)
        dt = time.perf_counter() - t0
        if s_ >= warmup:
            times.append(dt)
    scale = rows_total / sample
    step_s = statistics.mean(times) * scale
    return {
        "value": args.batch / step_s, "unit": "queries/s", "cores": threads, "kind": "port",
        "sample": f"{sample} of {rows_total} rows per step (oracle/cpu_scan.c, {threads} threads), "
                  f"time scaled x{scale:.1f} (a scan is linear in rows); {steps} timed steps of batch {args.batch} after {warmup} warm-up",
        "ms_per_step": statistics.mean(times) * 1e3,            # what a step really took here (over the sample)
        "ms_per_step_scaled_to_full_corpus": step_s * 1e3,     # what `value` is computed from
        "sample_rows": sample, "scale": scale,
        "last_step": last[:3],  # (labels, distances, counts) of the last timed step, over the sample
    }


def hnsw_arm(k_list=(10, 20)):
    """The reference's KIND of index, timed live on this box's host cores: an HNSW restatement with USearch's
    defaults (NOT USearch 0.22.3 -- that crate is not vendored and there is no cargo here; see
    oracle/hnsw_restatement.c) over BASELINE config C1 (100k f32 vectors, single queries), one search thread
    (the reference's model, src/bin/dawnsearch.rs:76-78) and all threads, with recall@k against the exact
    answer -- on the isotropic synthetic corpus and on a clustered, low-intrinsic-dimension one."""
    from oracle import oracle as O

    threads = O.cpu_threads()
    out = {"index": "HNSW restatement (NOT USearch 0.22.3): M=16, M0=32, efConstruction=128, efSearch=64, IP on f32",
           "host_threads": threads, "corpora": {}}
    nq = 256
    for name, n in (("isotropic_100k", 100_000), ("clustered_50k", 50_000)):
        if name.startswith("iso"):
            rows = np.concatenate([O.np_synth_rows_f32(SEED, i, min(20000, n - i)) for i in range(0, n, 20000)])
            qs = O.make_queries(SEED, SEED + 1, nq, n)
        else:
            rows = np.concatenate([O.np_clustered_rows_f32(SEED, i, min(10000, n - i)) for i in range(0, n, 10000)])
            qs = O.np_clustered_rows_f32(SEED, 1_000_000_000, nq)
        labels = np.arange(1, n + 1, dtype=np.uint64)
        t0 = time.perf_counter()
        h = O.Hnsw(16, 128, 64, 1)
        h.add_batch(labels, rows)
        build_s = time.perf_counter() - t0
        ent = {"rows": n, "queries": nq, "build_s_one_thread": round(build_s, 1),
               "add_us_per_vector": round(build_s / n * 1e6, 1)}
        stored16 = rows.astype(np.float16)
        for k in k_list:
            truth = np.stack([O.search_f32(rows, labels, q, k)[0] for q in qs[:64]])  # exact over the f32 vectors
            l1, _, _ = h.search_batch(qs[:64], k, 1)
            recall = float(np.mean([len(set(a.tolist()) & set(b.tolist())) / k for a, b in zip(l1, truth)]))
            lat = []
            for q in qs:
                t1 = time.perf_counter()
                h.search_batch(q[None, :], k, 1)
                lat.append(time.perf_counter() - t1)
            t1 = time.perf_counter()
            h.search_batch(qs, k, threads)
            mt = time.perf_counter() - t1
            ent[f"k{k}"] = {"recall_at_k": round(recall, 4), "p50_us_one_thread": round(statistics.median(lat) * 1e6, 1),
                            "qps_one_thread": round(1.0 / statistics.mean(lat), 1),
                            "qps_all_threads": round(nq / mt, 1)}
        # the exact CPU scan on the same corpus, one query at a time (what "exact" costs at the reference's scale)
        lat = []
        for q in qs[:32]:
            t1 = time.perf_counter()
            O.cpu_scan_f16(stored16, labels, q[None, :], 10, threads=threads)
            lat.append(time.perf_counter() - t1)
        ent["cpu_exact_scan_p50_us_all_threads"] = round(statistics.median(lat) * 1e6, 1)
        out["corpora"][name] = ent
    return out


def workload_name(args):
    return (f"exact top-{args.k} over {args.rows} x 384 {'fp16' if args.scalar == 'f16' else 'int8 (+f32 scale per vector)'} "
            f"(synthetic unit vectors), batch {args.batch} "
            f"per step, corpus sharded by id range over {args.gpus} GPU(s)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)  # as given: the driver compares step counts
    r = cpu_arm(args, steps, warmup, args.rows, args.cpu_budget_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"],
        "unit": "queries/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": r["ms_per_step"], "ms_per_step_scaled_to_full_corpus": r["ms_per_step_scaled_to_full_corpus"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 accumulate over fp16 storage", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows": args.rows, "batch": args.batch, "k": args.k,
                   "sample_rows_per_step": r["sample_rows"], "sample_scale": r["scale"],
                   "timing": "ms_per_step is the measured time of one step over the sample; `value` = batch / "
                             "(ms_per_step x sample_scale): the whole-corpus rate a linear scan implies",
                   "note": "the reference's USearch 0.22.3 path cannot be built here (no cargo, crate not vendored); "
                           "`value` is the CPU exact-scan port on all host threads over a bounded sample, scaled; the "
                           "reference's kind of (approximate) index is timed live under `hnsw_stand_in`"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_hnsw:
        line["hnsw_stand_in"] = hnsw_arm()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *r["last_step"])
    print_json(line)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from dawnsearch_b200 import synth as O  # workload generator (numpy twin of the device generator)
    from dawnsearch_b200.sharded import ResultBlock, ShardedIndex, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    first, n_local = shard_range(rank, world, args.rows)
    row_bytes = ROW_BYTES if args.scalar == "f16" else 388  # i8: 384 B + f32 scale
    sh = ShardedIndex(local, max(n_local, 1), quantization=0 if args.scalar == "f16" else 1)
    # fp16 corpus + int8 shadow (library option "shadow_i8", +388 B per row): batches are FILTERED on the int8 copy by the int8
    # tensor cores and every candidate is re-scored on the fp16 rows -- the answers are the exact top-k over the fp16 vectors,
    # bit for bit (the parity check below runs with the same option), at half the corpus bytes and twice the MMA rate.
    shadow = args.scalar == "f16" and not args.no_shadow
    if shadow:
        sh.index.set_option("shadow_i8", 1)
    t0 = time.perf_counter()
    sh.index.add_synthetic(SEED, first, n_local)
    fill_s = time.perf_counter() - t0

    B, k, K, W = args.batch, args.k, args.steps, args.warmup
    # a pool of distinct query batches, cycled (fresh queries every step)
    n_pool = min(K + W, 8)
    pool_host = [O.make_queries(SEED, SEED + 1 + i, B, args.rows, planted_fraction=0.25) for i in range(n_pool)]
    pool_dev = [torch.from_numpy(q).to(dev) for q in pool_host]

    e2e_esc = [0]  # queries re-run exactly by ShardedIndex.search (N > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_device(queries_dev, kk, steps, warm, sample_clocks=False):
        """Device-resident timing: CUDA events on the launching stream + the library's own per-kernel events.
        Also returns the result block of the last step (a workspace buffer the next search of that shape overwrites)."""
        # back-to-back batches: the exchange of batch i overlaps the search of batch i+1 (not worth it
        # for single queries, where the side-stream bookkeeping costs more than the 12 us exchange)
        pipe = world > 1 and queries_dev[0].shape[0] >= 16
        for s in range(warm):
            sh.search_device(queries_dev[s % len(queries_dev)], kk, pipelined=pipe)
        sh.wait_results()
        barrier()
        sh.index.set_profiling(True)
        sh.index.profile(reset=True)
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record()
        for s in range(steps):
            last = sh.search_device(queries_dev[(warm + s) % len(queries_dev)], kk, pipelined=pipe)
            if s == steps - 1:
                sh.wait_results()  # the last event must cover the last batch's exchange + merge
            ev[s + 1].record()
        barrier()
        clocks = sampler.stop() if sampler else None
        total_ms = allmax(ev[0].elapsed_time(ev[steps]))
        step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        prof = sh.index.profile(reset=True)
        prof["device_uncertified_all_ranks"] = allsum(prof["device_uncertified"])
        sh.index.set_profiling(False)
        return total_ms, step_ms, prof, clocks, last

    def e2e_call(q, kk):
        if world == 1:
            return sh.index.search_batch(q, kk)
        r = sh.search(q, kk)
        e2e_esc[0] += sh.last_search_escalated
        return r

    def timed_e2e(queries_host, kk, steps, warm):
        for s in range(warm):
            e2e_call(queries_host[s % len(queries_host)], kk)
        barrier()
        lat = []
        t0 = time.perf_counter()
        for s in range(steps):
            t1 = time.perf_counter()
            e2e_call(queries_host[(warm + s) % len(queries_host)], kk)
            lat.append((time.perf_counter() - t1) * 1e3)
        barrier()
        return allmax(time.perf_counter() - t0), lat

    def roofline_of(prof, batch, peaks):
        """Roofline of the dominant kernel of a device-resident run."""
        if prof["gemm_batches"] and batch < 128:
            # one query tile: the rounds stream the corpus (its int8 shadow, or the int8 corpus) once per batch -> HBM-bound
            gms = prof["gemm_ms"] / int(prof["gemm_batches"])
            rb = 388 if (args.scalar == "i8" or prof.get("shadow_batches")) else row_bytes
            algo = n_local * rb
            ach = algo / (gms / 1e3) / 1e9
            ratio = ncu_traffic_ratio("gemm_i8_topk_kernel<2> final round" if rb == 388 else "gemm_topk_kernel<2> final round")
            return {"bound": "hbm", "kernel": ("gemm_i8_topk_kernel<1> (one query tile; all rounds of a batch incl. the exact re-score selects)"
                                               + (" over the int8 shadow of the fp16 corpus" if prof.get("shadow_batches") else ""))
                                              if rb == 388 else "gemm_topk_kernel<1> (one query tile; all rounds of a batch incl. select)",
                    "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                    "traffic": ratio * algo if ratio else None,
                    "traffic_note": "DRAM ratio of the CTA-pair kernel's capture (profiles/ncu_summary.json) x this batch's algorithmic bytes",
                    "peak_source": peaks["source"] + " hbm_gbs", "frac_of_nominal_8TBs": ach / 8000.0,
                    "algorithmic_bytes_per_batch": algo, "avg_batch_ms": gms, "avg_launch_ms": gms, "batches_timed": int(prof["gemm_batches"])}
        if prof["gemm_batches"]:
            gms = prof["gemm_ms"] / int(prof["gemm_batches"])
            flops = 2.0 * batch * n_local * DIM
            ach = flops / (gms / 1e3) / 1e12
            if args.scalar == "i8" or prof.get("shadow_batches"):
                # int8 tensor path (tcgen05 kind::i8): MEASURED_PEAKS.json holds no int8 figure; the int8 pipe is specified at
                # twice the bf16 rate (4.5 vs 2.25 POP/s dense), so the denominator is 2 x the measured sustained bf16 peak
                peak = 2.0 * peaks["tf_sustained"]
                ratio = ncu_traffic_ratio("gemm_i8_topk_kernel<2> final round")
                i8_bytes = 388  # what the int8 kernel streams per row (the shadow copy of an fp16 corpus, or the int8 corpus itself)
                return {"bound": "tensor", "kernel": "gemm_i8_topk_kernel (tcgen05 kind::i8; all rounds of a batch incl. the exact re-score selects)"
                                                     + (" over the int8 shadow of the fp16 corpus" if args.scalar == "f16" else ""),
                        "achieved": ach, "peak": peak, "unit": "TOP/s (int8)", "frac": ach / peak,
                        "traffic": ratio * n_local * i8_bytes if ratio else None,
                        "peak_source": "2 x " + peaks["source"] + " bf16_tflops_sustained (no measured int8 peak on this pool; the int8 pipe is rated at 2x bf16)",
                        "frac_of_nominal_4500": ach / 4500.0, "algorithmic_ops_per_batch": flops, "avg_batch_ms": gms,
                        "corpus_stream_gbps": n_local * i8_bytes / (gms / 1e3) / 1e9}
            ratio = ncu_traffic_ratio("gemm_topk_kernel<2> final round")
            return {"bound": "tensor", "kernel": "gemm_topk_kernel (tcgen05; all rounds of a batch incl. select)",
                    "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                    "frac": ach / peaks["tf_sustained"],
                    "traffic": ratio * n_local * row_bytes if ratio else None,
                    "traffic_note": "DRAM bytes per batch = ncu dram bytes / corpus bytes of the captured round "
                                    "(profiles/ncu_summary.json) x this shard's corpus bytes",
                    "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step)",
                    "frac_of_burst_peak": ach / peaks["tf_burst"], "frac_of_nominal_2250": ach / 2250.0,
                    "algorithmic_flops_per_batch": flops, "avg_batch_ms": gms,
                    "corpus_stream_gbps": n_local * row_bytes / (gms / 1e3) / 1e9}
        launches = max(int(prof["scan_launches"]), 1)
        sms = prof["scan_ms"] / launches
        algo = n_local * row_bytes
        ach = algo / (sms / 1e3) / 1e9 if sms > 0 else 0.0
        ratio = ncu_traffic_ratio("scan_topk_f16_kernel<1>" if args.scalar == "f16" else "scan_topk_i8_kernel<1>")
        return {"bound": "hbm", "kernel": "scan_topk_f16_kernel" if args.scalar == "f16" else "scan_topk_i8_kernel", "achieved": ach, "peak": peaks["hbm"],
                "unit": "GB/s", "frac": ach / peaks["hbm"], "traffic": ratio * algo if ratio else None,
                "traffic_note": "ncu dram bytes / algorithmic bytes of the captured launch (profiles/ncu_summary.json) x this launch's algorithmic bytes",
                "peak_source": peaks["source"] + " hbm_gbs", "frac_of_nominal_8TBs": ach / 8000.0,
                "algorithmic_bytes_per_launch": algo, "avg_launch_ms": sms, "launches_timed": int(prof["scan_launches"])}

    peaks = measured_peaks()

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- parity check, BEFORE any timing: the N-rank search path against the CPU oracle -------------
    # (oracle/ is used here as the checker only.)  A sub-corpus of <= --parity-rows rows is sharded over the
    # same N ranks by the same rule; 64 queries go through the host path (ShardedIndex.search: local exact
    # top-k, packed all-gather, device merge, certificate-driven re-runs), 1 query through the single-query
    # path, and the same 64 through the device-resident pipelined path that `value` times.  Rank 0 compares
    # labels and distance BITS with oracle.cpu_scan_f16 / search_i8.
    parity = None
    if not args.no_parity_check:
        from oracle import oracle as CK  # checker only

        p_rows = min(args.rows, args.parity_rows if args.scalar == "f16" else min(args.parity_rows, 200_000))
        pf, pn = shard_range(rank, world, p_rows)
        shp = ShardedIndex(local, max(pn, 1), quantization=0 if args.scalar == "f16" else 1)
        if shadow:
            shp.index.set_option("shadow_i8", 1)
        shp.index.add_synthetic(SEED, pf, pn)
        pq = O.make_queries(SEED, SEED + 99, 64, p_rows, planted_fraction=0.25)
        got = shp.search(pq, k)
        got1 = shp.search(pq[:1], k)
        esc = allsum(shp.last_search_escalated)
        d_pq = torch.from_numpy(pq).to(dev)
        blk_dev = shp.search_device(d_pq, k, pipelined=world > 1)
        shp.wait_results()
        torch.cuda.synchronize()
        dl, dd, dc = ResultBlock(64, k).views(blk_dev.cpu())
        pprof = shp.index.profile()
        dev_unc = allsum(pprof["device_uncertified"])
        shadow_used = allsum(pprof["shadow_batches"])
        if rank == 0:
            if args.scalar == "f16":
                stored = CK.synth_rows_f16(SEED, 0, p_rows)
                wl, wd, wc, _ = CK.cpu_scan_f16(stored, None, pq, k)
            else:
                rows32 = np.concatenate([CK.np_synth_rows_f32(SEED, i, min(20000, p_rows - i)) for i in range(0, p_rows, 20000)])
                q8, sc = CK.store_i8(rows32)
                lab = np.arange(1, p_rows + 1, dtype=np.uint64)
                res = [CK.search_i8(q8, sc, lab, q, k) for q in pq]
                wl = np.stack([r[0] for r in res])
                wd = np.stack([r[1] for r in res])
                wc = np.full(64, k)
            same_host = bool((got[2] == wc).all() and (got[0] == wl).all() and (got[1].view(np.uint32) == wd.view(np.uint32)).all())
            same_one = bool((got1[0][0] == wl[0]).all() and (got1[1][0].view(np.uint32) == wd[0].view(np.uint32)).all())
            same_dev = bool((dl.numpy().astype(np.uint64) == wl).all() and (dd.numpy().view(np.uint32) == wd.view(np.uint32)).all())
            parity = {"n_ranks": world, "rows": p_rows, "queries": 64, "k": k,
                      "bit_identical": same_host and same_one and same_dev,
                      "host_path_batch64": same_host, "host_path_single_query": same_one, "device_pipelined_path": same_dev,
                      "escalated_to_exact_scan": int(esc), "device_path_uncertified": int(dev_unc),
                      "batches_through_the_int8_shadow_all_ranks": int(shadow_used),
                      "checker": "oracle/cpu_scan.c dawn_cpu_scan_f16" if args.scalar == "f16" else "oracle/dawn_oracle.c dawn_oracle_search_i8"}
            assert parity["bit_identical"], f"parity check failed: {parity}"
        shp.close()
        del shp

    # ---- latency configuration: one query per step -----------------------------------------
    # (measured BEFORE the throughput run: that one leaves the chip on its 1000 W power cap for seconds,
    #  and single-query latency is a separate workload, not a tail of it)
    batch1 = None
    if args.latency_steps > 0 and B != 1:
        q1_host = [pool_host[0][i:i + 1] for i in range(min(B, 16))]
        q1_dev = [pool_dev[0][i:i + 1] for i in range(min(B, 16))]
        t_ms, s_ms, p1, _, _ = timed_device(q1_dev, k, args.latency_steps, 20)
        e_s, l1 = timed_e2e(q1_host, k, args.latency_steps, 20)
        l1s = sorted(l1)
        batch1 = {"qps_device": args.latency_steps / (t_ms / 1e3), "qps_e2e": args.latency_steps / e_s,
                  "latency_ms": {"device_p50": statistics.median(s_ms), "device_max": max(s_ms),
                                 "e2e_p50": statistics.median(l1), "e2e_p99": l1s[min(len(l1s) - 1, int(0.99 * len(l1s)))]},
                  "roofline": roofline_of(p1, 1, peaks)}

    # ---- main workload -------------------------------------------------------------------
    total_ms, step_ms, prof, clocks, last_block = timed_device(pool_dev, k, K, W, sample_clocks=True)
    last_step = [a.numpy() for a in ResultBlock(B, k).views(last_block.cpu())] if args.dump_outputs and rank == 0 else None
    value = B * K / (total_ms / 1e3)
    e2e_esc[0] = 0
    e2e_s, lat = timed_e2e(pool_host, k, K, min(W, 3))
    prof_e2e = sh.index.profile(reset=True)
    e2e_escalated = int(allsum(prof_e2e["escalations"] + e2e_esc[0]))

    # ---- the same batches on the fp16 tensor-core tiles (shadow off), a few steps, for the record ----
    fp16_tiles = None
    if shadow and prof.get("shadow_batches"):
        sh.index.set_option("shadow_i8", 0)
        t_ms, _, pf16, _, _ = timed_device(pool_dev, k, min(K, 5), 2)
        sh.index.set_option("shadow_i8", 1)
        fp16_tiles = {"value": B * min(K, 5) / (t_ms / 1e3), "unit": "queries/s", "ms_per_step": t_ms / min(K, 5), "steps": min(K, 5),
                      "note": "option shadow_i8 off: gemm_topk_kernel (tcgen05 kind::f16 tiles straight from the fp16 rows)",
                      "roofline": roofline_of(pf16, B, peaks)}

    # sanity: a planted neighbour must come back first (a wrong kernel cannot post a number)
    planted = O.planted_rows(SEED + 1, B, args.rows, 0.25)
    if len(planted):
        probe = e2e_call(pool_host[0], k)
        assert int(probe[0][0][0]) == int(planted[0]) + 1, "planted neighbour not returned first"
        sh.index.profile(reset=True)

    # ---- optional sweep over (batch, k): device-resident, 3 warm-up + 10 timed steps each ---
    sweep = []
    if args.sweep:
        for item in args.sweep.split(","):
            sb, sk = (int(x) for x in item.split(":")) if ":" in item else (int(item), k)
            q = [torch.from_numpy(O.make_queries(SEED, SEED + 5, sb, args.rows)).to(dev)]
            t_ms, _, p, _, _ = timed_device(q, sk, 10, 3)
            ms = t_ms / 10
            ent = {"batch": sb, "k": sk, "qps": sb / (ms / 1e3), "ms_per_step": ms,
                   "finalize_ms": p["finalize_ms"] / max(int(p["finalize_launches"]), 1)}
            r = roofline_of(p, sb, peaks)
            if p["gemm_batches"] and r["bound"] == "hbm":
                ent.update({"path": "tcgen05 (int8 shadow)" if p.get("shadow_batches") else "tcgen05", "gemm_ms": r["avg_batch_ms"],
                            "corpus_gbps": r["achieved"]})
            elif p["gemm_batches"]:
                ent.update({"path": "tcgen05 (int8 shadow)" if p.get("shadow_batches") else "tcgen05", "gemm_ms": r["avg_batch_ms"],
                            "tflops": r["achieved"], "corpus_gbps": r["corpus_stream_gbps"]})
            else:
                ent.update({"path": "scan", "scan_passes": int(p["scan_launches"]) // 10,
                            "scan_ms_per_pass": r["avg_launch_ms"], "scan_gbps": r["achieved"]})
            sweep.append(ent)

    if rank == 0:
        lat_sorted = sorted(lat)
        line = {
            "metric": METRIC, "value": value, "unit": "queries/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": ("s8 x s8 -> s32 filter on an int8 shadow (tensor cores) / f32 scan, exact f32 re-score over the fp16 rows" if shadow else
                                                          "f16 x f16 -> f32 (tensor cores) / f32 scan, exact f32 re-score" if args.scalar == "f16" else
                                                          "s8 x s8 -> s32 (tensor cores) / dp4a scan, exact f32 re-score"),
            "data": "synthetic",
            "config": {"workload": workload_name(args), "rows": args.rows, "rows_per_gpu": n_local,
                       "batch": B, "k": k, "l2": "inputs larger than L2 (corpus shard >> 126 MB), no flush",
                       "multi_gpu": ("device-resident `value`: the all-gather + merge of batch i run on a side stream "
                                     "while batch i+1 is searched; e2e: synchronous per call") if world > 1 else None,
                       "int8_shadow": ("on: +388 B per row beside the 768 B fp16 row (library option shadow_i8); filter only, "
                                       "answers are exact over the fp16 rows") if shadow else None,
                       "corpus_fill_s": round(fill_s, 3)},
            "latency_ms": {"device_step_p50": statistics.median(step_ms), "device_step_max": max(step_ms),
                           "e2e_step_p50": statistics.median(lat),
                           "e2e_step_p99": lat_sorted[min(len(lat) - 1, int(0.99 * len(lat)))]},
            "e2e": {"value": B * K / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": B * DIM * 4,
                    "d2h_bytes_per_step": B * k * 12 + B * 8 + 4, "ms_per_step": e2e_s / K * 1e3},
            "gpu_launches": int(prof["kernel_launches"]) + (K if world > 1 else 0),  # + one merge kernel per step at N > 1
            "roofline": roofline_of(prof, B, peaks),
            "clocks": clocks,
            "exactness": {"value_leg_uncertified_queries": int(prof["device_uncertified_all_ranks"]),
                          "e2e_leg_uncertified_queries": int(prof_e2e["uncertified"]),
                          "e2e_leg_escalated_to_exact_scan": e2e_escalated,
                          "note": "value leg (device-resident, cannot escalate): (rank, query) results written without an "
                                  "exactness certificate, counted on the device by every finalize launch, summed over ranks; "
                                  "e2e leg: any query whose certificate fails on any shard is re-run through the exact f32 "
                                  "scan before the merge (N = 1: inside dawn_index_search_batch; N > 1: ShardedIndex.search)"},
            "parity_check": parity,
        }
        if fp16_tiles:
            line["fp16_tensor_path"] = fp16_tiles
        if batch1:
            line["batch1"] = batch1
        if sweep:
            line["batch_sweep"] = sweep
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_arm(args, steps=2, warmup=1, rows_total=args.rows, budget_s=20.0)
            line["cpu_baseline"] = {kk: r[kk] for kk in ("value", "unit", "cores", "kind", "sample")}
        if last_step:
            dump_outputs(args.dump_outputs, *last_step)
        print_json(line)
    sh.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_multi(args):
    """--front multi: ONE process drives all --gpus through the C ABI (dawn_multi_*: shards, NCCL all-gather
    and merge inside libdawn_b200.so) -- the path a one-process Rust binary would call.  Host buffers in and
    out on every call, so every number here is end to end; `value` is the device-side share of it (CUDA events:
    slowest shard's local search + exchange/merge on the first device)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import dawnsearch_b200 as D
    from dawnsearch_b200 import synth as O

    G, B, k, K, W = args.gpus, args.batch, args.k, args.steps, args.warmup
    scalar = 0 if args.scalar == "f16" else 1
    row_bytes = ROW_BYTES if args.scalar == "f16" else 388
    shadow = args.scalar == "f16" and not args.no_shadow  # see run(): int8 shadow of the fp16 corpus, filter only
    parity = None
    if not args.no_parity_check:
        from oracle import oracle as CK  # checker only

        p_rows = min(args.rows, args.parity_rows)
        with D.MultiIndex(list(range(G)), quantization=0) as mp:
            if shadow:
                mp.set_option("shadow_i8", 1)
            mp.reserve(p_rows)
            mp.add_synthetic(SEED, 0, p_rows)
            pq = O.make_queries(SEED, SEED + 99, 64, p_rows, planted_fraction=0.25)
            stored = CK.synth_rows_f16(SEED, 0, p_rows)
            wl, wd, wc, _ = CK.cpu_scan_f16(stored, None, pq, k)
            ok = {}
            for name, mode in (("nccl", 2), ("peer", 1)) if G > 1 else (("peer", 1),):
                mp.set_option("exchange", mode)
                gl, gd, gc = mp.search_batch(pq, k)
                m1 = mp.search(pq[0], k)
                ok[name] = bool((gc == wc).all() and (gl == wl).all() and (gd.view(np.uint32) == wd.view(np.uint32)).all()
                                and (m1.labels == wl[0]).all())
            parity = {"n_shards": G, "rows": p_rows, "queries": 64, "k": k, "bit_identical": all(ok.values()),
                      "exchange_modes": ok, "stats": mp.stats(), "checker": "oracle/cpu_scan.c dawn_cpu_scan_f16"}
            assert parity["bit_identical"], parity
    m = D.MultiIndex(list(range(G)), quantization=scalar)
    if shadow:
        m.set_option("shadow_i8", 1)
    m.reserve(args.rows)
    t0 = time.perf_counter()
    m.add_synthetic(SEED, 0, args.rows)
    fill_s = time.perf_counter() - t0
    n_pool = min(K + W, 8)
    pool = [O.make_queries(SEED, SEED + 1 + i, B, args.rows, planted_fraction=0.25) for i in range(n_pool)]

    def timed(queries, steps, warm):
        for s_ in range(warm):
            m.search_batch(queries[s_ % len(queries)], k)
        lat, dev_ms, xch_ms = [], [], []
        t0 = time.perf_counter()
        for s_ in range(steps):
            t1 = time.perf_counter()
            last = m.search_batch(queries[(warm + s_) % len(queries)], k)
            lat.append((time.perf_counter() - t1) * 1e3)
            st = m.stats()
            dev_ms.append(st["last_search_ms"] + st["last_exchange_ms"])
            xch_ms.append(st["last_exchange_ms"])
        return time.perf_counter() - t0, lat, dev_ms, xch_ms, last

    out_modes = {}
    for name, mode in ((("nccl", 2), ("peer", 1)) if G > 1 else (("peer", 1),)):
        m.set_option("exchange", mode)
        q1 = [pool[0][i:i + 1] for i in range(min(B, 16))]
        w1, l1, d1, x1, _ = timed(q1, max(args.latency_steps, 20), 20)
        out_modes[name] = {"batch1_e2e_p50_ms": statistics.median(l1), "batch1_e2e_p99_ms": sorted(l1)[int(0.99 * len(l1))],
                           "batch1_device_p50_ms": statistics.median(d1), "batch1_exchange_merge_p50_ms": statistics.median(x1)}
    m.set_option("exchange", 0)
    sampler = ClockSampler(0)
    sampler.start()
    wall, lat, dev_ms, xch_ms, last_step = timed(pool, K, W)
    clocks = sampler.stop()
    st = m.stats()
    probe = m.search_batch(pool[0], k)
    planted = O.planted_rows(SEED + 1, B, args.rows, 0.25)
    if len(planted):
        assert int(probe[0][0][0]) == int(planted[0]) + 1, "planted neighbour not returned first"
    line = {
        "metric": METRIC, "value": B * K / (sum(dev_ms) / 1e3), "unit": "queries/s", "n_gpus": G, "steps": K, "warmup": W,
        "ms_per_step": sum(dev_ms) / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": ("s8 x s8 -> s32 filter on an int8 shadow (tensor cores) / f32 scan, exact f32 re-score over the fp16 rows" if shadow
                  else "f16 x f16 -> f32 (tensor cores) / f32 scan, exact f32 re-score"), "data": "synthetic",
        "config": {"workload": workload_name(args), "front": "multi: one process, dawn_multi_* C ABI, NCCL all-gather inside the library",
                   "rows": args.rows, "rows_per_gpu": (args.rows + G - 1) // G, "batch": B, "k": k,
                   "l2": "inputs larger than L2 (corpus shard >> 126 MB), no flush", "corpus_fill_s": round(fill_s, 3),
                   "value_is": "device share of the call: slowest shard's local search + exchange and merge on the first device (CUDA events)"},
        "e2e": {"value": B * K / wall, "unit": "queries/s", "h2d_bytes_per_step": B * DIM * 4 * G,
                "d2h_bytes_per_step": B * k * 12 + B * 4 + G * B * 4, "ms_per_step": wall / K * 1e3},
        "latency_ms": {"e2e_step_p50": statistics.median(lat), "device_step_p50": statistics.median(dev_ms),
                       "exchange_merge_p50": statistics.median(xch_ms)},
        "exchange_ab": out_modes, "multi_stats": st, "gpu_launches": int(st["kernel_launches"]),
        "roofline": {"bound": "tensor" if B >= 256 else "hbm", "note": "per-kernel rooflines are reported by the default front; "
                     "this front reports the whole call", "achieved": 2.0 * B * args.rows * DIM / (statistics.median(dev_ms) / 1e3) / 1e12 / G,
                     "unit": ("TOP/s (int8) per GPU (whole call); peak = 2 x measured sustained bf16" if (shadow or args.scalar == "i8")
                              else "TFLOP/s per GPU (whole call)"),
                     "peak": measured_peaks()["tf_sustained"] * (2.0 if (shadow or args.scalar == "i8") else 1.0),
                     "frac": 2.0 * B * args.rows * DIM / (statistics.median(dev_ms) / 1e3) / 1e12 / G /
                             (measured_peaks()["tf_sustained"] * (2.0 if (shadow or args.scalar == "i8") else 1.0)),
                     "traffic": None, "corpus_stream_gbps_per_gpu": args.rows / G * row_bytes / (statistics.median(dev_ms) / 1e3) / 1e9},
        "clocks": clocks, "parity_check": parity,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_step)
    print_json(line)
    m.close()


def main():
    args = parse()
    # Only the JSON line may reach stdout (NCCL and torchrun print banners there): park the real
    # stdout, point fd 1 at stderr while working, and restore it for the final print.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    line_holder = []
    global print_json
    def print_json(obj):
        line_holder.append(json.dumps(obj))
    try:
        if args.impl == "reference":
            run_reference(args)
        elif args.front == "multi":
            run_multi(args)
        else:
            run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for ln in line_holder:
        print(ln, flush=True)


if __name__ == "__main__":
    main()
