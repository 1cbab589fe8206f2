"""Cost of dawn_index_remove_batch on a big fp16 corpus with the int8 shadow on, and what a removal does to the search after it.

    python tools/remove_rate.py [ROWS] [REPEATS]

Prints, for ROWS synthetic rows (labels 1..ROWS): the host-clock time of remove_batch (it returns after the device is done) for
m = 1, 1,000 and 1,000,000 random present labels and for 1,000 absent labels (mark and scan only: nothing moves), and the
batch-1024 k = 10 search time (device API, host clock around a synchronised call, median of REPEATS) before and after those
removals, i.e. after about 1 % of the rows moved.  With a library built with EXTRA=-DDAWN_COUNT_SLOW_PATH (see
tools/slow_path_count.py) it also prints the share of the int8 filter's warp-chunks that took the slow path, per round, before
and after: the holes that received a donor are 32-row shadow groups with two scales."""
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dawnsearch_b200 as D  # noqa: E402
from dawnsearch_b200 import synth  # noqa: E402

SEED = 0xDA5EA2C4
rows = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 10
batch, k = 1024, 10

assert torch.cuda.is_available(), "remove_rate.py measures on the GPU"
if rows < 4 * (1_000_000 + 1_000 * repeats + repeats):
    sys.exit(f"ROWS must be at least 4x the {1_000_000 + 1_000 * repeats + repeats} labels the removals take")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv", "-i", "0"],
                     capture_output=True, text=True).stdout.strip())
L = D.load_library()
counting = hasattr(L, "dawn_debug_slow_path_log")
if counting:
    L.dawn_debug_slow_path_log.argtypes = [C.POINTER(C.c_ulonglong), C.c_int, C.c_int]
    L.dawn_debug_slow_path_log.restype = C.c_int
    CAP = 4096
    log_buf = (C.c_ulonglong * (4 * CAP))()

idx = D.new_index(D.IndexOptions(capacity=rows))
idx.add_synthetic(SEED, 0, rows)
idx.set_option("shadow_i8", 1)
dev = torch.device("cuda:0")
q = torch.from_numpy(synth.make_queries(SEED, 3, batch, rows)).to(dev)
Lb = torch.zeros((batch, k), dtype=torch.int64, device=dev)
Db = torch.zeros((batch, k), dtype=torch.float32, device=dev)
Cn = torch.zeros(batch, dtype=torch.int32, device=dev)
Fl = torch.zeros(batch, dtype=torch.int32, device=dev)


def search():
    t = time.perf_counter()
    idx.search_device(q.data_ptr(), batch, k, Lb.data_ptr(), Db.data_ptr(), Cn.data_ptr(), Fl.data_ptr(), 0)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3


def search_report(when):
    for _ in range(3):
        search()
    t = sorted(search() for _ in range(repeats))
    shadow = idx.profile(reset=True)["shadow_batches"]
    print(f"search {when}: batch {batch} k {k} over {idx.size()} rows: median {t[len(t) // 2]:.2f} ms "
          f"(min {t[0]:.2f}, max {t[-1]:.2f}; {repeats} runs; shadow batches {shadow})", flush=True)
    if counting:
        L.dawn_debug_slow_path_log(log_buf, CAP, 1)
        search()
        n = min(L.dawn_debug_slow_path_log(log_buf, CAP, 1), CAP)
        log = [tuple(log_buf[4 * i:4 * i + 4]) for i in range(n)]
        for i, (s, c, tiles, _) in enumerate(log):
            print(f"  launch {i}: {tiles} tiles, warp-chunks {c}, slow path {s} = {100.0 * s / max(c, 1):.2f} %")
        print(f"  all launches: slow path {sum(e[0] for e in log)} of {sum(e[1] for e in log)} warp-chunks = "
              f"{100.0 * sum(e[0] for e in log) / max(sum(e[1] for e in log), 1):.2f} %", flush=True)


def timed_remove(labels):
    t = time.perf_counter()
    r = idx.remove_batch(labels)
    return (time.perf_counter() - t) * 1e3, r


print(f"{rows} rows, fp16 + int8 shadow; {torch.cuda.get_device_name(0)}")
search_report("before the removals")
rng = np.random.default_rng(1)
need = 1_000_000 + 1_000 * repeats + repeats  # distinct present labels the removals below take
pool = np.zeros(0, dtype=np.uint64)
while len(pool) < need:  # draws with replacement, repeats dropped (rows >= 4 * need, so this ends quickly)
    pool = np.unique(np.concatenate([pool, rng.integers(1, rows + 1, size=need, dtype=np.uint64)]))
pool = rng.permutation(pool)[:need]
at = 0
absent = np.arange(rows + 1, rows + 1001, dtype=np.uint64)
for m, reps in ((1, repeats), (1_000, repeats), (1_000_000, 1)):
    times = []
    for _ in range(reps):
        ms, r = timed_remove(pool[at:at + m])
        assert r == m, (r, m)
        at += m
        times.append(ms)
    times.sort()
    print(f"remove_batch m = {m}: median {times[len(times) // 2]:.3f} ms (min {times[0]:.3f}, max {times[-1]:.3f}; {reps} calls), "
          f"{idx.size()} rows left", flush=True)
times = sorted(timed_remove(absent)[0] for _ in range(repeats))
print(f"remove_batch m = 1000 absent labels (mark + scan, nothing moves): median {times[len(times) // 2]:.3f} ms "
      f"(min {times[0]:.3f}, max {times[-1]:.3f})", flush=True)
print(f"removed {rows - idx.size()} rows = {100.0 * (rows - idx.size()) / rows:.2f} %")
search_report("after the removals")
idx.close()
