"""File rates of dawn_multi_save / dawn_multi_load, and batch-1 search latency while a save runs.

    python tools/multi_persist_rate.py DIR ROWS SHARDS [REPEATS]

ROWS synthetic fp16 rows (dawn_multi_add_synthetic) on SHARDS shards: distinct devices when the box has that many, else
device 0 listed SHARDS times.  Prints, with the card's name and power limit:
  * save and load rates of the multi handle in GB/s of file bytes (host clock; both calls return after the last byte is on
    disk or on the device), median of REPEATS, the load into a fresh handle and into a reserved empty one (in place);
  * the same rows as SHARDS single indexes (dawn_index_save / _load), saved and loaded one after another;
  * batch-1 k = 10 search latency on the handle, idle and while a save runs (p50, p99, max), so one can see that a save
    does not hold searches for its duration.
DIR should be a tmpfs (/dev/shm) so that the numbers are the library's and not the disk's."""
import os
import shutil
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import dawnsearch_b200 as D  # noqa: E402
from dawnsearch_b200 import synth  # noqa: E402

SEED = 0xDA5EA2C4
if len(sys.argv) < 4:
    sys.exit(__doc__)
out_dir, rows, G = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
repeats = int(sys.argv[4]) if len(sys.argv) > 4 else 3
assert torch.cuda.is_available(), "multi_persist_rate.py measures on the GPU"
n_dev = torch.cuda.device_count()
devices = list(range(G)) if n_dev >= G else [0] * G
print(subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv"],
                     capture_output=True, text=True).stdout.strip())
os.makedirs(out_dir, exist_ok=True)
print(f"{rows} rows fp16 on {G} shards, devices {devices}; {out_dir}: {shutil.disk_usage(out_dir).free / 1e9:.1f} GB free")
path = os.path.join(out_dir, "multi.dawn")


def clock(fn):
    t = time.perf_counter()
    fn()
    return time.perf_counter() - t


def med(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def report(what, nbytes, secs):
    print(f"{what}: {nbytes / 1e9:.2f} GB, median {med(secs):.3f} s = {nbytes / med(secs) / 1e9:.2f} GB/s "
          f"(runs {', '.join(f'{s:.3f}' for s in secs)})", flush=True)


m = D.MultiIndex(devices)
m.reserve(rows)
m.add_synthetic(SEED, 0, rows)
qs = synth.make_queries(SEED, 3, 400, rows)
for q in qs[:20]:
    m.search_batch(q[None, :], 10)

saves = [clock(lambda: m.save(path)) for _ in range(repeats)]
nbytes = os.path.getsize(path)
report("dawn_multi_save", nbytes, saves)
loads, loads_in_place = [], []
for _ in range(repeats):
    with D.MultiIndex(devices) as m2:
        loads.append(clock(lambda: m2.load(path)))
    with D.MultiIndex(devices) as m2:
        m2.reserve(rows)
        loads_in_place.append(clock(lambda: m2.load(path)))
report("dawn_multi_load into a fresh handle", nbytes, loads)
report("dawn_multi_load into a reserved empty handle (in place)", nbytes, loads_in_place)


def latencies(n):
    out = []
    for i in range(n):
        t = time.perf_counter()
        m.search_batch(qs[i % len(qs)][None, :], 10)
        out.append((time.perf_counter() - t) * 1e3)
    return out


def lat_report(what, xs):
    xs = sorted(xs)
    print(f"batch-1 k=10 search {what}: {len(xs)} searches, p50 {xs[len(xs) // 2]:.3f} ms, "
          f"p99 {xs[min(len(xs) - 1, int(len(xs) * 0.99))]:.3f} ms, max {xs[-1]:.3f} ms", flush=True)


lat_report("idle", latencies(400))
during, done = [], threading.Event()
save_secs = []


def saver():
    save_secs.append(clock(lambda: m.save(path)))
    done.set()


th = threading.Thread(target=saver)
th.start()
while not done.is_set():
    t = time.perf_counter()
    m.search_batch(qs[len(during) % len(qs)][None, :], 10)
    during.append((time.perf_counter() - t) * 1e3)
th.join()
lat_report(f"during a save of {save_secs[0]:.3f} s", during)
m.close()
os.remove(path)

# the same rows as G single indexes, saved and then loaded one after another
per = -(-rows // G)
singles = []
for g in range(G):
    a = min(g * per, rows)
    idx = D.new_index(D.IndexOptions(device=devices[g]))
    idx.reserve(max(1, min(per, rows - a)))
    idx.add_synthetic(SEED, a, min(per, rows - a))
    singles.append(idx)
s_save, s_load = [], []
paths = [os.path.join(out_dir, f"single{g}.dawn") for g in range(G)]
for _ in range(repeats):
    s_save.append(sum(clock(lambda: idx.save(p)) for idx, p in zip(singles, paths)))
s_bytes = sum(os.path.getsize(p) for p in paths)
for idx in singles:
    idx.close()
for _ in range(repeats):
    t = 0.0
    for g, p in enumerate(paths):
        with D.new_index(D.IndexOptions(device=devices[g])) as idx:
            t += clock(lambda: idx.load(p))
    s_load.append(t)
report(f"{G} x dawn_index_save, one after another", s_bytes, s_save)
report(f"{G} x dawn_index_load, one after another", s_bytes, s_load)
for p in paths:
    os.remove(p)
