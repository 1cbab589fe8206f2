"""How often gemm_i8_topk_kernel's epilogue takes its slow path, per launch (round), for each setting of shadow_group_rows.
Needs the measurement build, which counts on the device (off in the shipped library):

    make -C dawnsearch_b200/csrc OUT=../lib_ab EXTRA=-DDAWN_COUNT_SLOW_PATH
    DAWN_B200_LIB=dawnsearch_b200/lib_ab/libdawn_b200.so python tools/slow_path_count.py [ROWS] [BATCH] [K] [GROUPS]

A warp-chunk is 32 queries (one epilogue warp) x 32 corpus columns; it takes the slow path (examine(): levels 2 and 3 of
the filter) when any of its queries passes level 1.  Also printed: the time of the first search after the option changed,
which includes rebuilding the shadow, next to the median of the searches after it."""
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import dawnsearch_b200 as D  # noqa: E402
from dawnsearch_b200 import synth  # noqa: E402

SEED = 0xDA5EA2C4
rows = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
batch = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
k = int(sys.argv[3]) if len(sys.argv) > 3 else 10
groups = [int(v) for v in sys.argv[4].split(",")] if len(sys.argv) > 4 else [1, 32]

L = D.load_library()
if not hasattr(L, "dawn_debug_slow_path_log"):
    sys.exit(f"{D.index.LIB_PATH} does not count the slow path: build it with EXTRA=-DDAWN_COUNT_SLOW_PATH (see above)")
L.dawn_debug_slow_path_log.argtypes = [C.POINTER(C.c_ulonglong), C.c_int, C.c_int]
L.dawn_debug_slow_path_log.restype = C.c_int
CAP = 4096
buf = (C.c_ulonglong * (4 * CAP))()


def read_log():
    n = L.dawn_debug_slow_path_log(buf, CAP, 1)
    if n < 0:
        sys.exit("reading the slow-path log failed")
    return [tuple(buf[4 * i:4 * i + 4]) for i in range(min(n, CAP))]


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


print(f"{rows} rows, batch {batch}, k {k}; {torch.cuda.get_device_name(0)}")
for g in groups:
    search()  # the previous setting's shadow is in place
    idx.set_option("shadow_group_rows", g)
    first = search()  # rebuilds the shadow
    rest = sorted(search() for _ in range(3))
    read_log()
    search()
    log = read_log()
    slow = sum(e[0] for e in log)
    chunks = sum(e[1] for e in log)
    print(f"shadow_group_rows {g}: first search after the change {first:.1f} ms (incl. the rebuild), then {rest[1]:.1f} ms")
    for i, (s, c, tiles, nq) in enumerate(log):
        print(f"  launch {i}: {tiles} tiles ({100.0 * tiles * 256 / rows:.1f} % of the rows), warp-chunks {c}, "
              f"slow path {s} = {100.0 * s / max(c, 1):.2f} %")
    print(f"  all launches: slow path {slow} of {chunks} warp-chunks = {100.0 * slow / max(chunks, 1):.2f} %", flush=True)
idx.close()
