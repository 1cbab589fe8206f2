"""`bench.py --impl reference` runs without a GPU (it times the CPU oracle port), so its JSON contract can be checked here:
one line, the driver's keys, the step counts as given, and rank > 0 exiting quietly under a multi-rank launch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0xDA5EA2C4  # bench.py's corpus and query seed


def run(extra, env=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "200000", "--batch", "64",
           "--steps", "2", "--warmup", "1", "--cpu-budget-s", "3", "--no-hnsw"] + extra
    return subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, **(env or {})), cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = run([])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["metric"].startswith("queries/sec") and "workload" in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    r = run(["--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def load_dump(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("labels", "distances", "counts")}


def check_dump_against_oracle(got, oracle, queries, rows, k):
    wl, wd, wc, _ = oracle.cpu_scan_f16(oracle.synth_rows_f16(SEED, 0, rows), None, queries, k)
    assert got["labels"].dtype == np.float64 and got["distances"].dtype == np.float32 and got["counts"].dtype == np.float64
    assert got["labels"].shape == got["distances"].shape == (len(queries), k) and got["counts"].shape == (len(queries),)
    assert (got["counts"] == wc).all() and (got["labels"] == wl.astype(np.float64)).all()
    assert (got["distances"].view(np.uint32) == wd.view(np.uint32)).all()


def test_reference_arm_dumps_its_last_step(tmp_path, oracle):
    """--dump-outputs: the last timed step's results, the same on every run with the same arguments."""
    dumps = []
    for i in range(2):
        r = run(["--dump-outputs", str(tmp_path / f"run{i}")])
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append(load_dump(tmp_path / f"run{i}"))
    # 200k rows: the arm's corpus sample is the whole corpus
    check_dump_against_oracle(dumps[0], oracle, oracle.make_queries(SEED, SEED + 1, 64, 200_000), 200_000, 10)
    for name, a in dumps[0].items():
        assert np.array_equal(a, dumps[1][name]), name


def test_steps_must_be_positive():
    r = run(["--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_default_path_dumps_its_last_step(tmp_path, oracle):
    rows, batch, steps, warmup = 200_000, 64, 3, 1
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(rows), "--batch", str(batch), "--steps", str(steps),
           "--warmup", str(warmup), "--latency-steps", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.splitlines()[-1])["steps"] == steps
    # the timed loop cycles a pool of min(steps + warmup, 8) query batches, the i-th drawn with query seed SEED + 1 + i
    last = (warmup + steps - 1) % min(steps + warmup, 8)
    queries = oracle.make_queries(SEED, SEED + 1 + last, batch, rows, planted_fraction=0.25)
    check_dump_against_oracle(load_dump(tmp_path), oracle, queries, rows, 10)
