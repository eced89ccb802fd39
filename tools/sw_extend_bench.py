"""BWA-MEM seed extension (sw_extend_batch) throughput on a B200, with its parity against the oracle and the oracle's
single-core rate.  Writes one JSON line; exits 1 on any mismatch.

Rates are in visited DP cells per second: the cells of ksw_extend2's inner loop, which the GPU counts and the oracle
counts too (a banded extension visits far fewer cells than q_len x t_len).  The jobs are BWA-like (sw.extension_jobs:
150-base reads, seeds of 19..50 bases, bwa mem's default scoring); a million of them is what BWA-MEM extends for a few
hundred thousand reads."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from oracle import ksw
from acc_genomics_b200 import sw


def card():
    """Name, power limit and max SM clock of GPU 0 (a read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                                   # the numbers still stand, without their card
        return dict(gpu=f"unknown ({e})")


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--jobs", type=int, default=1_000_000)
    ap.add_argument("--check", type=int, default=200_000, help="jobs compared with the oracle, field by field")
    ap.add_argument("--oracle-sample", type=int, default=20_000, help="jobs the oracle is timed on, one core")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    sc = sw.BWA_DEFAULTS
    args = (sc["mat"], sc["m"], sc["o_del"], sc["e_del"], sc["o_ins"], sc["e_ins"], sc["zdrop"])

    t0 = time.perf_counter()
    jobs = sw.extension_jobs(a.seed, a.jobs)
    gen_s = time.perf_counter() - t0
    ctx = sw.SmithWaterman(0)
    for _ in range(a.warmup):
        got = ctx.extend(jobs, *args)
    runs = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        got = ctx.extend(jobs, *args)
        py_ms = (time.perf_counter() - t0) * 1e3
        st = ctx.stats()
        runs.append((st["ms_kernel"], st["ms_total"], py_ms, st["cells"]))
    cells = runs[0][3]
    assert all(r[3] == cells for r in runs)
    ms_kernel = sorted(r[0] for r in runs)[len(runs) // 2]
    ms_call = sorted(r[1] for r in runs)[len(runs) // 2]
    ms_py = sorted(r[2] for r in runs)[len(runs) // 2]
    ctx.close()

    # parity: the first `check` jobs, on a few host threads (the oracle runs outside the GIL)
    n_check = min(a.check, len(jobs))
    parts = [(k, min(k + 10_000, n_check)) for k in range(0, n_check, 10_000)]
    with ThreadPoolExecutor(max(1, min(16, os.cpu_count() or 1))) as ex:
        res = list(ex.map(lambda p: ksw.extend_batch(jobs[p[0]:p[1]], sc["m"], sc["mat"], sc["o_del"], sc["e_del"],
                                                        sc["o_ins"], sc["e_ins"], sc["zdrop"]), parts))
    want = np.concatenate([r[0] for r in res]) if res else np.zeros((0, 6), np.int32)
    mismatches = int((got[:n_check] != want).any(axis=1).sum())

    # the oracle's rate on one core, on a seeded sample
    sample = sw.extension_jobs(a.seed + 1, a.oracle_sample)
    t0 = time.perf_counter()
    _, oc = ksw.extend_batch(sample, sc["m"], sc["mat"], sc["o_del"], sc["e_del"], sc["o_ins"], sc["e_ins"], sc["zdrop"])
    oracle_s = time.perf_counter() - t0

    rec = dict(metric="sw_extend_gcups_kernel", jobs=len(jobs), cells_visited=int(cells),
               cells_qlen_x_tlen=int(sum(len(q) * len(t) for q, t, *_ in jobs)),
               ms_kernel=round(ms_kernel, 3), ms_call=round(ms_call, 3), ms_python_call=round(ms_py, 3),
               gcups_kernel=round(cells / ms_kernel * 1e-6, 2), gcups_call=round(cells / ms_call * 1e-6, 2),
               jobs_per_s_call=round(len(jobs) / ms_call * 1e3),
               oracle_1core_gcups=round(int(oc.sum()) / oracle_s * 1e-9, 4), oracle_sample_jobs=len(sample),
               checked_jobs=n_check, mismatches=mismatches, reps=a.reps, warmup=a.warmup, generate_s=round(gen_s, 2),
               **card())
    line = json.dumps(rec)
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    return 1 if mismatches else 0


if __name__ == "__main__":
    sys.exit(main())
