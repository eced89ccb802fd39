"""Config 5 of BASELINE.json as a stream: regions of 100 reads x 40 haplotypes, length-bucketed by the planner, fed
through the multi-GPU work queue (pmm_pool_*) on every visible GPU -- whole regions per GPU, no collective.

    python tools/stream_cfg5.py [--scale 0.04] [--regions-per-job 25] [--contexts 3] [--mode exact|fast] [--check 2]

Prints one JSON line: pairs, cells, wall seconds, GCUPS end to end (host buffers in, float64 log10 out), per-device load.
"""
import argparse, json, os, sys, time
from collections import deque
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from acc_genomics_b200 import synth
from acc_genomics_b200.engine import PairHMMPool, concat_regions, load_library

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=float, default=0.04)
ap.add_argument("--regions-per-job", type=int, default=25)
ap.add_argument("--contexts", type=int, default=3)
ap.add_argument("--repeat", type=int, default=1, help="stream the same jobs this many times (longer timed region)")
ap.add_argument("--check", type=int, default=2, help="jobs to verify against the oracle afterwards")
ap.add_argument("--depth", type=int, default=0, help="jobs in flight (default: 2 per context, more for small jobs)")
args = ap.parse_args()

t0 = time.time()
regions = synth.config(5, scale=args.scale)
jobs = [regions[k:k + args.regions_per_job] for k in range(0, len(regions), args.regions_per_job)]
flat = [concat_regions(j) for j in jobs]
cells = sum(b.num_cells for b in regions); pairs = sum(b.num_pairs for b in regions)
print(f"[stream] {len(regions)} regions, {len(jobs)} jobs, {pairs} pairs, {cells / 1e9:.1f} Gcells, generated in {time.time() - t0:.1f}s", file=sys.stderr)

pool = PairHMMPool(contexts_per_device=args.contexts)
ndev = pool.num_devices
depth = args.depth or 2 * args.contexts * ndev * max(1, 25 // args.regions_per_job)


# one result buffer per job in flight (jobs repeat, and two jobs in flight must not share their output memory)
outs = [np.empty(max(f["pairs"] for f in flat), dtype=np.float64) for _ in range(depth + 1)]


def run(rep):
    live = deque(); nfb = 0; n = 0
    for _ in range(rep):
        for k in range(len(jobs)):
            if len(live) >= depth:
                nfb += pool.wait(live.popleft())[1]
            live.append(pool.submit(None, out=outs[n % (depth + 1)][: flat[k]["pairs"]], job=flat[k])); n += 1
    while live:
        nfb += pool.wait(live.popleft())[1]
    return nfb


run(1)                                     # warm-up: arenas grow to size, kernels load
t0 = time.perf_counter()
nfb = run(args.repeat)
wall = time.perf_counter() - t0
ok = None
if args.check:
    import oracle
    chk = oracle.reference() or oracle.port()
    ok = True
    for k in np.linspace(0, len(jobs) - 1, args.check).astype(int):
        want = np.concatenate([chk.batch(b, threads=os.cpu_count() or 1)[1].ravel() for b in jobs[k]])
        got = pool.wait(pool.submit(None, job=flat[k]))[0]
        ok &= bool(np.array_equal(want.view(np.uint64), got.view(np.uint64)))
print(json.dumps({"workload": synth.CONFIG_NAMES[5], "scale": args.scale, "regions": len(regions), "jobs": len(jobs) * args.repeat,
                  "pairs": pairs * args.repeat, "cells": cells * args.repeat, "n_gpus": ndev, "contexts_per_gpu": args.contexts,
                  "jobs_in_flight": depth, "wall_s": wall, "e2e_gcups": cells * args.repeat / wall * 1e-9, "fallback_pairs": nfb,
                  "bit_identical_to_oracle": ok, "device_load": pool.device_load()}))
pool.close()
