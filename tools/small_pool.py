"""GPU box: a stream of small jobs (config 1, 4 096 pairs each) through a one-GPU pool: throughput and where the time
between jobs goes (pool timeline)."""
import json, os, sys, time
from collections import deque
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from acc_genomics_b200 import synth
from acc_genomics_b200.engine import PairHMMPool, concat_regions
cfg = int(os.environ.get("CFG", "1")); ctxs = int(os.environ.get("CTX", "4")); depth = int(os.environ.get("DEPTH", "4"))
b = synth.config(cfg, scale=float(os.environ.get("SCALE", "1.0")))
job = concat_regions(b); cells = sum(x.num_cells for x in b)
pool = PairHMMPool(devices=[0], contexts_per_device=ctxs)
outs = [np.empty(job["pairs"]) for _ in range(depth + 1)]
def run(n):
    live = deque()
    for k in range(n):
        if len(live) > depth:
            pool.wait(live.popleft())
        live.append(pool.submit(None, out=outs[k % (depth + 1)], job=job))
    while live:
        pool.wait(live.popleft())
run(20)
pool.trace(True)
n = 200
t0 = time.perf_counter(); run(n); dt = time.perf_counter() - t0
pool.trace(False)
tr = pool.get_trace()
print(json.dumps({"cfg": cfg, "contexts": ctxs, "depth": depth, "us_per_job": round(dt / n * 1e6, 1),
                  "gcups": round(cells * n / dt * 1e-9, 1), "gpu_jobs": len(tr),
                  "stage_us": round(float(np.mean([r["t_staged"] - r["t_take"] for r in tr])) * 1e6, 1),
                  "launch_us": round(float(np.mean([r["t_launched"] - r["t_staged"] for r in tr])) * 1e6, 1),
                  "kernels_us": round(float(np.mean([r["d_end"] - r["d_start"] for r in tr])) * 1e6, 1),
                  "launch_to_start_us": round(float(np.mean([r["d_start"] - r["t_launched"] for r in tr])) * 1e6, 1),
                  "end_to_delivered_us": round(float(np.mean([r["t_fetched"] - r["d_end"] for r in tr])) * 1e6, 1)}))
pool.close()
