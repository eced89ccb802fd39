#!/usr/bin/env python
"""bench.py -- PairHMM forward throughput (GCUPS) on B200, BASELINE.json's metric on BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: row parameters, float forward kernels, the fallback-task builder,
the double re-run (pmm_launch of include/pairhmm_cuda.h).  At N = 1 the workload is configs[1] of BASELINE.json
(config 2, the GATK-HaplotypeCaller-like active region: 1000 reads x 151 bp against 64 haplotypes of 300-600 bp,
~4.4e9 cells).  With N > 1 (torch.distributed.run, one rank per GPU) every rank runs the same batch: pairs are independent,
nothing is reduced, so there is no data-path collective ("weak" scaling); NCCL carries only the barrier and the max over
ranks of the device time.

The JSON line
  value         whole-job GCUPS (cells = sum(read_len) * sum(hap_len), /root/reference/pairhmm/host/main.cpp:305-313) with
                inputs resident in HBM, CUDA events per step, L2 flushed between steps, launch overlap off
                (value_overlapped_no_l2_flush: back-to-back launches as a streaming caller issues them)
  e2e           the same metric with HOST buffers: pack + H2D + kernels + D2H + host log10 inside the timed region.
                `value` = through the work queue (pmm_pool_*, 4 contexts, neighbouring steps overlap); `serial_value` = one
                context, nothing overlapped; `plugin_value` = through the reference-named classes PairHMMClient +
                PairHMMWorker over the task plugin libPairHMMTask.so (pairhmm_worker_forward), one caller thread;
                `plugin_threads_value` = the same from three caller threads (GATK's threading model)
  parity        the GPU results of the batches timed here against the reference's CPU implementation, bit for bit
  roofline      float forward kernel vs the measured FP32 issue rate (12 FP32 instr per cell, SURVEY.md 8d)
  roofline_f64  double re-run vs the measured FP64 issue rate (12 DP instr per cell of the re-run pairs)
  per_config    the other BASELINE.json shapes (cfg1, 3, 4, a 5-slice): value, e2e, kernel fractions, fallback share,
                parity, fast mode -- 5 steps each (more for the small config 1: about 20 ms of timed work)
  queue         rank 0 only: the cfg5 stream through ONE pmm_pool over all N GPUs (north_star's host work queue), the same
                stream on one GPU in the same run, efficiency, per-GPU idle fraction from the pool's timeline
  cpu_baseline  the reference's AVX implementation (oracle/_ref) on this box's host cores -- reported, not the target
--impl reference times that CPU implementation as the step itself.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "pairhmm_forward_gcups"
UNIT = "GCUPS"
L2_NOTE = "GPU arm: L2 flushed between steps (256 MiB fill outside the timed bracket); CPU arm: not applicable"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json configs index (1-based), default 2")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; reported in config)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (and with them the parity check)")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the extra fast-mode measurement")
    ap.add_argument("--no-per-config", action="store_true", help="skip the per_config block")
    ap.add_argument("--no-queue", action="store_true", help="skip the work-queue block")
    ap.add_argument("--no-plugin", action="store_true", help="skip the plugin-path e2e")
    ap.add_argument("--no-sw", action="store_true", help="skip the Smith-Waterman block (SURVEY.md section 8f row 4)")
    ap.add_argument("--queue-jobs-per-gpu", type=int, default=192)
    ap.add_argument("--timeline", default="", help="write the pool's per-job timeline of the queue run to this .jsonl")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ---- clocks during the timed region ----------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and throttle reasons every 10 ms DURING the timed region (NVML; nvidia-smi -lms 20 if NVML is
    unavailable)."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index: int, period_s: float = 0.010):
        self.index, self.period = index, period_s
        self.rows, self.t0, self.t1 = [], None, None
        self._stop = threading.Event()
        self._thread = None
        self._smi = None
        self.how = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self._stop.is_set():
                    try:
                        self.rows.append((time.time(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                          pynvml.nvmlDeviceGetPowerUsage(h) * 1e-3, int(reasons(h))))
                    except Exception:
                        pass
                    self._stop.wait(self.period)
            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
            self.how = f"NVML every {int(self.period * 1e3)} ms"
        except Exception:
            self._start_smi()

    def _start_smi(self):
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self._smi = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self._lines = []
            threading.Thread(target=lambda: [self._lines.append(ln.strip()) for ln in self._smi.stdout], daemon=True).start()
            self.how = "nvidia-smi -lms 20"
        except Exception:
            self._smi = None

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1)
        if self._smi:
            import datetime
            self._smi.terminate()
            self.sm_max = None
            for ln in self._lines:
                f = [x.strip() for x in ln.split(",")]
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    mask = sum(bit for (bit, _), v in zip(self.REASONS, f[4:8]) if v.lower().startswith("active"))
                    self.rows.append((ts, float(f[1]), float(f[3]), mask)); self.sm_max = max(self.sm_max or 0, float(f[2]))
                except (ValueError, IndexError):
                    continue
        inside = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= self.t1]
        use = inside or self.rows
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "samples_inside_timed_region": 0, "how": self.how}
        mask = 0
        for r in use:
            mask |= r[3]
        return {"sm_mhz": float(np.median([r[1] for r in use])), "sm_max_mhz": self.sm_max, "power_w": float(np.median([r[2] for r in use])),
                "reasons": [name for bit, name in self.REASONS if mask & bit], "samples": len(use),
                "samples_inside_timed_region": len(inside), "how": self.how}


# ---- helpers ------------------------------------------------------------------------------------------------------------
def workload(cfg: int, seed: int, scale: float):
    from acc_genomics_b200 import synth
    return synth.config(cfg, seed=seed, scale=scale)


def cells_of(batches) -> int:
    return int(sum(b.num_cells for b in batches))


def config_dict(cfg: int, scale: float, batches) -> dict:
    """The `config` object of the JSON line -- the same keys and values from both arms (--impl ours / reference)."""
    from acc_genomics_b200 import synth
    return {"workload": synth.CONFIG_NAMES[cfg], "scale": scale, "seed": cfg, "cells_per_step_per_gpu": cells_of(batches),
            "pairs_per_step_per_gpu": int(sum(b.num_pairs for b in batches)), "mode": "exact", "l2": L2_NOTE,
            "parallelism": "the same region batch on every GPU, independent pairs, no collective"}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6547.5, "fallback: this pool's measured copy bandwidth quoted in the task (6547.5 GB/s)"


def ncu_traffic(cfg: int, scale: float, kernel: str):
    """dram read + written bytes of one launch of `kernel` on this workload, from the newest ncu --set full capture summarised
    under profiles/ (sidecars written by tools/ncu_digest.py); None when no capture matches the run."""
    best = None
    for path in glob.glob(os.path.join(ROOT, "profiles", "*_ncu.json")):
        try:
            with open(path) as f:
                d = json.load(f)
        except Exception:
            continue
        if d.get("config") == cfg and abs(float(d.get("scale", 1.0)) - scale) < 1e-9 and d.get("role") == kernel:
            if best is None or d.get("captured", "") > best.get("captured", ""):
                best = dict(d, path=os.path.relpath(path, ROOT))
    return best


def cpu_reference_pass(lib, batches, threads: int):
    """One pass of the reference's batch loop (FalconPairHMM::computePairhmmAVX) over the workload.
    -> (seconds, [(raw, log10, mask) per region])."""
    t0 = time.perf_counter()
    res = [lib.batch(b, threads=threads) for b in batches]
    return time.perf_counter() - t0, res


def parity_of(raw, out, mask, ref) -> dict:
    """Bit equality of the GPU's raw floats, fallback decision and final log10 with the CPU reference's (regions in order)."""
    raw_r = np.concatenate([r[0].ravel() for r in ref]); out_r = np.concatenate([r[1].ravel() for r in ref])
    fb_r = np.concatenate([r[2].ravel() for r in ref])
    return {"pairs": int(raw_r.size), "raw_bit_equal": bool(np.array_equal(raw.view(np.uint32), raw_r.view(np.uint32))),
            "fallback_decision_equal": bool(np.array_equal(mask.astype(bool), fb_r.astype(bool))),
            "log10_bit_equal": bool(np.array_equal(out.view(np.uint64), out_r.view(np.uint64)))}


DUMP_LIMIT_BYTES = 64_000_000          # 64 MB, files with their headers
NPY_HEADER_RESERVE = 1024              # per file; np.save writes 128 bytes of header for a 1-D array


def dump_outputs(path: str, raw, log10, mask, limit: int = DUMP_LIMIT_BYTES):
    """Write what a caller of the timed path receives, one entry per pair in job order (regions in order, read-major):
    raw.npy (float32 likelihoods of the float pass), log10.npy (float64 final log10 likelihoods) and fallback.npy (float32,
    1 where the pair was re-run in double).  The inputs depend only on the arguments, so two builds run with the same
    arguments can be compared file by file.  When the files would exceed `limit` bytes in all, a fixed seeded sample of the
    pairs is written instead, in pair order, and pair_index.npy (float64) names the pairs it holds."""
    arrays = {"raw": np.asarray(raw, dtype=np.float32).ravel(), "log10": np.asarray(log10, dtype=np.float64).ravel(),
              "fallback": np.asarray(mask, dtype=np.float32).ravel()}
    n = arrays["raw"].size
    per_pair = sum(a.itemsize for a in arrays.values())
    if n * per_pair + 3 * NPY_HEADER_RESERVE > limit:
        keep = (limit - 4 * NPY_HEADER_RESERVE) // (per_pair + 8)
        idx = np.sort(np.random.Generator(np.random.PCG64(0)).choice(n, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["pair_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def fallback_cells(batches, mask) -> int:
    """Cells (read_len x hap_len) of the pairs that take the double re-run."""
    pos, tot = 0, 0
    for b in batches:
        m = mask[pos:pos + b.num_pairs].reshape(b.num_read, b.num_hap); pos += b.num_pairs
        tot += int((b.read_lens[:, None].astype(np.int64) * b.hap_lens[None, :].astype(np.int64))[m].sum())
    return tot


_T0 = time.perf_counter()


def log(msg: str):
    print(f"[bench +{time.perf_counter() - _T0:7.2f}s] {msg}", file=sys.stderr, flush=True)


def max_over_ranks(vals, world: int, device) -> list:
    """Every timing of the JSON line is the slowest rank's: one all-reduce (MAX) of a float64 vector.  The collective is
    control plane only (NCCL on the GPU box, gloo in the CPU test); the data path has none."""
    if world <= 1:
        return [float(v) for v in vals]
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def checker():
    import oracle
    lib = oracle.reference()
    return (lib, "reference") if lib is not None else (oracle.port(), "port")


def run_reference(args, rank: int, out=sys.stdout):
    """--impl reference: the reference's own CPU implementation on the host cores (rank 0 only)."""
    if rank != 0:
        return
    lib, kind = checker()
    threads = os.cpu_count() or 1
    batches = workload(args.config, args.config, args.scale)
    cells = cells_of(batches)
    for _ in range(args.warmup):
        cpu_reference_pass(lib, batches, threads)
    total = 0.0
    for _ in range(args.steps):
        dt, res = cpu_reference_pass(lib, batches, threads)
        total += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *(np.concatenate([r[k].ravel() for r in res]) for k in range(3)))
    val = cells * args.steps / total * 1e-9
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic", "config": config_dict(args.config, args.scale, batches),
        "note": "reference AVX PairHMM (float pass, double re-run, log10) on host cores; no GPU involved",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "the full workload per step, all host threads, static split over reads"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), file=out, flush=True)


def main():
    args = parse()
    # Libraries (NCCL's version banner, for one) write to fd 1; the contract is ONE JSON line on stdout.  Keep the real
    # stdout aside and point fd 1 at stderr until the line is printed.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    try:
        _main(args, real_stdout)
    finally:
        real_stdout.flush()


# ---- measurement pieces (GPU) -----------------------------------------------------------------------------------------------
class Gpu:
    """The engine, a stream torch can see, an L2 flush buffer and the timing loops shared by the headline and per_config."""

    def __init__(self, local: int):
        import torch
        from acc_genomics_b200.engine import PairHMMEngine
        self.torch, self.local = torch, local
        self.eng = PairHMMEngine(local)
        self.side = torch.cuda.Stream()                    # torch.cuda.Event records on the current stream: make it this one
        torch.cuda.set_stream(self.side)
        self.eng.set_option("stream", self.side.cuda_stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")        # > 126 MB L2

    def timed_launches(self, steps: int):
        """Device time (s) of `steps` launches of the staged job, L2 flushed before each, CUDA events on the engine's stream.
        Launch overlap is switched off for it: every launch ends with its own double re-run, so the per-step brackets add
        up and the flush stays outside them.  The host runs ahead: no launch latency inside a bracket."""
        torch = self.torch
        self.eng.set_option("overlap", "off")
        self.eng.join()                                    # a double re-run of an earlier (overlapping) launch belongs to no bracket
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            self.flush.fill_(1)                            # evicts L2; on the same stream, outside the timed bracket
            a.record(); self.eng.launch(); b.record()
        ev[-1][1].synchronize()
        self.eng.set_option("overlap", "on")
        return sum(a.elapsed_time(b) for a, b in ev) * 1e-3

    def timed_overlapped(self, steps: int):
        """The same launches the way a streaming caller issues them: back to back with overlap on (the float pass of step
        k + 1 beside the double re-run of step k), ONE region from the first launch to the end of the last re-run, no L2
        flush (a fill between the steps would serialise them)."""
        torch = self.torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.eng.join()
        a.record()
        for _ in range(steps):
            self.eng.launch()
        self.eng.join()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) * 1e-3

    def kernel_ms(self, reps: int):
        """(float pass ms, double re-run ms) from the engine's own events (read_params + forward launches | builders + double)."""
        f32, fb = [], []
        for _ in range(reps):
            self.flush.fill_(1)
            self.eng.launch(); self.eng.sync()
            st = self.eng.stats()
            f32.append(st["ms_f32"]); fb.append(st["ms_fallback"])
        return float(np.mean(f32)), float(np.mean(fb))

    def results(self):
        raw = self.eng.fetch_raw(); out, nfb = self.eng.fetch_log10(); mask = self.eng.fetch_fallback_mask()
        return raw, out, mask, nfb

    def pool_e2e(self, job, pairs: int, steps: int, depth: int = 4):
        """Seconds for `steps` jobs through a one-GPU pool with `depth` contexts (host buffers in, float64 log10 out)."""
        from collections import deque
        from acc_genomics_b200.engine import PairHMMPool
        pool = PairHMMPool(devices=[self.local], contexts_per_device=depth)
        outs = [np.empty(pairs, dtype=np.float64) for _ in range(depth + 1)]

        def run(n):
            live = deque()
            for k in range(n):
                if len(live) > depth:
                    pool.wait(live.popleft())
                live.append(pool.submit(None, out=outs[k % (depth + 1)], job=job))
            while live:
                pool.wait(live.popleft())
        run(2 * depth)
        self.torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(steps)
        dt = time.perf_counter() - t0
        pool.close()
        return dt, outs[0]


def measure_fast(gpu: Gpu, steps: int, out_exact, nfb_exact):
    """Fast mode on the staged job (restaged): device time, float-pass ms, agreement with the exact results."""
    eng = gpu.eng
    eng.set_option("mode", "fast")
    eng.restage()
    for _ in range(3):
        eng.launch()
    dev_s = gpu.timed_launches(steps)
    f32_ms, _ = gpu.kernel_ms(min(5, steps))
    out_f, nfb_f = eng.fetch_log10()
    fin = np.isfinite(out_exact)
    res = {"steps": steps, "dev_s": dev_s, "f32_ms": f32_ms, "recheck_pairs": int(eng.stats()["recheck_pairs"]),
           "same_decision": bool(nfb_f == nfb_exact and np.array_equal(np.isfinite(out_f), fin)),
           "max_rel": float(np.max(np.abs(out_f[fin] - out_exact[fin]) / np.abs(out_exact[fin]))) if fin.any() else 0.0}
    eng.set_option("mode", "exact")
    eng.restage()
    return res


def measure_config(gpu: Gpu, cfg: int, scale: float, steps: int, fast: bool):
    """One per_config entry (this rank's share): device-resident and queue e2e seconds, kernel ms, results for parity."""
    batches = workload(cfg, cfg, scale)
    eng = gpu.eng
    job = eng.stage(batches)
    for _ in range(3):
        eng.launch()
    # a small configuration (config 1 is 0.13 ms per step) gets more steps: about 20 ms of timed work, at least `steps`
    probe = gpu.timed_launches(2) / 2
    steps = int(max(steps, min(200, 0.02 / max(probe, 1e-6))))
    dev_s = gpu.timed_launches(steps)
    f32_ms, fb_ms = gpu.kernel_ms(min(5, steps))
    raw, out, mask, nfb = gpu.results()
    st = eng.stats()
    e2e_s, pool_out = gpu.pool_e2e(job, int(st["pairs"]), steps)
    rec = {"cfg": cfg, "scale": scale, "batches": batches, "cells": cells_of(batches), "pairs": int(st["pairs"]), "steps": steps,
           "dev_s": dev_s, "e2e_s": e2e_s, "f32_ms": f32_ms, "fb_ms": fb_ms, "raw": raw, "out": out, "mask": mask.astype(bool), "nfb": nfb,
           "flush_pairs": int(st["flush_pairs"]), "pool_same": bool(np.array_equal(pool_out.view(np.uint64), out.view(np.uint64))),
           "launches": int(st["kernel_launches"])}
    if fast:
        rec["fast"] = measure_fast(gpu, steps, out, nfb)
    return rec


def measure_plugin(batch, steps: int, local: int, threads: int):
    """Seconds per batch through PairHMMClient + PairHMMWorker over libPairHMMTask.so (pairhmm_worker_forward): serialize,
    task prepare()/compute() on two slots, tiles pipelined, final doubles out.  threads > 1: that many caller threads, each
    with its own client and its own copy of the batch."""
    from acc_genomics_b200 import hostlayer
    os.environ.setdefault("PAIRHMM_DEVICES", str(local))
    os.environ.setdefault("PAIRHMM_SLOTS", "4")
    jobs = [hostlayer.WorkerJob(batch) for _ in range(threads)]
    for j in jobs:
        hostlayer.worker_forward(j)
    if threads == 1:
        for _ in range(3):
            hostlayer.worker_forward(jobs[0])
        t0 = time.perf_counter()
        for _ in range(steps):
            hostlayer.worker_forward(jobs[0])
        return (time.perf_counter() - t0) / steps, jobs[0].out.copy()
    per = max(8, steps // threads)                 # batches per thread: the start and the end of the run are ragged
    go = threading.Barrier(threads + 1)

    def work(j):
        hostlayer.worker_forward(j)
        go.wait()
        for _ in range(per):
            hostlayer.worker_forward(j)
    th = [threading.Thread(target=work, args=(j,)) for j in jobs]
    [t.start() for t in th]
    go.wait()
    t0 = time.perf_counter()
    [t.join() for t in th]
    return (time.perf_counter() - t0) / (per * threads), jobs[0].out.copy()


def measure_queue(n_gpus: int, jobs_per_gpu: int, timeline_path: str, contexts: int = 4):
    """The cfg5 stream (jobs of 25 regions, host buffers in, float64 log10 out) through ONE pool over n_gpus devices, and the
    same stream through a one-GPU pool in the same run.  -> dict for the JSON line (+ the jobs for the parity leg)."""
    from collections import deque
    from acc_genomics_b200.engine import PairHMMPool, concat_regions
    regs = workload(5, 5, 0.06)                                   # 150 regions of 100 reads x 40 haplotypes
    jobs = [concat_regions(regs[k:k + 25]) for k in range(0, len(regs), 25)]
    job_cells = [cells_of(regs[k:k + 25]) for k in range(0, len(regs), 25)]

    def stream(devices, n_jobs, trace):
        pool = PairHMMPool(devices=devices, contexts_per_device=contexts)
        window = 2 * contexts * len(devices) + 6
        outs = [np.empty(jobs[0]["pairs"], dtype=np.float64) for _ in range(window + 1)]

        def run(n, keep=None):
            live = deque()
            for k in range(n):
                if len(live) >= window:
                    t, slot, which = live.popleft(); pool.wait(t)
                    if keep is not None:
                        keep.append((which, outs[slot].copy()))
                slot = k % (window + 1)
                live.append((pool.submit(None, out=outs[slot], job=jobs[k % len(jobs)]), slot, k % len(jobs)))
            while live:
                t, slot, which = live.popleft(); pool.wait(t)
                if keep is not None:
                    keep.append((which, outs[slot].copy()))
        run(window + len(jobs))                                   # warm-up: every context has grown its buffers
        pool.trace(trace)
        t0 = time.perf_counter()
        run(n_jobs)
        dt = time.perf_counter() - t0
        pool.trace(False)
        tr = pool.get_trace() if trace else []
        kept = []
        run(len(jobs) * max(2, len(devices)), keep=kept)           # untimed: outputs of every distinct job, for the parity leg
        load = pool.device_load()
        pool.close()
        cells = sum(job_cells[k % len(jobs)] for k in range(n_jobs))
        return cells / dt * 1e-9, dt, tr, load, kept

    one_gcups, one_s, _, _, _ = stream([0], jobs_per_gpu, False)
    all_gcups, all_s, tr, load, kept = stream(list(range(n_gpus)), jobs_per_gpu * n_gpus, True)
    # per-device: share of the traced window with no kernel of ours on the device (union of the jobs' kernel spans)
    idle, host = {}, {}
    lo = min(r["d_start"] for r in tr); hi = max(r["d_end"] for r in tr)
    for d in range(n_gpus):
        spans = sorted((r["d_start"], r["d_end"]) for r in tr if r["device"] == d)
        busy, cur_a, cur_b = 0.0, None, None
        for a, b in spans:
            if cur_b is None or a > cur_b:
                busy += (cur_b - cur_a) if cur_b is not None else 0.0
                cur_a, cur_b = a, b
            else:
                cur_b = max(cur_b, b)
        busy += (cur_b - cur_a) if cur_b is not None else 0.0
        idle[str(d)] = round(1.0 - busy / (hi - lo), 4)
    for key, a, b in (("stage_ms", "t_take", "t_staged"), ("launch_call_ms", "t_staged", "t_launched"), ("fetch_ms", "t_launched", "t_fetched"),
                      ("kernels_ms", "d_start", "d_end")):
        host[key] = round(float(np.mean([r[b] - r[a] for r in tr])) * 1e3, 4)
    if timeline_path:
        with open(timeline_path, "w") as f:
            for r in tr:
                f.write(json.dumps(r) + "\n")
    return {"workload": "cfg5 stream: jobs of 25 regions (100 reads x 40 haps each) from 150 distinct regions, host buffers in, float64 log10 out",
            "path": f"pmm_pool_submit_flat / pmm_pool_wait, ONE pool in ONE process over all GPUs, {contexts} contexts per GPU, no collective",
            "n_gpus": n_gpus, "jobs": jobs_per_gpu * n_gpus, "gcups": all_gcups, "seconds": all_s, "gcups_1gpu": one_gcups, "seconds_1gpu": one_s,
            "efficiency": all_gcups / (one_gcups * n_gpus), "per_device": load, "gpu_idle_frac": idle, "mean_per_job": host,
            "gpu_jobs_traced": len(tr)}, regs, kept


def measure_sw(local: int, sm_mhz):
    """SURVEY.md section 8f row 4, reported aside: Smith-Waterman with backtrack on 2 080 haplotype-to-reference pairs
    (8 windows x 260 alternates, 250-500 bp): kernel-only and whole-call GCUPS, the reference's AVX2 kernel on one host
    thread beside it, CIGAR/offset equality on the pairs the CPU ran."""
    import torch
    from acc_genomics_b200 import sw
    al = sw.SmithWaterman(local)
    pairs = sw.haplotype_pairs(1, 2080, ref_len=(250, 500), per_ref=260)
    cells = sum(len(r) * len(a) for r, a in pairs)
    al.align(pairs[:64], 0)
    best = [float("inf"), float("inf")]                        # kernel ms, whole-call ms: best of five each
    for _ in range(5):
        out = al.align(pairs, 0)
        st = al.stats()
        best = [min(best[0], st["ms_kernel"]), min(best[1], st["ms_total"])]
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    # ~11.5 ALU-pipe instructions per cell (adds, min/max, funnel shifts), half rate: 23 issue cycles per cell and lane
    bound = sms * 128 / 23.0 * (sm_mhz or 1965.0) * 1e6 * 1e-9
    rec = {"workload": "2 080 haplotype-to-reference pairs (8 windows x 260 alternates, 250-500 bp), soft-clip overhangs, GATK weights",
           "pairs": len(pairs), "cells": cells, "kernel_ms": best[0], "call_ms": best[1], "kernel_gcups": cells / best[0] * 1e-6,
           "call_gcups": cells / best[1] * 1e-6, "alu_pipe_bound_gcups": bound, "frac_of_alu_bound": cells / best[0] * 1e-6 / bound,
           "backtrack_mb": st["bytes_backtrack"] / 1e6,
           "path": "sw_align_batch (include/smithwaterman_cuda.h): host buffers in, CIGARs out; kernel_ms from CUDA events"}
    # the same kernel with the GPU full: 64 windows x 260 alternates (one window's worth of pairs leaves most warps a single
    # pair, so the small batch above is bounded by its longest pairs)
    big = sw.haplotype_pairs(1, 16640, ref_len=(250, 500), per_ref=260)
    big_cells = sum(len(r) * len(a) for r, a in big)
    kb = float("inf")
    for _ in range(3):
        al.align(big, 0)
        kb = min(kb, al.stats()["ms_kernel"])
    rec["large_batch"] = {"pairs": len(big), "cells": big_cells, "kernel_ms": kb, "kernel_gcups": big_cells / kb * 1e-6,
                          "frac_of_alu_bound": big_cells / kb * 1e-6 / bound}
    try:
        import oracle
        ref = oracle.sw_reference()
        if ref is not None:
            sub = [(k, r, a) for k, (r, a) in enumerate(pairs[:208]) if len(a) <= 1536 and len(r) <= 1536]
            t0 = time.perf_counter()
            got = [ref.align(r, a, 0) for _, r, a in sub]
            dt = time.perf_counter() - t0
            rec["cpu_avx2_1thread_gcups"] = sum(len(r) * len(a) for _, r, a in sub) / dt * 1e-9
            rec["parity"] = {"pairs_checked": len(sub),
                             "offset_and_cigar_equal": bool(all(tuple(g[:2]) == (out[k][0], out[k][1]) for g, (k, _, _) in zip(got, sub)))}
    except Exception as e:
        rec["cpu_avx2_1thread_gcups"] = None; rec["parity"] = {"error": f"{type(e).__name__}: {e}"}
    al.close()
    return rec


def _main(args, real_stdout):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, real_stdout)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the PairHMM engine has no CPU path")
    torch.cuda.set_device(local)
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")          # barrier that keeps the other ranks' GPUs idle (queue block)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload: the same batch on every rank (weak scaling of independent batches, no exchange) ------------------------
    batches = workload(args.config, args.config, args.scale)
    cells = cells_of(batches)
    gpu = Gpu(local)
    eng = gpu.eng
    log("workload generated")
    job = eng.stage(batches)
    warm = max(args.warmup, 3)

    # ---- device-resident timing (value) ----------------------------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(warm):
        eng.launch()
    barrier()
    sampler.t0 = time.time()
    dev_s = gpu.timed_launches(args.steps)
    barrier()
    sampler.t1 = time.time()
    raw, out, mask, nfb = gpu.results()                    # the last timed step's results
    mask = mask.astype(bool)
    dev_noflush_s = gpu.timed_overlapped(args.steps)
    clocks = sampler.stop()
    log("timed region done")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, raw, out, mask)
    f32_ms, fb_ms = gpu.kernel_ms(min(args.steps, 10))
    st = eng.stats()
    pairs = int(st["pairs"])
    assert np.isfinite(raw).all() and not np.isnan(out).any()

    # ---- end to end with host buffers ----------------------------------------------------------------------------------------
    # (a) one job at a time on one context: stage (pack, H2D) -> launch -> fetch (D2H, host log10), nothing overlapped
    res = np.empty(pairs, dtype=np.float64)
    for _ in range(3):
        eng.restage(); eng.launch(); eng.fetch_log10(res)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.restage(); eng.launch(); eng.fetch_log10(res)
    e2e_serial_s = time.perf_counter() - t0
    st2 = eng.stats()
    serial_same = bool(np.array_equal(res.view(np.uint64), out.view(np.uint64)))
    # (b) the same steps through the work queue a host application uses (three contexts overlap neighbouring steps)
    barrier()
    e2e_s, pool_out = gpu.pool_e2e(job, pairs, args.steps)
    pool_same = bool(np.array_equal(pool_out.view(np.uint64), out.view(np.uint64)))
    log("e2e done")
    # (c) through the reference-named client classes and the task plugin
    plugin = None
    if not args.no_plugin and len(batches) == 1:
        barrier()
        p1_s, p_out = measure_plugin(batches[0], args.steps, local, 1)
        barrier()
        p3_s, p3_out = measure_plugin(batches[0], args.steps, local, 3)
        plugin = {"s_per_step": p1_s, "s_per_step_threads3": p3_s,
                  "same": bool(np.array_equal(p_out.view(np.uint64), out.view(np.uint64)) and np.array_equal(p3_out.view(np.uint64), out.view(np.uint64)))}
        log("plugin path done")

    # ---- fast mode on the headline workload, reported aside -------------------------------------------------------------------
    fast = None if args.no_fast_mode else measure_fast(gpu, min(args.steps, 50), out, nfb)

    # ---- the other configurations -------------------------------------------------------------------------------------------
    per = []
    if not args.no_per_config:
        for cfg, scale in ((1, 1.0), (3, 1.0), (4, 1.0), (5, 0.02)):
            if cfg == args.config:
                continue
            barrier()
            per.append(measure_config(gpu, cfg, scale, 5, not args.no_fast_mode))
        log("per_config done")

    # ---- issue peaks, measured on this GPU ---------------------------------------------------------------------------------------
    peak32, _ = eng.measure_fp32_peak()
    peak64 = eng.measure_fp64_peak()

    # ---- max over ranks ------------------------------------------------------------------------------------------------------
    vals = [dev_s, e2e_s, e2e_serial_s, plugin["s_per_step"] if plugin else 0.0, plugin["s_per_step_threads3"] if plugin else 0.0, dev_noflush_s]
    for r in per:
        vals += [r["dev_s"], r["e2e_s"]]
    vals = max_over_ranks(vals, world, "cuda")
    dev_s, e2e_s, e2e_serial_s, p1_s, p3_s, dev_noflush_s = vals[:6]
    for k, r in enumerate(per):
        r["dev_s"], r["e2e_s"] = vals[6 + 2 * k], vals[7 + 2 * k]

    # ---- the work queue over all GPUs: rank 0 drives one pool, the other ranks sit at a CPU barrier with idle GPUs ----------------
    queue = queue_regs = queue_kept = None
    eng_alive = True
    if not args.no_queue:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)
        if rank == 0:
            queue, queue_regs, queue_kept = measure_queue(world, args.queue_jobs_per_gpu, args.timeline)
            log("queue done")
        if world > 1:
            dist.barrier(group=cpu_group)

    if rank == 0:
        job_cells = float(cells) * world
        value = job_cells * args.steps / dev_s * 1e-9
        f32_cps = cells / (f32_ms * 1e-3)
        achieved = f32_cps * 12 * 1e-12
        peak = peak32 * 1e-12
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        nominal_peak = sms * 128 * clocks["sm_mhz"] * 1e6 * 1e-12 if clocks.get("sm_mhz") else None
        cap = ncu_traffic(args.config, args.scale, "f32")
        traffic = (cap["dram_bytes_read"] + cap["dram_bytes_write"]) if cap else None
        hbm, hbm_src = hbm_peak()
        fcells = fallback_cells(batches, mask)
        ach64 = fcells * 12 / (fb_ms * 1e-3) * 1e-12 if fb_ms > 0 else 0.0
        cap64 = ncu_traffic(args.config, args.scale, "f64")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (exact op order, no FMA contraction) + f64 re-run of underflowed pairs", "data": "synthetic",
            "config": config_dict(args.config, args.scale, batches),
            "fallback_pairs": int(nfb), "flush_pairs": int(st["flush_pairs"]),
            "value_overlapped_no_l2_flush": job_cells * args.steps / dev_noflush_s * 1e-9,
            "value_overlapped_note": "not the headline: the same launches back to back on one context with launch overlap on (float "
                                     "pass of step k+1 beside the double re-run of step k), one timed region, no L2 fill between steps",
            "e2e": {"value": job_cells * args.steps / e2e_s * 1e-9, "unit": UNIT, "h2d_bytes_per_step": int(st2["h2d_bytes"]),
                    "d2h_bytes_per_step": int(st2["d2h_bytes"]), "ms_per_step": e2e_s / args.steps * 1e3,
                    "path": "pmm_pool_submit_flat / pmm_pool_wait, 4 contexts (2 feeder threads) on the GPU: per step pack + H2D + kernels + D2H + host "
                            "log10, host numpy buffers in, float64 log10 out, steps overlapped by the queue",
                    "serial_value": job_cells * args.steps / e2e_serial_s * 1e-9, "serial_ms_per_step": e2e_serial_s / args.steps * 1e3,
                    "serial_path": "pmm_stage_flat + pmm_launch + pmm_fetch_log10 on one context, one step at a time"},
            "gpu_launches": int(st["kernel_launches"]) * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "fp32_issue", "kernel": "pmm_forward_kernel<float,K,W> (float pass)", "achieved": achieved, "peak": peak,
                         "unit": "T FP32 lane-instr/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": (f"{cap['path']}: dram__bytes_read.sum {cap['dram_bytes_read']} + dram__bytes_write.sum "
                                            f"{cap['dram_bytes_write']} per launch ({cap.get('kernel', '')})") if cap else
                                           "no ncu --set full capture of this workload under profiles/ (tools/ncu_digest.py writes them)",
                         "kernel_ms": f32_ms, "kernel_gcups": f32_cps * 1e-9,
                         "kernel_ms_note": "CUDA events around read_params_kernel + the float forward launch(es) on the engine's stream",
                         "algorithmic": "12 FP32 instr per cell (8 FMUL + 4 FADD) x cells per launch",
                         "peak_source": "measured live: independent FMUL/FADD streams (pmm_measure_fp32_peak); MEASURED_PEAKS.json has no FP32 figure",
                         "frac_flop_convention": achieved / (2 * peak), "nominal_peak": nominal_peak,
                         "frac_vs_nominal": (achieved / nominal_peak) if nominal_peak else None,
                         "nominal_peak_note": "SMs x 128 FP32 lanes x the SM clock sampled during the timed region",
                         "hbm_view": {"achieved": traffic / (f32_ms * 1e-3) * 1e-9 if traffic else None, "peak": hbm, "unit": "GB/s",
                                      "frac": traffic / (f32_ms * 1e-3) * 1e-9 / hbm if traffic else None, "peak_source": hbm_src}},
            "roofline_f64": {"bound": "fp64_issue", "kernel": "fallback_scan_kernel + fallback_tasks_kernel + pmm_forward_kernel<double,K,32> (double re-run)",
                             "achieved": ach64, "peak": peak64 * 1e-12, "unit": "T FP64 lane-instr/s", "frac": ach64 / (peak64 * 1e-12),
                             "pass_ms": fb_ms, "fallback_pairs": int(nfb), "fallback_cells": fcells,
                             "algorithmic": "12 FP64 instr per cell (8 DMUL + 4 DADD) x cells of the pairs whose float result is below 1e-28f",
                             "peak_source": "measured live: independent DMUL/DADD streams (pmm_measure_fp64_peak)",
                             "traffic": (cap64["dram_bytes_read"] + cap64["dram_bytes_write"]) if cap64 else None,
                             "traffic_source": cap64["path"] if cap64 else None},
        }
        if plugin:
            line["e2e"].update({
                "plugin_value": job_cells / p1_s * 1e-9, "plugin_ms_per_step": p1_s * 1e3,
                "plugin_path": "pairhmm_worker_forward -> PairHMMClient::setup (serialize) + PairHMMWorker::run (tiles, all in flight on their own slots of "
                               "libPairHMMTask.so: prepare = stage, compute = launch + fetch) + getOutput; one caller thread, one batch at a time",
                "plugin_threads_value": job_cells / p3_s * 1e-9, "plugin_threads": 3, "plugin_bit_equal": plugin["same"]})
        if fast:
            fcps = cells / (fast["f32_ms"] * 1e-3)
            line["fast_mode"] = {
                "note": "opt-in pmm_set_option(mode=fast): contracted float cell update, exact re-check of results near the 1e-28f "
                        "threshold; decision identical, log10 within 1e-5 relative. This rank only; not the headline value",
                "value": cells * fast["steps"] / fast["dev_s"] * 1e-9, "unit": UNIT, "ms_per_step": fast["dev_s"] / fast["steps"] * 1e3,
                "kernel_gcups": fcps * 1e-9, "roofline_frac_8_instr_per_cell": fcps * 8 / peak32,
                "recheck_pairs": fast["recheck_pairs"], "same_decision_as_exact": fast["same_decision"],
                "max_rel_log10_vs_exact": fast["max_rel"]}
        log("gpu side done")

        # ---- CPU legs: baseline timing, and with its outputs the parity of everything timed above -----------------------------------
        parity = {"checked": False}
        if not args.no_cpu_baseline:
            try:
                lib, kind = checker()
                threads = os.cpu_count() or 1
                cpu_reference_pass(lib, batches, threads)
                runs = [cpu_reference_pass(lib, batches, threads) for _ in range(3)]
                best = min(r[0] for r in runs)
                parity = parity_of(raw, out, mask, runs[0][1])
                parity.update({"checked": True, "against": f"oracle kind={kind}", "serial_path_bit_equal": serial_same,
                               "queue_path_bit_equal": pool_same, "plugin_path_bit_equal": plugin["same"] if plugin else None})
                small = [batches[0].slice_reads(0, max(1, batches[0].num_read // 16))]
                one = cpu_reference_pass(lib, small, 1)[0]
                line["cpu_baseline"] = {"value": cells / best * 1e-9, "unit": UNIT, "cores": threads, "kind": kind,
                                        "sample": "the full workload (all pairs incl. double re-run and log10), best of 3 passes",
                                        "one_thread_gcups": cells_of(small) / one * 1e-9,
                                        "build": "g++ -O3 -mavx -ffp-contract=off (the arithmetic of Intel GKL's AVX build: no FMA contraction)"}
                try:
                    with open("/proc/cpuinfo") as f:
                        info = f.read()
                except OSError:
                    info = ""
                import oracle
                fma = oracle.reference(fma=True) if kind == "reference" and " fma" in info and " avx2" in info else None
                if fma is not None:                      # the build the reference's own Makefile makes (-march=native), timing only
                    cpu_reference_pass(fma, batches, threads)
                    line["cpu_baseline"]["fma_contracted_build_gcups"] = cells / min(cpu_reference_pass(fma, batches, threads)[0] for _ in range(3)) * 1e-9
                model = [ln.split(":", 1)[1].strip() for ln in info.splitlines() if ln.startswith("model name")]
                line["cpu_baseline"]["cpu_model"] = model[0] if model else None
                for r in per:
                    t, ref = cpu_reference_pass(lib, r["batches"], threads)
                    r["parity"] = parity_of(r["raw"], r["out"], r["mask"], ref)
                    r["parity"]["queue_path_bit_equal"] = r["pool_same"]
                    r["cpu_gcups"] = r["cells"] / t * 1e-9
                if queue is not None:
                    want = []
                    for k in range(0, len(queue_regs), 25):
                        want.append(np.concatenate([lib.batch(b, threads=threads)[1].ravel() for b in queue_regs[k:k + 25]]))
                    ok = all(np.array_equal(o.view(np.uint64), want[which].view(np.uint64)) for which, o in queue_kept)
                    queue["parity"] = {"jobs_checked": len(queue_kept), "pairs_checked": int(sum(o.size for _, o in queue_kept)), "log10_bit_equal": bool(ok)}
            except Exception as e:  # the baseline is a report, never a reason to lose the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": f"{type(e).__name__}: {e}"}
        line["parity"] = parity
        if per:
            line["per_config"] = []
            for r in per:
                fc = fallback_cells(r["batches"], r["mask"])
                cps = r["cells"] / (r["f32_ms"] * 1e-3)
                ent = {"workload": config_dict(r["cfg"], r["scale"], r["batches"])["workload"], "scale": r["scale"], "steps": r["steps"],
                       "cells_per_step_per_gpu": r["cells"], "pairs_per_step_per_gpu": r["pairs"],
                       "value": r["cells"] * world * r["steps"] / r["dev_s"] * 1e-9, "ms_per_step": r["dev_s"] / r["steps"] * 1e3,
                       "e2e": r["cells"] * world * r["steps"] / r["e2e_s"] * 1e-9,
                       "f32_pass_ms": r["f32_ms"], "f32_frac": cps * 12 / peak32, "f64_pass_ms": r["fb_ms"],
                       "f64_frac": (fc * 12 / (r["fb_ms"] * 1e-3) / peak64) if r["fb_ms"] > 0 and fc else None,
                       "fallback_frac": r["nfb"] / r["pairs"], "flush_pairs": r["flush_pairs"], "launches_per_step": r["launches"],
                       "parity": r.get("parity", {"checked": False}), "cpu_gcups": r.get("cpu_gcups")}
                if "fast" in r:
                    f = r["fast"]
                    ent["fast_mode"] = {"value": r["cells"] * f["steps"] / f["dev_s"] * 1e-9, "f32_pass_ms": f["f32_ms"],
                                        "roofline_frac_8_instr_per_cell": r["cells"] / (f["f32_ms"] * 1e-3) * 8 / peak32,
                                        "recheck_pairs": f["recheck_pairs"], "same_decision_as_exact": f["same_decision"],
                                        "max_rel_log10_vs_exact": f["max_rel"]}
                line["per_config"].append(ent)
        if queue is not None:
            line["queue"] = queue
        if not args.no_sw:
            try:
                line["sw"] = measure_sw(local, clocks.get("sm_mhz"))
            except Exception as e:
                line["sw"] = {"error": f"{type(e).__name__}: {e}"}
        log("cpu legs done")
        print(json.dumps(line), file=real_stdout, flush=True)
    if eng_alive:
        eng.close()
    try:
        from acc_genomics_b200 import hostlayer
        hostlayer.shutdown()
    except Exception:
        pass
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
