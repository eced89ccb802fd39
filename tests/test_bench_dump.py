"""bench.py --dump-outputs: the results of the last timed step, identical from run to run with the same arguments, and a
fixed sample of the pairs when the outputs are large.  The GPU arm's dump is checked against the CPU oracle; the reference
arm runs that oracle itself, so its test checks the plumbing (pair order, dtypes, reproducibility)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_bits_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def run_bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900,
                       cwd=ROOT, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def load(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("raw", "log10", "fallback")}


def assert_matches_checker(got, port, cfg):
    b = bench.workload(cfg, cfg, 1.0)[0]
    raw, out, mask = port.batch(b, threads=os.cpu_count() or 1)
    assert got["raw"].dtype == np.float32 and got["log10"].dtype == np.float64 and got["fallback"].dtype == np.float32
    assert_bits_equal(got["raw"], raw.ravel(), "raw")
    assert_bits_equal(got["log10"], out.ravel(), "log10")
    assert np.array_equal(got["fallback"], mask.ravel().astype(np.float32))


def test_reference_arm_dumps_its_last_step(port, tmp_path):
    dumps = []
    for k in range(2):
        line = run_bench("--impl", "reference", "--config", "1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path / str(k)))
        assert line["steps"] == 2
        dumps.append(load(tmp_path / str(k)))
    for name in dumps[0]:
        assert_bits_equal(dumps[0][name], dumps[1][name], name)
    assert_matches_checker(dumps[0], port, 1)


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "--steps" in p.stderr


NAMES = ("raw", "log10", "fallback", "pair_index")


def dumped_bytes(d):
    return sum(os.path.getsize(os.path.join(d, n + ".npy")) for n in NAMES if os.path.exists(os.path.join(d, n + ".npy")))


def test_large_outputs_are_sampled_the_same_way_every_time(tmp_path):
    rng = np.random.Generator(np.random.PCG64(3))
    raw = rng.random(5000, dtype=np.float32); out = np.log10(raw.astype(np.float64)); mask = raw < 0.1
    limit = 16 << 10
    for k in range(2):
        bench.dump_outputs(str(tmp_path / str(k)), raw, out, mask, limit=limit)
    assert dumped_bytes(tmp_path / "0") <= limit
    got = {n: np.load(tmp_path / "0" / (n + ".npy")) for n in NAMES}
    for n in NAMES:
        assert np.array_equal(got[n], np.load(tmp_path / "1" / (n + ".npy")))
    idx = got["pair_index"].astype(np.int64)
    assert 0 < idx.size < raw.size and (np.diff(idx) > 0).all()
    assert np.array_equal(got["raw"], raw[idx]) and np.array_equal(got["log10"], out[idx])
    assert np.array_equal(got["fallback"], mask[idx].astype(np.float32))


@pytest.mark.parametrize("pairs", [3_999_000, 5_000_000])
def test_dump_stays_within_64_mb(tmp_path, pairs):
    """Just under the point where sampling starts, and past it: the files with their headers stay within 64e6 bytes."""
    raw = np.ones(pairs, dtype=np.float32)
    bench.dump_outputs(str(tmp_path), raw, raw.astype(np.float64), raw < 0)
    assert dumped_bytes(tmp_path) <= 64_000_000 and bench.DUMP_LIMIT_BYTES == 64_000_000
    assert os.path.exists(tmp_path / "pair_index.npy") == (pairs == 5_000_000)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(port, tmp_path):
    line = run_bench("--config", "1", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-fast-mode", "--no-per-config",
                     "--no-queue", "--no-plugin", "--no-sw", "--dump-outputs", str(tmp_path))
    assert line["steps"] == 3
    assert_matches_checker(load(tmp_path), port, 1)
