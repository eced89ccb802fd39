"""A short run of tools/fuzz_gpu.py: random region shapes and multi-region jobs through every entry point (staged, serialized,
read_t/hap_t arrays, pool), exact and fast mode, plus Smith-Waterman -- every result against the oracle."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_fuzz_for_a_few_seconds(built):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_gpu.py"), "12", "20261018"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode == 0 and "fuzz ok" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]


@pytest.mark.gpu
def test_planner_shapes_for_a_few_seconds(built):
    """tools/fuzz_plan_gpu.py: random large multi-region jobs under random graded-run / queue-depth / widening settings give
    the result of the plainest plan bit for bit, and that one equals the oracle's."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_plan_gpu.py"), "8", "20261019"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode == 0 and "plan fuzz ok" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]
