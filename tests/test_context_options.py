"""Planner options: PMM_SMALL_JOB_WIDENING and PMM_RUN_TIERS are the defaults pmm_plan_flat and every new context start
from; "small_job_widening" and "run_tiers" set through pmm_set_option apply to that context alone."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from acc_genomics_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the 10 x 5 toy region of test_plan.test_small_jobs_get_wider_lanes and config 2 at full size, as pmm_plan_flat cuts them
PLAN_SUMMARY = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from acc_genomics_b200 import engine, synth
toy = synth.region(np.random.Generator(np.random.PCG64(11)), [151] * 10, [400] * 5)
out = {}
for name, job in (("toy", toy), ("cfg2", synth.config(2))):
    t = engine.plan(job)
    out[name] = dict(tasks=len(t), variants=sorted({(x["K"], x["W"]) for x in t}), haps=sorted({x["num_hap"] for x in t}))
print(json.dumps(out))
"""


def plan_summary(**env):
    """The environment is read once per process: each setting gets a process of its own."""
    e = {k: v for k, v in os.environ.items() if k not in ("PMM_SMALL_JOB_WIDENING", "PMM_RUN_TIERS")}
    e.update(env)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", PLAN_SUMMARY, ROOT]
    r = subprocess.run(cmd, env=e, cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout)


def test_environment_defaults_reach_plan_flat(built):
    d = plan_summary()
    assert d["toy"]["tasks"] == 50 and d["toy"]["variants"] == [[5, 32]]
    assert d["cfg2"]["tasks"] == 7000 and d["cfg2"]["haps"] == [1, 2, 3, 4]
    narrow = plan_summary(PMM_SMALL_JOB_WIDENING="0")
    assert narrow["toy"]["tasks"] == 15 and narrow["toy"]["variants"] == [[19, 8]]
    assert narrow["cfg2"] == d["cfg2"]                          # not a small job
    flat = plan_summary(PMM_RUN_TIERS="0")
    assert flat["cfg2"]["tasks"] == 16000 and flat["cfg2"]["haps"] == [1]
    assert flat["toy"] == d["toy"]


@pytest.mark.gpu
def test_planner_options_stay_with_their_context(built):
    import torch
    from acc_genomics_b200 import engine
    from acc_genomics_b200.engine import PairHMMEngine

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    toy = synth.region(np.random.Generator(np.random.PCG64(11)), [151] * 10, [400] * 5)
    cfg2 = synth.config(2)
    # the defaults' plans, taken before any context's option is set (50 and 7 000 tasks on 148 SMs)
    want_toy, want_cfg2 = len(engine.plan(toy, sm_count=sms)), len(engine.plan(cfg2, sm_count=sms))
    a, b = PairHMMEngine(0), PairHMMEngine(0)
    try:
        def tasks(eng, job):
            eng.stage(job)
            return eng.stats()["f32_tasks"]

        a.set_option("small_job_widening", "off")
        assert tasks(b, toy) == want_toy
        assert tasks(a, toy) == 15                              # 3 groups of 4 reads at 19 x 8, one haplotype per task
        a.set_option("run_tiers", "0")
        assert tasks(b, cfg2) == want_cfg2
        assert tasks(a, cfg2) == 16000                          # 250 groups x 64 haplotypes, one per task
        # pmm_plan_flat keeps planning from the defaults
        assert len(engine.plan(toy, sm_count=sms)) == want_toy and len(engine.plan(cfg2, sm_count=sms)) == want_cfg2
    finally:
        a.close(); b.close()
