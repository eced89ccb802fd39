"""The multi-GPU work queue (pmm_pool_*): many regions in flight over every visible GPU, results identical to the
single-context path and to the oracle.  Runs on one GPU too (the feeders then share it)."""
import numpy as np
import pytest

from acc_genomics_b200 import synth
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu


def test_pool_matches_oracle_and_spreads_jobs(built, checker):
    from acc_genomics_b200.engine import PairHMMPool
    pool = PairHMMPool(contexts_per_device=2)
    regions = synth.config(5, scale=0.008, seed=11)                     # 20 ragged regions
    jobs = [regions[k:k + 2] for k in range(0, len(regions), 2)]        # 10 jobs of 2 regions
    tickets = [pool.submit(j) for j in jobs]
    for j, t in zip(jobs, tickets):
        out, nfb, dev = pool.wait(t)
        want = np.concatenate([checker.batch(b, threads=8)[1].ravel() for b in j])
        assert_bits_equal(out, want, "pool job")
        assert 0 <= dev
    load = pool.device_load()
    assert sum(d["jobs"] for d in load) == len(jobs)
    assert sum(d["cells"] for d in load) == sum(b.num_cells for b in regions)
    if pool.num_devices > 1:
        assert all(d["jobs"] > 0 for d in load), load
    pool.close()


def test_pool_rejects_bad_jobs(built):
    from acc_genomics_b200.engine import PairHMMPool, PmmError
    pool = PairHMMPool(devices=[0], contexts_per_device=1)
    b = synth.config(1, scale=0.1)[0]
    with pytest.raises(PmmError):
        pool.submit(b, out=np.empty(3, dtype=np.float64))                # output too small
    with pytest.raises(PmmError):
        pool.wait(12345)                                                 # unknown ticket
    t = pool.submit(b)
    out, _, _ = pool.wait(t)
    assert np.isfinite(out).all()
    pool.close()
    with pytest.raises(PmmError):
        PairHMMPool(devices=[99])


def test_many_small_jobs_queued_at_once(built, checker):
    """Many small jobs queued at once on one context: every caller gets exactly its own results and its own fallback
    count, in the first round and in a second that reuses the context's buffers."""
    from acc_genomics_b200.engine import PairHMMPool
    pool = PairHMMPool(devices=[0], contexts_per_device=1)
    regions = synth.config(5, scale=0.016, seed=12)                      # 40 regions
    regions += [synth.config(3, scale=0.02, seed=13)[0]]                 # one fallback-heavy region
    want = [checker.batch(b, threads=8) for b in regions]
    for rep in range(2):                                                 # second round: buffers reused
        tickets = [pool.submit(b) for b in regions]
        for b, t, (_, out_r, fb_r) in zip(regions, tickets, want):
            out, nfb, _ = pool.wait(t)
            assert_bits_equal(out, out_r.ravel(), f"small job, round {rep}")
            assert nfb == int(fb_r.sum())
    pool.close()


def test_bad_job_fails_alone_and_trace_has_one_record_per_job(built, checker):
    """A malformed job (a read of length 0) is refused at submit time and never reaches a GPU; the good jobs queued
    around it run, and the pool's timeline has one record per job with sane times."""
    from acc_genomics_b200.engine import PairHMMPool, PmmError, concat_regions
    pool = PairHMMPool(devices=[0], contexts_per_device=2)
    pool.trace(True)
    regions = synth.config(5, scale=0.004, seed=21)
    tickets = [pool.submit(b) for b in regions[:5]]
    bad = concat_regions([regions[5]])
    bad["read_off"] = bad["read_off"].copy(); bad["read_off"][3] = bad["read_off"][2]          # read 2 has length 0
    with pytest.raises(PmmError):
        pool.submit(None, job=bad)
    tickets += [pool.submit(b) for b in regions[5:]]
    for b, t in zip(regions, tickets):
        out, nfb, _ = pool.wait(t)
        assert_bits_equal(out, checker.batch(b, threads=8)[1].ravel(), "job next to a refused one")
    pool.trace(False)
    tr = pool.get_trace()
    assert len(tr) == len(regions) and sum(r["cells"] for r in tr) == sum(b.num_cells for b in regions)
    for r in tr:
        assert r["t_take"] <= r["t_staged"] <= r["t_launched"] <= r["t_fetched"]
        assert r["d_start"] <= r["d_f32_end"] <= r["d_end"]
        assert r["t_take"] - 0.05 <= r["d_start"] and r["d_end"] <= r["t_fetched"] + 0.05      # device and host clocks line up
    pool.close()


@pytest.mark.parametrize("contexts,sync", [(3, "spin"), (4, "auto"), (2, "block"), (5, "hybrid")])
def test_every_feeder_shape_and_wait_mode_gives_the_same_answers(built, checker, contexts, sync, monkeypatch):
    """Feeders drive their contexts in pairs (an odd one out alone); waits spin, sleep, poll or pick by themselves: the
    results are the oracle's either way, and every job is accounted for once."""
    from acc_genomics_b200.engine import PairHMMPool
    monkeypatch.setenv("PMM_POOL_SYNC", sync)
    pool = PairHMMPool(devices=[0], contexts_per_device=contexts)
    regions = synth.config(5, scale=0.012, seed=31)                      # 30 ragged regions
    jobs = [regions[k:k + 3] for k in range(0, len(regions), 3)] * 2     # 20 jobs, every one twice
    want = [np.concatenate([checker.batch(b, threads=8)[1].ravel() for b in j]) for j in jobs[:10]] * 2
    tickets = [pool.submit(j) for j in jobs]
    for w, t in zip(want, tickets):
        out, _, dev = pool.wait(t)
        assert_bits_equal(out, w, f"{contexts} contexts, {sync}")
    assert sum(d["jobs"] for d in pool.device_load()) == len(jobs)
    pool.close()
