"""GPU box: randomized parity fuzz -- random region shapes, multi-region jobs, every entry point (staged, serialized,
read_t/hap_t, GKL testcases, client/worker/task plugin, pool), exact and fast mode,
PairHMM and Smith-Waterman, each result compared with the oracle (bit-exact where the contract says so).
    python tools/fuzz_gpu.py [seconds] [seed]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import oracle
from acc_genomics_b200 import hostlayer, synth, sw
from acc_genomics_b200 import batch as B
from acc_genomics_b200.engine import PairHMMEngine, PairHMMPool

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 60.0
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
rng = np.random.Generator(np.random.PCG64(seed))
chk = oracle.reference() or oracle.port()
swport = oracle.sw_port()
swchk = oracle.sw_reference() or swport
eng = PairHMMEngine(0); fast = PairHMMEngine(0); fast.set_option("mode", "fast")
pool = PairHMMPool(devices=[0], contexts_per_device=2); pool.set_merge(True)
al = sw.SmithWaterman(0)
t0 = time.time(); it = 0; pairs = 0; swpairs = 0


def rand_region():
    nr, nh = int(rng.integers(1, 24)), int(rng.integers(1, 12))
    style = rng.integers(0, 5)
    if style == 0:   rl = rng.integers(1, 40, nr); hl = rng.integers(1, 60, nh)
    elif style == 1: rl = rng.integers(60, 260, nr); hl = rng.integers(80, 700, nh)
    elif style == 2: rl = np.full(nr, int(rng.integers(100, 160))); hl = rng.integers(250, 620, nh)
    elif style == 3: rl = rng.integers(400, 900, max(1, nr // 6)); hl = rng.integers(500, 1600, max(1, nh // 3))
    else:            rl = rng.integers(1, 300, nr); hl = rng.integers(1, 400, nh)
    return synth.region(rng, [int(x) for x in rl], [int(x) for x in hl], decoy_frac=float(rng.choice([0, 0, 0.5])),
                        low_read_frac=float(rng.choice([0, 0.25])))


def same(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint64 if a.dtype.itemsize == 8 else np.uint32),
                          np.ascontiguousarray(b).view(np.uint64 if b.dtype.itemsize == 8 else np.uint32))


while time.time() - t0 < budget:
    it += 1
    regs = [rand_region() for _ in range(int(rng.integers(1, 5)))]
    # these jobs are small: with widening on they run on the 32- and 16-lane variants, off on the ones large jobs use
    eng.set_option("small_job_widening", str(rng.choice(["on", "off"])))     # eng's own calls only, not the plugin's or the pool's
    want = [chk.batch(b, threads=8) for b in regs]
    pairs += sum(b.num_pairs for b in regs)
    # staged multi-region job, exact
    eng.stage(regs); eng.launch()
    raw = eng.fetch_raw(); out, nfb = eng.fetch_log10(); mask = eng.fetch_fallback_mask()
    assert same(raw, np.concatenate([w[0].ravel() for w in want])), ("raw", it)
    assert same(out, np.concatenate([w[1].ravel() for w in want])), ("log10", it)
    assert np.array_equal(mask, np.concatenate([w[2].ravel() for w in want])), ("mask", it)
    # serialized one-shot and struct entry on the first region
    b0 = regs[0]
    o2, _ = eng.forward_log10_serialized(B.serialize_reads(b0), B.serialize_haps(b0), b0.num_pairs)
    assert same(o2.ravel(), want[0][1].ravel()), ("serialized", it)
    o3, _ = eng.forward_log10_structs(b0)
    assert same(o3.ravel(), want[0][1].ravel()), ("structs", it)
    # GKL-shaped testcase batch over all regions of the job (pointer-sharing pairs, regions found again by the engine)
    tc = []
    for b in regs:
        reads = [tuple(bytes(x) for x in b.read(k)) for k in range(b.num_read)]
        haps = [bytes(b.haplotype(k)) for k in range(b.num_hap)]
        tc += [(r, h) for r in reads for h in haps]
    o4, nfb4 = eng.forward_log10_testcases(tc)
    assert same(o4, np.concatenate([w[1].ravel() for w in want])) and nfb4 == nfb, ("testcases", it)
    # the client path: PairHMMClient + PairHMMWorker over the task plugin, a random number of tiles
    os.environ["PAIRHMM_WORKER_TILES"] = str(int(rng.integers(1, 6)))
    o5, nre = hostlayer.worker_forward(b0)
    assert same(o5, want[0][1].ravel()) and nre == int(want[0][2].sum()), ("worker", it)
    # pool (merging of small jobs included)
    tk = [pool.submit(b) for b in regs]
    for t, w in zip(tk, want):
        assert same(pool.wait(t)[0], w[1].ravel()), ("pool", it)
    # fast mode: same decision, log10 within 1e-5 relative, double results identical
    fast.stage(regs); fast.launch()
    fo, _ = fast.fetch_log10(); fm = fast.fetch_fallback_mask()
    wl = np.concatenate([w[1].ravel() for w in want]); wm = np.concatenate([w[2].ravel() for w in want])
    assert np.array_equal(fm, wm), ("fast mask", it)
    fin = np.isfinite(wl)
    assert np.array_equal(np.isfinite(fo), fin) and (np.abs(fo[fin] - wl[fin]) <= 1e-5 * np.abs(wl[fin])).all(), ("fast tol", it)
    # Smith-Waterman
    n = int(rng.integers(1, 40)); lo = int(rng.integers(1, 300))
    ps = sw.haplotype_pairs(int(rng.integers(1 << 30)), n, ref_len=(lo, lo + int(rng.integers(0, 300))), per_ref=int(rng.integers(1, 9)),
                            sub=float(rng.choice([0.0, 0.03, 0.2])), indel=float(rng.choice([0.0, 0.01, 0.05])))
    st = int(rng.integers(0, 4))
    # weights: GATK's default, small random ones, or anywhere in the accepted domain [-2^16, 2^16] (where the -10^8 clamp
    # can act on long pairs); bytes beyond ACGT: N, lowercase, any byte
    wkind = int(rng.integers(0, 3))
    if wkind == 0:   w = sw.DEFAULT_WEIGHTS
    elif wkind == 1: w = tuple(int(x) for x in rng.integers(-30, 31, 4))
    else:            w = tuple(int(x) for x in rng.integers(-(1 << 16), (1 << 16) + 1, 4))
    if wkind == 2 and rng.random() < 0.3:
        # a long pair and a steep mismatch: the chunk runs the kernel with the clamp, which may act
        w = (w[0], -int(rng.integers(60000, (1 << 16) + 1)), w[2], w[3])
        L = int(rng.integers(1700, 4096))
        r = bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), L))
        ps.append((r, bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), int(rng.integers(1, L + 1))))))
    if rng.random() < 0.3:
        ps = [(r, bytes(x if rng.random() > 0.05 else int(rng.choice([78, 110, 97, 0, 255, int(rng.integers(0, 256))])) for x in a))
              for r, a in ps]
    got = al.align(ps, st, w, cigar_cap=int(rng.choice([2, 16, 64])))
    for (r, a), (off, cig, score) in zip(ps, got):
        sw_want = swport.align_scored(r, a, st, w)
        assert (off, cig, score) == sw_want, ("sw", it, st, w, len(r), len(a))
        if swchk is not swport and len(r) <= 1536 and len(a) <= 1536:
            assert (off, cig) == swchk.align(r, a, st, w), ("sw reference", it, st, w, len(r), len(a))
    swpairs += len(ps)
print(f"fuzz ok: {it} iterations, {pairs} PairHMM pairs, {swpairs} Smith-Waterman pairs, {time.time() - t0:.0f} s, seed {seed}, "
      f"checkers {chk.kind}/{swchk.kind}")
