"""BWA-MEM seed extension on the GPU (sw_extend_batch): every field of every job, and the number of DP cells visited,
must equal the oracle's (oracle/ksw_oracle.c, a restatement of ksw_extend2 of bwa 0.7.17).  BWA-like jobs, random
matrices and gaps, the band and chunk edges of the kernel (32 columns per chunk), every way a job ends, and the
domain of the C ABI."""
import ctypes as C

import numpy as np
import pytest

from oracle import ksw
from acc_genomics_b200 import sw

pytestmark = pytest.mark.gpu

ENC = {c: i for i, c in enumerate("ACGTN")}
BWA = (5, sw.bwa_matrix(), 6, 1, 6, 1, 100)          # m, mat, o_del, e_del, o_ins, e_ins, zdrop


def enc(s: str) -> bytes:
    return bytes(ENC[c] for c in s)


@pytest.fixture(scope="module")
def ctx(built):
    a = sw.SmithWaterman(0)
    yield a
    a.close()


def check(ctx, jobs, scoring=BWA):
    """GPU against the oracle, field by field and cell count; returns the results."""
    m, mat, o_del, e_del, o_ins, e_ins, zdrop = scoring
    got = ctx.extend(jobs, mat, m, o_del, e_del, o_ins, e_ins, zdrop)
    want, cells = ksw.extend_batch(jobs, m, mat, o_del, e_del, o_ins, e_ins, zdrop)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert len(bad) == 0, [(int(k), len(jobs[k][0]), len(jobs[k][1]), jobs[k][2:], got[k].tolist(), want[k].tolist())
                           for k in bad[:5]]
    st = ctx.stats()
    assert st["pairs"] == len(jobs) and st["cells"] == int(cells.sum()), (st, int(cells.sum()))
    assert st["kernel_launches"] == 1 and st["chunks"] == 1 and st["bytes_backtrack"] == 0
    return got


def related(rng, m, n, like=None, p=0.9):
    """n bytes < m; copies of `like` with substitutions when given."""
    s = rng.integers(0, m, n).astype(np.uint8)
    if like is not None:
        k = min(n, len(like))
        s[:k] = np.where(rng.random(k) < p, np.frombuffer(like[:k], np.uint8), s[:k])
    return s.tobytes()


def test_worked_cases(ctx):
    table = [("ACGTACGTAC", "ACGTACGTAC", 20, 100, (30, 10, 10, 10, 30, 0)),
             ("ACGTACGTAC", "ACGTACGTACGGGG", 20, 100, (30, 10, 10, 10, 30, 0)),
             ("ACGTAGGTAC", "ACGTACGTAC", 20, 100, (25, 5, 5, 10, 25, 0)),
             ("ACGTACGTAC", "ACGTACCGTAC", 20, 100, (26, 6, 6, 11, 23, 0)),
             ("AAAAAAAAAA", "CCCCCCCCCC", 3, 100, (3, 0, 0, 1, 0, 0)),
             ("ACGTACGTAC", "ACGTACGTAC", 20, 0, (30, 10, 10, 10, 30, 0))]
    got = check(ctx, [(enc(q), enc(t), h0, w, 5) for q, t, h0, w, _ in table])
    assert [tuple(r) for r in got.tolist()] == [want for *_, want in table]
    assert ctx.stats()["cells"] == 100 + 134 + 100 + 110 + 10 + 10


def test_bwa_like_jobs(ctx):
    jobs = sw.extension_jobs(20000, 20000)
    got = check(ctx, jobs)
    assert (got[:, 1] == np.array([len(j[0]) for j in jobs])).mean() > 0.7
    # and a batch of 150-base reads with more errors
    check(ctx, sw.extension_jobs(7, 4000, read_len=250, sub=0.06, indel=0.01))


def test_random_matrices_gaps_and_zdrop(ctx):
    """Alphabets of 1 .. 16 letters with random matrices, asymmetric gap penalties, Z-drop off (<= 0) and small enough to
    act, on related and unrelated sequences."""
    rng = np.random.Generator(np.random.PCG64(1616))
    for k in range(48):
        m = 1 + k % 16
        if k % 3 == 0:
            mat = rng.integers(-128, 128, m * m).astype(np.int8)
        else:
            a, b = int(rng.integers(1, 8)), int(rng.integers(1, 12))
            mat = np.array([a if x == y else -b for x in range(m) for y in range(m)], np.int8)
        gaps = (int(rng.integers(0, 20)), int(rng.integers(1, 6)), int(rng.integers(0, 20)), int(rng.integers(1, 6)))
        zdrop = [-5, 0, 1, 5, 20, 100][k % 6]
        jobs = []
        for _ in range(60):
            q = related(rng, m, int(rng.integers(1, 300)))
            t = related(rng, m, int(rng.integers(1, 400)), q if rng.random() < 0.7 else None, float(rng.uniform(0.6, 1.0)))
            jobs.append((q, t, int(rng.integers(1, 80)), int(rng.choice([0, 5, 30, 100, 1000])), int(rng.integers(0, 20))))
        check(ctx, jobs, (m, mat, *gaps, zdrop))


def test_band_and_chunk_edges(ctx):
    """w of 0, 1, 15, 16, 31, 32, 33, 47, 48 and large (rows of 2w + 1 = 32k +- 1 columns); query lengths at the
    32-column chunk boundaries against targets of 1 base, shorter, equal and far longer; h0 of 1 and 2^24."""
    rng = np.random.Generator(np.random.PCG64(3232))
    jobs = []
    for qlen in (1, 2, 31, 32, 33, 63, 64, 65, 95, 96, 97, 4095):
        q = related(rng, 4, qlen)
        for tlen in sorted({1, max(1, qlen // 2), qlen, 4 * qlen + 50}):
            t = related(rng, 4, tlen, q, 0.95)
            for w in (0, 1, 15, 16, 31, 32, 33, 47, 48, 65535):
                for h0 in (1, 30, 1 << 24):
                    jobs.append((q, t, h0, w, 5))
    check(ctx, jobs)
    # no Z-drop and a bonus that keeps w: the bands stay as wide as the query
    check(ctx, jobs[::3], (5, sw.bwa_matrix(), 6, 1, 6, 1, 0))


def test_how_jobs_end(ctx):
    """Jobs that end by an all-zero row, by Z-drop, by running out of target, by an empty band (beg >= end), and jobs
    whose gscore stays -1 (no row reaches the end of the query)."""
    rng = np.random.Generator(np.random.PCG64(99))
    jobs = []
    for _ in range(40):
        q = related(rng, 4, int(rng.integers(20, 200)))
        jobs.append((q, bytes((b + 1) % 4 for b in q), 3, 100, 5))                        # all-zero row soon
        tail = related(rng, 4, 300)
        jobs.append((q, q[:len(q) // 2] + tail, 20, 100, 5))                                # Z-drop in the tail
        jobs.append((q, q[:int(rng.integers(1, len(q)))], 20, 100, 5))                     # out of target
        jobs.append((q, q + related(rng, 4, 50), 20, 0, 5))                                # band empties past the query
        jobs.append((q + related(rng, 4, 400), q[:10], 15, 100, 5))                       # gscore stays -1
    got = check(ctx, jobs)
    assert (got[4::5, 4] == -1).all()
    assert (got[:, 4] >= 0).any()
    check(ctx, jobs, (5, sw.bwa_matrix(), 6, 1, 6, 1, 3))                                   # Z-drop acting often


def test_mixed_job_parameters_in_one_batch(ctx):
    rng = np.random.Generator(np.random.PCG64(5))
    base = sw.extension_jobs(55, 3000)
    jobs = [(q, t, int(rng.integers(1, 200)), int(rng.choice([0, 3, 17, 32, 100, 500])), int(rng.integers(0, 40)))
            for q, t, *_ in base]
    check(ctx, jobs)


def test_largest_jobs(ctx):
    """The largest query and target the domain admits, with h0 = 2^24 (every cell of the band stays positive)."""
    rng = np.random.Generator(np.random.PCG64(65535))
    q = related(rng, 4, 4095)
    jobs = [(q, related(rng, 4, 65535, q * 16, 0.97), 1 << 24, 65535, 65536),
            (q[:200], related(rng, 4, 65535), 1 << 24, 65535, 0),
            (q[:1], related(rng, 4, 65535), 1, 65535, 5)]
    check(ctx, jobs, (5, sw.bwa_matrix(), 4096, 4096, 4096, 4096, -1))
    check(ctx, jobs[1:], (5, sw.bwa_matrix(), 0, 1, 0, 1, 0))


# ---- domain ---------------------------------------------------------------------------------------------------------
def _raw(ctx, jobs, m, mat, o_del, e_del, o_ins, e_ins, zdrop, out):
    """sw_extend_batch through the C ABI; jobs as (q_start, q_len, t_start, t_len, h0, w, end_bonus) over two blobs."""
    desc = np.array([j[2] for j in jobs], np.int64).astype(np.uint32).reshape(-1, 7)
    qb = np.frombuffer(jobs[0][0], np.uint8); tb = np.frombuffer(jobs[0][1], np.uint8)
    mt = np.ascontiguousarray(mat, np.int8)
    return ctx.lib.sw_extend_batch(ctx.h, len(jobs), qb.ctypes.data, tb.ctypes.data, desc.ctypes.data, m, mt.ctypes.data,
                                   o_del, e_del, o_ins, e_ins, zdrop, out.ctypes.data)


def test_domain(ctx):
    """One step outside each edge of the domain: SW_ERR_INVALID and the output untouched.  At the edges: accepted and
    equal to the oracle (as far as a job of that size is cheap to check)."""
    qbuf, tbuf = bytes(5000), bytes(70000)             # all zero: valid bytes for any m >= 1
    good = (0, 10, 0, 20, 10, 100, 5)

    def run(desc, m=5, mat=None, gaps=(6, 1, 6, 1), zdrop=100, q=qbuf, t=tbuf):
        mat = sw.bwa_matrix() if mat is None else mat
        out = np.full((1, 6), -7, np.int32)
        rc = _raw(ctx, [(q, t, desc)], m, mat, *gaps, zdrop, out)
        return rc, out

    rc, out = run(good)
    assert rc == sw.SW_OK and (out != -7).all()
    outside = []
    for pos, vals in ((1, (0, 4096)), (3, (0, 65536)), (4, (0, (1 << 24) + 1, -1)), (5, (-1, 65536)), (6, (-1, 65537))):
        for v in vals:
            d = list(good); d[pos] = v
            outside.append(dict(desc=tuple(d)))
    for pos, v in ((0, -1), (0, 4097), (1, 0), (1, 4097), (2, -1), (2, 4097), (3, 0), (3, 4097)):
        g = [6, 1, 6, 1]; g[pos] = v
        outside.append(dict(desc=good, gaps=tuple(g)))
    mat17 = np.zeros(17 * 17, np.int8)
    outside += [dict(desc=good, m=0, mat=mat17), dict(desc=good, m=17, mat=mat17),
                dict(desc=good, q=bytes([0] * 9 + [5]) + bytes(4990)),        # a query byte == m
                dict(desc=good, t=bytes([0] * 19 + [5]) + bytes(70000)),      # a target byte == m
                dict(desc=good, m=1, mat=np.ones(1, np.int8), q=bytes([1]) + bytes(4999))]
    for kw in outside:
        rc, out = run(**kw)
        assert rc == 1 and (out == -7).all(), kw                             # SW_ERR_INVALID, nothing written
    # bytes past a job's ranges are not the job's: not checked
    rc, _ = run(good, q=bytes(10) + bytes([9]) * 10, t=bytes(20) + bytes([9]))
    assert rc == sw.SW_OK
    # n_jobs == 0
    assert ctx.lib.sw_extend_batch(ctx.h, 0, None, None, None, 5, None, 6, 1, 6, 1, 100, None) == sw.SW_OK
    # at the edges
    rng = np.random.Generator(np.random.PCG64(16))
    for m in (1, 16):
        mat = rng.integers(-128, 128, m * m).astype(np.int8)
        q = related(rng, m, 300); t = related(rng, m, 500, q)
        for gaps in ((0, 1, 0, 1), (4096, 4096, 4096, 4096), (0, 4096, 4096, 1)):
            check(ctx, [(q, t, 1, 0, 0), (q, t, 1 << 24, 65535, 65536), (q[:1], t[:1], 1, 1, 0)], (m, mat, *gaps, -(1 << 31)))
            check(ctx, [(q, t, 50, 33, 7)], (m, mat, *gaps, (1 << 31) - 1))


def test_shares_the_context_with_the_aligner(built):
    """sw_align_batch, sw_extend_batch, sw_align_batch on one context: both alignments equal a fresh context's."""
    pairs = sw.haplotype_pairs(3, 300, ref_len=(100, 400), per_ref=10)
    fresh = sw.SmithWaterman(0)
    try:
        want = fresh.align(pairs, sw.SOFTCLIP)
    finally:
        fresh.close()
    a = sw.SmithWaterman(0)
    try:
        assert a.align(pairs, sw.SOFTCLIP) == want
        check(a, sw.extension_jobs(8, 5000))
        assert a.align(pairs, sw.SOFTCLIP) == want
        assert a.stats()["pairs"] == len(pairs)
    finally:
        a.close()
