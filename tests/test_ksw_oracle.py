"""BWA-MEM seed extension oracle (CPU): oracle/ksw_oracle.c, a restatement of ksw_extend2 of bwa 0.7.17, against cases
worked out by hand and against a second, independent transcription of the recurrence in Python."""
import os
import re

import numpy as np
import pytest

from oracle import ksw
from acc_genomics_b200 import sw

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENC = {c: i for i, c in enumerate("ACGTN")}


def enc(s: str) -> bytes:
    return bytes(ENC[c] for c in s)


def ksw_extend2_py(q, t, m, mat, o_del, e_del, o_ins, e_ins, w, end_bonus, zdrop, h0):
    """ksw_extend2 once more, written from the recurrence without looking at the C: (score, qle, tle, gtle, gscore,
    max_off, cells)."""
    qlen, tlen = len(q), len(t)
    H, E = [0] * (qlen + 1), [0] * (qlen + 1)
    H[0] = h0
    H[1] = h0 - (o_ins + e_ins) if h0 > o_ins + e_ins else 0
    j = 2
    while j <= qlen and H[j - 1] > e_ins:
        H[j] = H[j - 1] - e_ins; j += 1
    mx = max([0] + list(mat))
    w = min(w, max(int((qlen * mx + end_bonus - o_ins) / e_ins + 1.), 1), max(int((qlen * mx + end_bonus - o_del) / e_del + 1.), 1))
    best, max_i, max_j, max_ie, gscore, max_off = h0, -1, -1, -1, -1, 0
    beg, end, cells = 0, qlen, 0
    for i in range(tlen):
        beg = max(beg, i - w)
        end = min(end, i + w + 1, qlen)
        h1 = max(h0 - (o_del + e_del * (i + 1)), 0) if beg == 0 else 0
        f, rm, mj = 0, 0, -1
        for j in range(beg, end):
            M, e = H[j], E[j]
            H[j] = h1
            M = M + mat[t[i] * m + q[j]] if M else 0
            h = max(M, e, f)
            h1 = h
            if h >= rm:
                rm, mj = h, j
            E[j] = max(e - e_del, M - o_del - e_del, 0)
            f = max(f - e_ins, M - o_ins - e_ins, 0)
            cells += 1
        H[end], E[end] = h1, 0
        if max(beg, end) == qlen:
            if h1 >= gscore:
                gscore, max_ie = h1, i
        if rm == 0:
            break
        if rm > best:
            best, max_i, max_j = rm, i, mj
            max_off = max(max_off, abs(mj - i))
        elif zdrop > 0:
            di, dj = i - max_i, mj - max_j
            if (best - rm - (di - dj) * e_del if di > dj else best - rm - (dj - di) * e_ins) > zdrop:
                break
        nz = [k for k in range(beg, end + 1) if H[k] or E[k]]
        beg = next((k for k in nz if k < end), end)
        last = max((k for k in nz if k >= beg), default=beg - 1)
        end = min(last + 2, qlen)
    return best, max_j + 1, max_i + 1, max_ie + 1, gscore, max_off, cells


BWA = (5, list(sw.bwa_matrix()), 6, 1, 6, 1)
# query, target, h0, w -> score qle tle gtle gscore max_off, cells (bwa's defaults: end_bonus 5, zdrop 100)
TABLE = [("ACGTACGTAC", "ACGTACGTAC", 20, 100, (30, 10, 10, 10, 30, 0), 100),
         ("ACGTACGTAC", "ACGTACGTACGGGG", 20, 100, (30, 10, 10, 10, 30, 0), 134),
         ("ACGTAGGTAC", "ACGTACGTAC", 20, 100, (25, 5, 5, 10, 25, 0), 100),
         ("ACGTACGTAC", "ACGTACCGTAC", 20, 100, (26, 6, 6, 11, 23, 0), 110),
         ("AAAAAAAAAA", "CCCCCCCCCC", 3, 100, (3, 0, 0, 1, 0, 0), 10),
         ("ACGTACGTAC", "ACGTACGTAC", 20, 0, (30, 10, 10, 10, 30, 0), 10)]


@pytest.mark.parametrize("q,t,h0,w,want,cells", TABLE)
def test_worked_cases(built, q, t, h0, w, want, cells):
    got = ksw.extend(enc(q), enc(t), *BWA, w, 5, 100, h0)
    assert got == want + (cells,)
    assert ksw_extend2_py(enc(q), enc(t), *BWA, w, 5, 100, h0) == want + (cells,)


def random_job(rng):
    """A small job with a random alphabet, matrix, gaps, band, bonus, Z-drop and h0; the target often related to the
    query so that extensions run long."""
    m = int(rng.integers(1, 17))
    mat = [int(x) for x in rng.integers(-12, 13, m * m)]
    if rng.random() < 0.5:                                     # a match / mismatch matrix
        a, b = int(rng.integers(1, 6)), int(rng.integers(1, 9))
        mat = [a if x == y else -b for x in range(m) for y in range(m)]
    qlen, tlen = int(rng.integers(1, 40)), int(rng.integers(1, 60))
    q = rng.integers(0, m, qlen).astype(np.uint8)
    t = rng.integers(0, m, tlen).astype(np.uint8)
    if rng.random() < 0.6:
        k = min(qlen, tlen)
        t[:k] = np.where(rng.random(k) < 0.85, q[:k], t[:k])
    gaps = [int(x) for x in (rng.integers(0, 12), rng.integers(1, 5), rng.integers(0, 12), rng.integers(1, 5))]
    w = int(rng.choice([0, 1, 2, 3, 5, 10, 100]))
    end_bonus = int(rng.integers(0, 10))
    zdrop = int(rng.choice([-1, 0, 1, 3, 10, 100]))
    h0 = int(rng.choice([1, 2, 5, 10, 30, 200]))
    return q.tobytes(), t.tobytes(), m, mat, gaps, w, end_bonus, zdrop, h0


def test_c_oracle_equals_python_transcription(built):
    rng = np.random.Generator(np.random.PCG64(2017))
    gscores = set()
    for _ in range(3000):
        q, t, m, mat, gaps, w, eb, zd, h0 = random_job(rng)
        c = ksw.extend(q, t, m, mat, *gaps, w, eb, zd, h0)
        p = ksw_extend2_py(q, t, m, mat, *gaps, w, eb, zd, h0)
        assert c == p, (q, t, m, mat, gaps, w, eb, zd, h0)
        gscores.add(c[4] == -1)
    assert gscores == {True, False}                        # some jobs never reach the end of the query


def test_batch_entry_equals_single_calls(built):
    jobs = sw.extension_jobs(5, 300)
    got, cells = ksw.extend_batch(jobs, 5, sw.bwa_matrix(), 6, 1, 6, 1, 100)
    for k, (q, t, h0, w, eb) in enumerate(jobs):
        want = ksw.extend(q, t, 5, sw.bwa_matrix(), 6, 1, 6, 1, w, eb, 100, h0)
        assert tuple(got[k]) + (int(cells[k]),) == want, k


def test_extension_jobs_are_bwa_like(built):
    jobs = sw.extension_jobs(3, 2000)
    assert len(jobs) == 2000 and jobs == sw.extension_jobs(3, 2000)
    for q, t, h0, w, eb in jobs:
        assert 1 <= len(q) <= 131 and len(q) <= len(t) <= len(q) + 5 * len(q) + w + 1
        assert 19 <= h0 <= 50 and (w, eb) == (100, 5) and max(q) < 4 and max(t) < 4
    res, _ = ksw.extend_batch(jobs, 5, sw.bwa_matrix(), 6, 1, 6, 1, 100)
    # most extensions run to the end of the read, as for reads that belong where their seed is
    assert (res[:, 1] == np.array([len(j[0]) for j in jobs])).mean() > 0.7


def test_library_exports_sw_extend_batch(built):
    from acc_genomics_b200 import engine
    hdr = open(os.path.join(ROOT, "include", "smithwaterman_cuda.h")).read()
    assert "sw_extend_batch" in re.findall(r"\b(sw_[a-z_]+)\s*\(", hdr)
    assert "sw_extend_batch" in sw.SW_EXPORTS
    assert hasattr(engine.load_library(), "sw_extend_batch")
