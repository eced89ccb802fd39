"""Smith-Waterman on the GPU at its edges: every weight set GATK uses plus tie-heavy and extreme ones, both builds of the
kernel (with and without the -10^8 clamp), all 256 byte values, long gaps and diagonal runs at the traceback's tile
borders, every row-block shape against the loop-entry column counts, batches that run in several chunks, truncated CIGAR
rows and the weight domain.  Offset, CIGAR and score must equal the oracle's."""
import ctypes as C
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
from acc_genomics_b200 import sw

pytestmark = pytest.mark.gpu

STRATEGIES = (sw.SOFTCLIP, sw.INDEL, sw.LEADING_INDEL, sw.IGNORE)
GATK_WEIGHTS = [(200, -150, -260, -11), (3, -1, -4, -3), (25, -50, -110, -6), (10, -15, -30, -5)]
W = 1 << 16                                   # the largest |weight| sw_align_batch accepts
CUTOFF = -100_000_000                         # MATRIX_MIN_CUTOFF
MAX_LEN = 4095
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
# homopolymers and tandem repeats: many equal scores (as test_gpu_sw.test_repeats_and_ties)
TIES = [(b"A" * 60, b"A" * 37), (b"AC" * 40, b"AC" * 31 + b"A"), (b"ACG" * 30, b"ACG" * 12 + b"T" + b"ACG" * 10),
        (b"T" * 100, b"T" * 100), (b"GATTACA" * 12, b"GATTACA" * 5 + b"GATACA" + b"GATTACA" * 4), (b"C" * 9, b"G" * 9),
        (b"ACGT" * 25, b"TGCA" * 25), (b"A" * 200 + b"C" * 50, b"C" * 50 + b"A" * 200)]


@pytest.fixture(scope="module")
def aligner(built):
    a = sw.SmithWaterman(0)
    yield a
    a.close()


_local = threading.local()


def _port_align(pair, strategy, weights):
    if not hasattr(_local, "port"):
        _local.port = oracle.sw_port()        # one instance per thread: its CIGAR buffers are its own
    return _local.port.align_scored(pair[0], pair[1], strategy, weights)


def expected(pairs, strategy, weights):
    """The oracle's (offset, cigar, score) for every pair, each distinct pair computed once.  The C restatement runs
    outside the GIL, so distinct pairs go to a few threads.  Where the reference's own code is built and both sequences
    fit its 1536-base buffers, offset and CIGAR come from it (it reports no score)."""
    distinct = list(dict.fromkeys(pairs))
    with ThreadPoolExecutor(max(1, min(8, os.cpu_count() or 1))) as ex:
        res = dict(zip(distinct, ex.map(lambda p: _port_align(p, strategy, weights), distinct)))
    ref = oracle.sw_reference()
    if ref is not None:
        for p in distinct:
            if len(p[0]) <= 1536 and len(p[1]) <= 1536:
                res[p] = ref.align(p[0], p[1], strategy, weights) + (res[p][2],)
    return [res[p] for p in pairs]


def check(al, pairs, strategy, weights=sw.DEFAULT_WEIGHTS, cigar_cap=64):
    got = al.align(pairs, strategy, weights, cigar_cap=cigar_cap)
    for k, ((r, a), g, w) in enumerate(zip(pairs, got, expected(pairs, strategy, weights))):
        assert g == w, (f"pair {k} strategy {strategy} weights {weights} ref {len(r)} alt {len(a)}: "
                        f"{sw.cigar_string(g[1])} @ {g[0]} score {g[2]} vs {sw.cigar_string(w[1])} @ {w[0]} score {w[2]}")
    return got


def clamp_can_act(L: int, weights) -> bool:
    """launch_align's choice of the kernel build (sw_kernels.cu), restated: with L the longest sequence of the chunk, can
    any diagonal term reach the -10^8 clamp?"""
    match, mismatch, open_, extend = weights
    bmin = min(0, open_, open_ + (L - 1) * extend)
    return bmin + (L + 1) * min(match, mismatch, 0) <= CUTOFF


def pick_rows_per_lane(l1: int) -> int:
    """sw_kernels.cu's pick_rows_per_lane, restated: K rows per lane, blocks of 32 K rows."""
    nblk = -(-l1 // (32 * 14))
    k = -(-(-(-l1 // nblk)) // 32)
    return min(v for v in (4, 6, 8, 10, 12, 14) if v >= k)


def mutate(rng, s: bytes, sub=0.03, indel=0.01) -> bytes:
    out, k = bytearray(), 0
    while k < len(s):
        u = rng.random()
        if u < sub:
            out.append(int(ACGT[rng.integers(0, 4)])); k += 1
        elif u < sub + indel:
            out += ACGT[rng.integers(0, 4, int(rng.integers(1, 6)))].tobytes()
        elif u < sub + 2 * indel:
            k += int(rng.integers(1, 6))
        else:
            out.append(s[k]); k += 1
    return bytes(out) or s[:1]


def random_acgt(rng, n: int) -> bytes:
    return ACGT[rng.integers(0, 4, n)].tobytes()


# ---- weights --------------------------------------------------------------------------------------------------------
DEGENERATE_WEIGHTS = [(0, 0, 0, 0), (7, 7, -9, -3), (10, -10, -1, -20), (10, -20, 5, 3), (-5, -10, -20, -2), (-3, 4, -6, -1),
                      (W, -W, -W, -W), (W, W, W, W), (-W, -W, -W, -W), (-W, W, -W, W), (1, -W, W, -1)]


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_weight_grid(aligner, strategy):
    """GATK's four parameter sets, sets made of ties (all zero, match == mismatch, opening cheaper than extending),
    positive gaps, a negative match and corners of the weight domain, on haplotype pairs and repeats."""
    pairs = sw.haplotype_pairs(41 + strategy, 48, ref_len=(60, 220), per_ref=8) + TIES
    for w in GATK_WEIGHTS + DEGENERATE_WEIGHTS:
        got = check(aligner, pairs, strategy, w)
        if w in GATK_WEIGHTS and strategy != sw.IGNORE:
            # the reported score is the score of the returned alignment
            for (r, a), (off, cig, score) in zip(pairs, got):
                assert oracle.sw_rescore(r, a, w, off, cig) == score, (w, strategy, sw.cigar_string(cig), off)


# ---- the -10^8 clamp ------------------------------------------------------------------------------------------------
def test_both_kernel_builds_and_the_clamp(aligner):
    """The host launches the kernel without the clamp when no diagonal term can reach -10^8.  Cases one unit either side
    of that bound (in weight and in length) run both builds; in the cases where the clamp acts, INDEL and LEADING_INDEL
    scores of -10^8 prove it did (without it, A x 3000 against C x 3000 would score about -1.97e8)."""
    rng = np.random.Generator(np.random.PCG64(8))
    cases = []                                  # (pairs, weights): every pair of a case runs in one chunk

    def longest(L):                             # a batch whose longest sequence has exactly L bases
        r = random_acgt(rng, L)
        return [(r, mutate(rng, r)[:L]), (b"A" * L, b"C" * (L - 3)), (r[:300], r[40:250])]

    cases += [(longest(1999), (1, -49999, -2000, 0)), (longest(1999), (1, -49999, -1999, 0)),
              (longest(1999), (1, -50000, 0, 0)), (longest(1998), (1, -50000, 0, 0))]
    acting = [(b"A" * 3000, b"C" * 3000), (b"AC" * 2000, b"GT" * 1100), (b"G" * MAX_LEN, b"T" * 2000), (b"T" * 1700, b"A" * 3900)]
    cases += [(acting, (1, -W, -W, -W)), (acting[:2], (W, -W // 2, -W, -30000))]
    sides = set()
    for pairs, w in cases:
        L = max(max(len(r), len(a)) for r, a in pairs)
        sides.add(clamp_can_act(L, w))
        for st in STRATEGIES:
            got = check(aligner, pairs, st, w)
            if w == (1, -W, -W, -W) and st in (sw.INDEL, sw.LEADING_INDEL):
                assert got[0][2] == CUTOFF, got[0][2]           # A x 3000 / C x 3000: the clamped corner
    assert sides == {True, False}
    assert clamp_can_act(1999, (1, -49999, -2000, 0)) and not clamp_can_act(1999, (1, -49999, -1999, 0))
    assert clamp_can_act(1999, (1, -50000, 0, 0)) and not clamp_can_act(1998, (1, -50000, 0, 0))


# ---- bytes ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_all_byte_values(aligner, strategy):
    """Bases are compared as bytes: all 256 values in both sequences, runs of N, lowercase against uppercase, 0x00 and
    0xFF at the first and last positions (the fill pads rows past the matrix with -1)."""
    rng = np.random.Generator(np.random.PCG64(256 + strategy))
    every = bytes(rng.permutation(256).astype(np.uint8))
    pairs = []
    for k in range(10):
        ref = bytearray(random_acgt(rng, int(rng.integers(100, 400))))
        ref[int(rng.integers(0, len(ref))):0] = every
        ref[int(rng.integers(0, len(ref))):0] = b"N" * int(rng.integers(5, 40))
        ref = bytes(ref)
        alt = bytearray(mutate(rng, ref, sub=0.02, indel=0.01))
        # substitutions by any byte, lowercase copies of stretches, N runs
        for p in rng.integers(0, len(alt), 12):
            alt[p] = int(rng.integers(0, 256))
        a0 = int(rng.integers(0, len(alt) - 30))
        alt[a0:a0 + 30] = bytes(alt[a0:a0 + 30]).lower()
        a1 = int(rng.integers(0, len(alt) - 20))
        alt[a1:a1 + 20] = b"N" * 20
        alt[int(rng.integers(0, len(alt))):0] = every[::-1]
        ends = [(0x00, 0xFF), (0xFF, 0x00), (0x00, 0x00), (0xFF, 0xFF)][k % 4]
        ref = bytes([ends[0]]) + ref[1:-1] + bytes([ends[1]])
        alt = bytes([ends[1]]) + bytes(alt[1:-1]) + bytes([ends[0]])
        pairs.append((ref, alt))
    pairs += [(every, every), (every, every[::-1]), (b"\x00" * 40, b"\xff" * 40), (b"\xff" * 33 + b"\x00", b"\xff" * 34),
              (b"n" * 50 + b"ACGT" * 10, b"N" * 50 + b"acgt" * 10), (b"\x00", b"\x00"), (b"\xff", b"\x00")]
    assert all(len(set(r)) == 256 and len(set(a)) == 256 for r, a in pairs[:10])
    for w in (sw.DEFAULT_WEIGHTS, (3, -1, -4, -3)):
        check(aligner, pairs, strategy, w)


# ---- traceback tiles ------------------------------------------------------------------------------------------------
def _distinct_from_neighbours(rng, left: int, right: int) -> int:
    return int(rng.choice([b for b in ACGT if b != left and b != right]))


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_long_gaps_and_runs_at_tile_edges(aligner, strategy):
    """The traceback reads 32-row x 64-column tiles.  Deletions of 31 .. 500 bases starting at rows = 0, 1, 31 (mod 32),
    insertions of 63 .. 300 bases starting at columns = 0, 1, 63 (mod 64), and diagonal runs of exactly 31, 32 and 33
    cells between one-base gaps.  The weights make the long gap the optimum: the CIGAR must hold it."""
    rng = np.random.Generator(np.random.PCG64(3232))
    ref = random_acgt(rng, 1400)
    w = (200, -150, -260, -1)
    pairs, want_elem = [], []
    for d in (31, 32, 33, 64, 100, 500):
        for res in (0, 1, 31):
            s = 32 * 12 + res                           # 1-based row of the first deleted base
            pairs.append((ref, ref[:s - 1] + ref[s - 1 + d:])); want_elem.append((d, 2))
    for n in (63, 64, 65, 130, 300):
        for res in (0, 1, 63):
            c = 64 * 6 + res                            # 1-based column of the first inserted base
            pairs.append((ref, ref[:c - 1] + random_acgt(rng, n) + ref[c - 1:])); want_elem.append((n, 1))
    for k in (31, 32, 33):
        # one-base deletions after every k reference bases, the deleted base unlike its neighbours (no equivalent shift)
        r = bytearray(random_acgt(rng, 1300))
        alt = bytearray()
        for p in range(0, len(r) - k - 2, k + 1):
            q = p + k
            r[q] = _distinct_from_neighbours(rng, r[q - 1], r[q + 1])
            alt += r[p:q]
        pairs.append((bytes(r), bytes(alt))); want_elem.append((k, 0))
        # one-base insertions after every k alternate bases
        r2 = random_acgt(rng, 1300)
        alt = bytearray()
        for p in range(0, len(r2) - k, k):
            alt += r2[p:p + k]
            alt.append(_distinct_from_neighbours(rng, r2[p + k - 1], r2[p + k]))
        pairs.append((r2, bytes(alt))); want_elem.append((k, 0))
    got = check(aligner, pairs, strategy, w)
    for (r, a), (_, cig, _), e in zip(pairs, got, want_elem):
        if e[1] == 0:                                   # most runs are exactly k long
            assert sum(1 for x in cig if x == e) >= len(r) // (e[0] + 1) // 2, (e, sw.cigar_string(cig))
        else:
            assert e in cig, (e, sw.cigar_string(cig))
    # the same gaps under GATK's default weights too
    check(aligner, pairs, strategy)


# ---- shapes ---------------------------------------------------------------------------------------------------------
def _shape_rows():
    """Row counts at the edges (last row, and one either side) of every (blocks, K) combination pick_rows_per_lane
    produces up to 4095 rows."""
    combos = {}
    for l1 in range(1, MAX_LEN + 1):
        K = pick_rows_per_lane(l1)
        combos.setdefault((-(-l1 // (32 * K)), K), []).append(l1)
    rows = set()
    for ls in combos.values():
        for e in (ls[0], ls[-1]):
            rows.update(x for x in (e - 1, e, e + 1) if 1 <= x <= MAX_LEN)
    return combos, sorted(rows)


def test_shapes_every_row_block_against_loop_entry_columns(aligner):
    """The steady 8-step loop runs from 40 columns on; 1, 2, 31 .. 49 and 4095 columns against every row-block shape."""
    combos, rows = _shape_rows()
    assert len(combos) > 10 and all(any(x in rows for x in ls) for ls in combos.values())
    rng = np.random.Generator(np.random.PCG64(4095))
    by_strategy = {st: [] for st in STRATEGIES}
    for n1 in rows:
        ref = random_acgt(rng, n1)
        for n2 in (1, 2, 31, 32, 33, 39, 40, 41, 47, 48, 49, MAX_LEN):
            alt = mutate(rng, ref)
            alt = (alt * (n2 // len(alt) + 1))[:n2]
            if rng.random() < 0.5 and n2 < n1:
                s = int(rng.integers(0, n1 - n2 + 1))
                alt = mutate(rng, ref[s:s + n2])[:n2] or ref[s:s + 1]
            by_strategy[STRATEGIES[(n1 + n2) % 4]].append((ref, alt))
    for st, pairs in by_strategy.items():
        check(aligner, pairs, st)


# ---- chunks ---------------------------------------------------------------------------------------------------------
def test_batches_in_several_chunks(built):
    """A batch whose backtrack matrices exceed the 2^30-word budget runs as several launches, which share the compact
    CIGAR cursor.  Then, on the same context, a batch whose CIGARs overflow the compact estimate while in several chunks,
    so the engine repeats it with room for everything."""
    rng = np.random.Generator(np.random.PCG64(1 << 30))
    a = sw.SmithWaterman(0)
    try:
        big = []
        for k in range(4):
            r = random_acgt(rng, MAX_LEN)
            big.append((r, (mutate(rng, r) + r)[:MAX_LEN - 3 * k]))
        small = sw.haplotype_pairs(5, 40, ref_len=(30, 200), per_ref=8)
        pairs = []
        for k in range(1000):
            pairs.append(big[k % 4])
            if k % 5 == 0:
                pairs.append(small[(k // 5) % len(small)])
        check(a, pairs, sw.SOFTCLIP)
        st = a.stats()
        print(f"chunks: {st['chunks']}, kernel launches: {st['kernel_launches']}, backtrack bytes: {st['bytes_backtrack']}")
        assert st["chunks"] >= 2 and st["kernel_launches"] == st["chunks"] and st["pairs"] == len(pairs)

        noisy = [(r[:MAX_LEN], alt[:MAX_LEN]) for r, alt in sw.haplotype_pairs(6, 4, ref_len=MAX_LEN, per_ref=1, sub=0.06, indel=0.05)]
        pairs = []
        for k in range(1000):
            pairs.append(noisy[k % 4])
            if k % 5 == 0:
                pairs.append(small[(k // 5) % len(small)])
        got = check(a, pairs, sw.INDEL, cigar_cap=4096)
        total = sum(len(c) for _, c, _ in got)
        assert total > max(16 * len(pairs), 1 << 16), f"{total} CIGAR elements: the compact estimate was not exceeded"
        st = a.stats()
        print(f"chunks: {st['chunks']}, CIGAR elements: {total}")
        assert st["chunks"] >= 2 and st["pairs"] == len(pairs)
    finally:
        a.close()


# ---- truncated rows -------------------------------------------------------------------------------------------------
def _call(al, pairs, weights, strategy, cigar_cap, cig, ne, off, sc):
    blob1, blob2 = b"".join(r for r, _ in pairs), b"".join(a for _, a in pairs)
    l1 = np.array([len(r) for r, _ in pairs], np.uint32); l2 = np.array([len(a) for _, a in pairs], np.uint32)
    s1 = np.concatenate([[0], np.cumsum(l1)[:-1]]).astype(np.uint32); s2 = np.concatenate([[0], np.cumsum(l2)[:-1]]).astype(np.uint32)
    b1 = np.frombuffer(blob1, np.uint8); b2 = np.frombuffer(blob2, np.uint8)
    return al.lib.sw_align_batch(al.h, len(pairs), b1.ctypes.data, s1.ctypes.data, l1.ctypes.data, b2.ctypes.data, s2.ctypes.data,
                                 l2.ctypes.data, *weights, strategy, cigar_cap, cig.ctypes.data, ne.ctypes.data, off.ctypes.data,
                                 sc.ctypes.data if sc is not None else None)


def test_truncated_cigar_rows(aligner):
    """Through the C ABI (SmithWaterman.align retries): with cigar_cap smaller than a CIGAR, n_elem is the full count,
    the row holds the last cigar_cap elements in forward order, and nothing past min(n_elem, cigar_cap) is touched."""
    pairs = sw.haplotype_pairs(12, 24, ref_len=(150, 600), per_ref=6, sub=0.04, indel=0.03) + [(b"ACGT" * 20, b"ACGT" * 20)]
    cap = 5
    for st in STRATEGIES:
        want = expected(pairs, st, sw.DEFAULT_WEIGHTS)
        assert any(len(c) > cap for _, c, _ in want) and any(len(c) < cap for _, c, _ in want)
        cig = np.full((len(pairs), cap, 2), -7, np.int32)
        ne = np.full(len(pairs), -7, np.int32); off = np.full(len(pairs), -7, np.int32); sc = np.full(len(pairs), -7, np.int32)
        assert _call(aligner, pairs, sw.DEFAULT_WEIGHTS, st, cap, cig, ne, off, sc) == sw.SW_OK
        for p, (w_off, w_cig, w_sc) in enumerate(want):
            stored = min(len(w_cig), cap)
            assert (ne[p], off[p], sc[p]) == (len(w_cig), w_off, w_sc), p
            assert [tuple(e) for e in cig[p, :stored].tolist()] == w_cig[len(w_cig) - stored:], (p, cig[p], w_cig)
            assert (cig[p, stored:] == -7).all(), (p, cig[p])
        # a NULL score array is allowed
        assert _call(aligner, pairs, sw.DEFAULT_WEIGHTS, st, cap, cig, ne, off, None) == sw.SW_OK
        assert ne.tolist() == [len(c) for _, c, _ in want]


# ---- weight domain --------------------------------------------------------------------------------------------------
def test_weight_domain(aligner):
    """|weight| <= 2^16 is accepted and matches the oracle at the corners (with 4095-base sequences, where scores are
    largest); one past the domain, INT_MIN and INT_MAX are rejected with SW_ERR_INVALID."""
    imin, imax = -(1 << 31), (1 << 31) - 1
    for pos in range(4):
        for v in (W + 1, -W - 1, imin, imax):
            w = list(sw.DEFAULT_WEIGHTS); w[pos] = v
            with pytest.raises(sw.SwError, match="weight"):
                aligner.align([(b"ACGT", b"ACGT")], sw.SOFTCLIP, tuple(w))
            cig = np.zeros((1, 4, 2), np.int32); ne = np.zeros(1, np.int32); off = np.zeros(1, np.int32)
            assert _call(aligner, [(b"ACGT", b"ACGT")], w, sw.SOFTCLIP, 4, cig, ne, off, None) == 1    # SW_ERR_INVALID
    rng = np.random.Generator(np.random.PCG64(65536))
    small = sw.haplotype_pairs(17, 24, ref_len=(40, 160), per_ref=6) + TIES[:4]
    corners = [(W * a, W * b, W * c, W * d) for a in (1, -1) for b in (1, -1) for c in (1, -1) for d in (1, -1)]
    assert len(set(corners)) == 16
    for k, w in enumerate(corners):
        check(aligner, small, STRATEGIES[k % 4], w)
    r = random_acgt(rng, MAX_LEN)
    longest = [(r, mutate(rng, r)[:MAX_LEN]), (r, r)]
    for w in ((W, W, W, W), (-W, -W, -W, -W), (W, -W, -W, -W)):
        for st in STRATEGIES:
            check(aligner, longest, st, w)
