"""Smith-Waterman oracle (CPU): the C restatement against the golden vectors minted from the reference's own code,
and against the reference live when oracle/_ref/libsw_ref.so is present (build container, or an AVX2 GPU box)."""
import json
import os

import pytest

import oracle
from acc_genomics_b200 import sw

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sw_golden():
    with open(os.path.join(ROOT, "tests", "golden", "sw_golden.json")) as f:
        return json.load(f)


def test_port_reproduces_golden_vectors(built, sw_golden):
    port = oracle.sw_port()
    assert len(sw_golden) > 150
    for c in sw_golden:
        off, cig = port.align(c["ref"].encode(), c["alt"].encode(), c["strategy"], tuple(c.get("weights", oracle.SW_WEIGHTS)))
        assert off == c["offset"] and [list(e) for e in cig] == c["cigar"], c


def test_cigar_consumes_both_sequences(built, sw_golden):
    """Size-independent property: M+I+S lengths add up to the alternate; with INDEL strategy M+D add up to the reference."""
    for c in sw_golden:
        q = sum(n for n, s in c["cigar"] if s in (0, 1, 4))
        assert q == len(c["alt"]), c
        if c["strategy"] == oracle.SW_INDEL:
            assert sum(n for n, s in c["cigar"] if s in (0, 2)) == len(c["ref"]), c
        assert all(n > 0 for n, _ in c["cigar"])
        assert all(c["cigar"][k][1] != c["cigar"][k + 1][1] for k in range(len(c["cigar"]) - 1))   # runs are merged


def test_port_equals_reference_live(built):
    ref = oracle.sw_reference()
    if ref is None:
        pytest.skip("reference Smith-Waterman not built here")
    port = oracle.sw_port()
    pairs = sw.haplotype_pairs(7, 120, ref_len=(1, 260), per_ref=3)
    for r, a in pairs:
        for st in range(4):
            assert port.align(r, a, st) == ref.align(r, a, st), (r, a, st)
            rc, off, cig = ref.align_falcon(r, a, st, 1)          # Falcon's own implementation agrees too
            assert rc != 0 or (off, cig) == port.align(r, a, st)


# opening at least as expensive as extending (else two touching gaps merge into one element) and far from the -10^8 clamp
RESCORE_WEIGHTS = [(200, -150, -260, -11), (3, -1, -4, -3), (25, -50, -110, -6), (10, -15, -30, -5)]


@pytest.mark.parametrize("strategy", [oracle.SW_SOFTCLIP, oracle.SW_INDEL, oracle.SW_LEADING_INDEL])
def test_port_score_is_the_score_of_its_alignment(built, strategy):
    """For SOFTCLIP, INDEL and LEADING_INDEL the reported score is the score of the returned alignment, recomputed from the
    sequences, weights, offset and CIGAR.  (INDEL starts its traceback at the corner, not at the end cell of the search.)"""
    port = oracle.sw_port()
    pairs = sw.haplotype_pairs(11, 60, ref_len=(20, 160), per_ref=6, sub=0.05, indel=0.04)
    pairs += [(b"A" * 60, b"A" * 37), (b"AC" * 40, b"AC" * 31 + b"A"), (b"ACG" * 30, b"ACG" * 12 + b"T" + b"ACG" * 10),
              (b"C" * 9, b"G" * 9), (b"ACGT" * 25, b"TGCA" * 25), (b"A" * 200 + b"C" * 50, b"C" * 50 + b"A" * 200),
              (b"ACGTTGCA" * 4, b"TTGCA"), (b"G", b"GATTACA"), (b"GATTACA", b"T")]
    for w in RESCORE_WEIGHTS:
        for r, a in pairs:
            off, cig, score = port.align_scored(r, a, strategy, w)
            assert oracle.sw_rescore(r, a, w, off, cig) == score, (w, r, a, sw.cigar_string(cig), off, score)


def test_library_exports_the_sw_abi(built):
    import re
    from acc_genomics_b200 import engine
    hdr = open(os.path.join(ROOT, "include", "smithwaterman_cuda.h")).read()
    declared = set(re.findall(r"\b(sw_[a-z_]+)\s*\(", hdr))
    assert declared == set(sw.SW_EXPORTS)
    L = engine.load_library()
    for name in declared:
        assert hasattr(L, name), name
    # no GPU here -> creation must fail loudly, never fall back
    import ctypes as C
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(sw.SwError):
            sw.SmithWaterman(0)
