"""Row a14 of SURVEY.md section 8: the wire format pinned to the REFERENCE's own writer.

tests/golden/wire_format_golden.npz holds the bytes the reference's serialize() writes for the cases below (see
tests/golden/make_wire_golden.py).  Checked here, byte for byte: those bytes == the Python writer (acc_genomics_b200/batch.py)
== this repo's serialize() after reading them (pairhmm/interface, through the selftest binary).  Where
oracle/_ref/libhostif_ref.so has been built from the reference's PairHMMHostInterface.cpp (oracle/Makefile; its one
un-vendored include, ksight/tools.h, is a two-macro stub), the reference's serialize() is also run live, for both overload
sets, and it deserialises the Python writer's output and writes it back unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from acc_genomics_b200 import batch as B
from acc_genomics_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "libhostif_ref.so")
SELFTEST = os.path.join(ROOT, "pairhmm", "bin", "selftest")


GOLDEN = os.path.join(ROOT, "tests", "golden", "wire_format_golden.npz")


def load_reference():
    """The reference's writer and reader, or None where oracle/_ref/libhostif_ref.so has not been built."""
    if not os.path.exists(REF):
        return None
    L = C.CDLL(REF)
    vp = C.c_void_p
    L.refif_serialize_reads.restype = C.c_uint64; L.refif_serialize_reads.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp]
    L.refif_serialize_haps.restype = C.c_uint64; L.refif_serialize_haps.argtypes = [vp, C.c_int, vp, vp]
    L.refif_serialize_reads_str.restype = C.c_uint64; L.refif_serialize_reads_str.argtypes = [vp, C.c_uint64, C.c_int, vp, vp, vp, vp, vp, vp]
    L.refif_serialize_haps_str.restype = C.c_uint64; L.refif_serialize_haps_str.argtypes = [vp, C.c_uint64, C.c_int, vp, vp]
    L.refif_reserialize_reads.restype = C.c_uint64; L.refif_reserialize_reads.argtypes = [vp, C.c_uint64, vp, C.c_int, C.POINTER(C.c_int)]
    L.refif_reserialize_haps.restype = C.c_uint64; L.refif_reserialize_haps.argtypes = [vp, C.c_uint64, vp, C.c_int, C.POINTER(C.c_int)]
    return L


@pytest.fixture(scope="module")
def ref(built):
    return load_reference()


@pytest.fixture(scope="module")
def wire_golden():
    g = np.load(GOLDEN)
    return {k: g[k].tobytes() for k in g.files}


def ref_serialize(L, b):
    ro = np.ascontiguousarray(b.read_off, dtype=np.int32); ho = np.ascontiguousarray(b.hap_off, dtype=np.int32)
    tr = [np.ascontiguousarray(x, dtype=np.uint8) for x in (b.rs, b.q, b.i, b.d, b.c)]
    hp = np.ascontiguousarray(b.hap, dtype=np.uint8)
    cap_r = 4 + 4 * b.num_read + 5 * int(ro[-1]) + 64; cap_h = 4 + 4 * b.num_hap + int(ho[-1]) + 64
    out = {}
    for name, fn_r, fn_h in (("ptr", None, None), ("str", None, None)):
        rbuf = np.zeros(cap_r, dtype=np.uint8); hbuf = np.zeros(cap_h, dtype=np.uint8)
        if name == "ptr":
            nr = L.refif_serialize_reads(rbuf.ctypes.data, b.num_read, ro.ctypes.data, *[t.ctypes.data for t in tr])
            nh = L.refif_serialize_haps(hbuf.ctypes.data, b.num_hap, ho.ctypes.data, hp.ctypes.data)
        else:
            nr = L.refif_serialize_reads_str(rbuf.ctypes.data, cap_r, b.num_read, ro.ctypes.data, *[t.ctypes.data for t in tr])
            nh = L.refif_serialize_haps_str(hbuf.ctypes.data, cap_h, b.num_hap, ho.ctypes.data, hp.ctypes.data)
        out[name] = (rbuf[:nr].tobytes(), hbuf[:nh].tobytes())
    return out


def ref_reserialize(L, rs, hs, which):
    ro = np.zeros(len(rs) + 64, dtype=np.uint8); ho = np.zeros(len(hs) + 64, dtype=np.uint8)
    n1, n2 = C.c_int(), C.c_int()
    a = L.refif_reserialize_reads(rs, len(rs), ro.ctypes.data, which, C.byref(n1))
    b = L.refif_reserialize_haps(hs, len(hs), ho.ctypes.data, which, C.byref(n2))
    return ro[:a].tobytes(), ho[:b].tobytes(), n1.value, n2.value


def ours_reserialize(tmp_path, rs, hs):
    (tmp_path / "r.bin").write_bytes(rs); (tmp_path / "h.bin").write_bytes(hs)
    p = subprocess.run([SELFTEST, "reserialize", str(tmp_path / "r.bin"), str(tmp_path / "h.bin"), str(tmp_path / "r.out"),
                        str(tmp_path / "h.out")], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0 and p.stdout.startswith("ok"), p.stdout + p.stderr
    return (tmp_path / "r.out").read_bytes(), (tmp_path / "h.out").read_bytes()


CASES = {
    "cfg1": lambda: synth.config(1)[0],
    "cfg5_ragged_region": lambda: synth.config(5, scale=0.0008)[1],
    "cfg4_slice": lambda: synth.config(4, scale=0.02)[0],
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_reference_writer_equals_ours_and_python(ref, wire_golden, tmp_path, case):
    b = CASES[case]()
    want = (wire_golden[f"{case}/reads"], wire_golden[f"{case}/haps"])
    py = (B.serialize_reads(b), B.serialize_haps(b))
    assert py == want, "the Python writer differs from the reference's serialize() bytes"
    # this repo's C++ reads the reference's bytes and writes them back unchanged (all overloads, inside selftest)
    assert ours_reserialize(tmp_path, *want) == want
    if case == "cfg1":                              # sizes SURVEY.md section 8a quotes for configuration 1
        assert len(want[0]) == 65156 and len(want[1]) == 12932
    if ref is not None:
        got = ref_serialize(ref, b)
        assert got["ptr"] == want, "reference serialize(void*, ...) differs from the stored bytes"
        assert got["str"] == want, "reference serialize() -> std::string differs from the stored bytes"
        # the reference reads our bytes (= the Python writer's, just shown equal to ours) and writes them back unchanged
        for which in (0, 1):
            r2, h2, nr, nh = ref_reserialize(ref, py[0], py[1], which)
            assert (r2, h2) == py and nr == b.num_read and nh == b.num_hap


def test_empty_batch(ref, tmp_path):
    empty = B.Batch(np.zeros(1, np.int32), *[np.zeros(0, np.uint8)] * 5, np.zeros(1, np.int32), np.zeros(0, np.uint8))
    zero = np.int32(0).tobytes()
    assert (B.serialize_reads(empty), B.serialize_haps(empty)) == (zero, zero)
    assert ours_reserialize(tmp_path, zero, zero) == (zero, zero)
    if ref is not None:
        got = ref_serialize(ref, empty)
        assert got["ptr"] == (zero, zero) and got["str"] == (zero, zero)
        for which in (0, 1):
            assert ref_reserialize(ref, zero, zero, which) == (zero, zero, 0, 0)
