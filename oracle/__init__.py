"""ctypes front end of the CPU checkers.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs may import
this package; the product (``acc_genomics_b200``) never does.

Two libraries with the same call surface:
  * ``port``      -- oracle/liboracle.so, our C restatement (oracle/pairhmm_oracle.c)
  * ``reference`` -- oracle/_ref/libpairhmm_ref.so, the reference's own AVX sources compiled with pinned flags
                     (oracle/Makefile); ``reference_fma`` is the same with FMA contraction, timing only.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PAIR_ARGS = [C.c_int, C.c_int] + [C.c_char_p] * 6
_BATCH_ARGS = [C.c_int, C.c_void_p] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]


def build(quiet: bool = True) -> None:
    """Compile liboracle.so and, when /root/reference is present, oracle/_ref (see oracle/Makefile)."""
    subprocess.run(["make", "-C", _HERE], check=True,
                   stdout=subprocess.DEVNULL if quiet else None, stderr=subprocess.STDOUT if quiet else None)


class _Lib:
    def __init__(self, path: str, prefix: str, batch: str):
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        self.kind = prefix
        names = {"f32": "pmm_oracle_f32", "f64": "pmm_oracle_f64"} if prefix == "port" else \
                {"f32": "ref_avxs", "f64": "ref_avxd"}
        self._f32 = getattr(L, names["f32"]); self._f32.restype = C.c_float; self._f32.argtypes = _PAIR_ARGS
        self._f64 = getattr(L, names["f64"]); self._f64.restype = C.c_double; self._f64.argtypes = _PAIR_ARGS
        self._batch = getattr(L, batch); self._batch.restype = None; self._batch.argtypes = _BATCH_ARGS
        pre = "pmm_oracle_" if prefix == "port" else "ref_"
        for nm, ty in (("ph2pr_f32", C.c_float), ("ph2pr_f64", C.c_double), ("m2m_f32", C.c_float), ("m2m_f64", C.c_double)):
            f = getattr(L, pre + nm); f.restype = C.POINTER(ty); f.argtypes = []
        for nm, ty in (("log10_ic_f32", C.c_float), ("log10_ic_f64", C.c_double)):
            f = getattr(L, pre + nm); f.restype = ty; f.argtypes = []
        if prefix != "port":
            for nm, ty in (("ref_baseline_f32", C.c_float), ("ref_baseline_f64", C.c_double)):
                f = getattr(L, nm); f.restype = ty; f.argtypes = _PAIR_ARGS
        self._pre = pre

    # -- tables ------------------------------------------------------------------------------------------
    def table(self, name: str) -> np.ndarray:
        n = 128 if name.startswith("ph2pr") else 8256   # the m2m entries reachable with quals masked to 0..127
        p = getattr(self.lib, self._pre + name)()
        return np.ctypeslib.as_array(p, shape=(n,)).copy()

    def log10_ic(self):
        return getattr(self.lib, self._pre + "log10_ic_f32")(), getattr(self.lib, self._pre + "log10_ic_f64")()

    # -- one pair ----------------------------------------------------------------------------------------
    @staticmethod
    def _pair(rs, q, i, d, c, hap):
        bs = [np.ascontiguousarray(x, dtype=np.uint8).tobytes() for x in (rs, q, i, d, c, hap)]
        return [len(bs[0]), len(bs[5])] + bs

    def f32(self, rs, q, i, d, c, hap) -> np.float32:
        return np.float32(self._f32(*self._pair(rs, q, i, d, c, hap)))

    def f64(self, rs, q, i, d, c, hap) -> np.float64:
        return np.float64(self._f64(*self._pair(rs, q, i, d, c, hap)))

    def baseline_f32(self, rs, q, i, d, c, hap) -> np.float32:
        return np.float32(self.lib.ref_baseline_f32(*self._pair(rs, q, i, d, c, hap)))

    def baseline_f64(self, rs, q, i, d, c, hap) -> np.float64:
        return np.float64(self.lib.ref_baseline_f64(*self._pair(rs, q, i, d, c, hap)))

    # -- whole batch (the contract of FalconPairHMM::computePairhmmAVX) -----------------------------------
    def batch(self, b, float_only: bool = False, threads: int = 1):
        """Returns (raw_f32 [R,H], log10 [R,H] float64 or None, fallback mask [R,H] bool)."""
        n = b.num_pairs
        raw = np.zeros(n, dtype=np.float32)
        out = np.zeros(n, dtype=np.float64)
        fb = np.zeros(n, dtype=np.uint8)
        arrs = [np.ascontiguousarray(x, dtype=np.uint8) for x in (b.rs, b.q, b.i, b.d, b.c, b.hap)]
        ro = np.ascontiguousarray(b.read_off, dtype=np.int32)
        ho = np.ascontiguousarray(b.hap_off, dtype=np.int32)
        self._batch(b.num_read, ro.ctypes.data, *[a.ctypes.data for a in arrs[:5]], b.num_hap, ho.ctypes.data,
                    arrs[5].ctypes.data, raw.ctypes.data, out.ctypes.data, fb.ctypes.data,
                    1 if float_only else 0, int(threads))
        shape = (b.num_read, b.num_hap)
        return raw.reshape(shape), (None if float_only else out.reshape(shape)), fb.reshape(shape).astype(bool)


_cache: dict = {}


def port() -> _Lib:
    if "port" not in _cache:
        p = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(p):
            build()
        _cache["port"] = _Lib(p, "port", "pmm_oracle_batch")
    return _cache["port"]


def reference(fma: bool = False) -> _Lib | None:
    """The reference's own implementation, or None when oracle/_ref has not been built."""
    key = "reference_fma" if fma else "reference"
    if key not in _cache:
        p = os.path.join(_HERE, "_ref", "libpairhmm_ref_fma.so" if fma else "libpairhmm_ref.so")
        if not os.path.exists(p) and os.path.isdir("/root/reference/pairhmm/xlnx/host"):
            build()
        _cache[key] = _Lib(p, key, "ref_batch") if os.path.exists(p) else None
    return _cache[key]


# ---- Smith-Waterman (SURVEY.md section 8f row 4) ------------------------------------------------------------------
SW_SOFTCLIP, SW_INDEL, SW_LEADING_INDEL, SW_IGNORE = 0, 1, 2, 3
SW_WEIGHTS = (200, -150, -260, -11)        # W_MATCH, W_MISMATCH, W_OPEN, W_EXTEND (htc-sw/host/common.h:15-18)
_CIGAR_CAP = 8192                          # the most elements a CIGAR of two 4095-base sequences can have


class _SwLib:
    """align(ref, alt, strategy, weights) -> (offset, [(length, state), ...]); states 0 M, 1 I, 2 D, 4 S."""

    def __init__(self, path: str, kind: str):
        self.kind = kind
        self.lib = C.CDLL(path)
        ip = C.POINTER(C.c_int)
        if kind == "port":
            f = self.lib.sw_oracle_align
            f.restype = C.c_int
            f.argtypes = [C.c_int] * 4 + [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, ip, ip, C.c_int, ip, ip]
        else:
            f = self.lib.ref_sw_gkl
            f.restype = C.c_int
            f.argtypes = [C.c_int] * 4 + [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, ip, ip, C.c_int, ip]
            g = self.lib.ref_sw_falcon
            g.restype = C.c_int
            g.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, ip, ip, C.c_int, ip, ip]
        self._len = (C.c_int * _CIGAR_CAP)()
        self._st = (C.c_int * _CIGAR_CAP)()

    def align(self, ref: bytes, alt: bytes, strategy: int, weights=SW_WEIGHTS):
        n = C.c_int()
        if self.kind != "port" and (len(ref) > 1536 or len(alt) > 1536):
            raise ValueError("the reference's Smith-Waterman has fixed 1536-base buffers (MAX_SEQ_LEN); use sw_port()")
        if self.kind == "port":
            return self.align_scored(ref, alt, strategy, weights)[:2]
        off = self.lib.ref_sw_gkl(*weights, ref, len(ref), alt, len(alt), strategy, self._len, self._st, _CIGAR_CAP, C.byref(n))
        return off, [(self._len[k], self._st[k]) for k in range(n.value)]

    def align_scored(self, ref: bytes, alt: bytes, strategy: int, weights=SW_WEIGHTS):
        """(offset, cigar, score): score is H of the cell the traceback starts from.  The C restatement only: the
        reference's runSWOnePairBT returns no score."""
        if self.kind != "port":
            raise ValueError("only the C restatement reports a score; use sw_port()")
        n, sc = C.c_int(), C.c_int()
        off = self.lib.sw_oracle_align(*weights, ref, len(ref), alt, len(alt), strategy, self._len, self._st, _CIGAR_CAP,
                                       C.byref(n), C.byref(sc))
        return off, [(self._len[k], self._st[k]) for k in range(n.value)], sc.value

    def align_falcon(self, ref: bytes, alt: bytes, strategy: int, option: int = 1):
        """Falcon's own SWPairwiseAlignmentOneBatch (fixed weights); option 1 = scalar baseline, 0 = its SIMD variant."""
        n, rc = C.c_int(), C.c_int()
        off = self.lib.ref_sw_falcon(ref, len(ref), alt, len(alt), strategy, option, self._len, self._st, _CIGAR_CAP,
                                     C.byref(n), C.byref(rc))
        return rc.value, off, [(self._len[k], self._st[k]) for k in range(n.value)]


def sw_rescore(ref: bytes, alt: bytes, weights, offset: int, cigar) -> int:
    """The score of an alignment given by its offset and CIGAR: match / mismatch per M base, open + (L - 1) * extend per
    I or D element of length L, nothing for S."""
    match, mismatch, open_, extend = weights
    i, j, s = offset, 0, 0
    for n, st in cigar:
        if st == 0:
            s += sum(match if ref[i + k] == alt[j + k] else mismatch for k in range(n))
            i += n; j += n
        elif st in (1, 2):
            s += open_ + (n - 1) * extend
            i, j = (i, j + n) if st == 1 else (i + n, j)
        else:
            if st != 4:
                raise ValueError(f"CIGAR state {st}")
            j += n
    if j != len(alt) or i > len(ref):
        raise ValueError("the CIGAR does not fit the sequences")
    return s


def sw_port() -> "_SwLib":
    p = os.path.join(_HERE, "liboracle.so")
    if not os.path.exists(p):
        build()
    return _SwLib(p, "port")


def sw_reference():
    """The reference's own Smith-Waterman (oracle/_ref/libsw_ref.so); None if absent or the CPU lacks AVX2."""
    p = os.path.join(_HERE, "_ref", "libsw_ref.so")
    if not os.path.exists(p):
        if os.path.isdir("/root/reference/htc-sw"):
            build()
        if not os.path.exists(p):
            return None
    try:
        with open("/proc/cpuinfo") as f:
            if "avx2" not in f.read():
                return None
    except OSError:
        pass
    return _SwLib(p, "reference")
