"""ctypes front end of oracle/ksw_oracle.c, the CPU restatement of ksw_extend2 of bwa 0.7.17 (BWA-MEM's seed
extension).  TEST INFRASTRUCTURE ONLY, like the rest of this package: the product never imports it.  The library is
oracle/libksw_oracle.so (oracle/ksw.mk)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ("score", "qle", "tle", "gtle", "gscore", "max_off")
_lib = None


def build(quiet: bool = True) -> None:
    subprocess.run(["make", "-C", _HERE, "-f", "ksw.mk"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None, stderr=subprocess.STDOUT if quiet else None)


def _load():
    global _lib
    if _lib is None:
        p = os.path.join(_HERE, "libksw_oracle.so")
        if not os.path.exists(p):
            build()
        L = C.CDLL(p)
        vp, i = C.c_void_p, C.c_int
        L.ksw_oracle_extend.restype = i
        L.ksw_oracle_extend.argtypes = [i, C.c_char_p, i, C.c_char_p, i, vp] + [i] * 8 + [vp, vp]
        L.ksw_oracle_extend_batch.restype = None
        L.ksw_oracle_extend_batch.argtypes = [i, vp, vp, vp, i, vp] + [i] * 5 + [vp, vp]
        _lib = L
    return _lib


def extend(query: bytes, target: bytes, m: int, mat, o_del: int, e_del: int, o_ins: int, e_ins: int, w: int,
           end_bonus: int, zdrop: int, h0: int):
    """One extension: (score, qle, tle, gtle, gscore, max_off, cells)."""
    L = _load()
    mt = np.ascontiguousarray(mat, dtype=np.int8)
    out = np.zeros(6, np.int32); cells = np.zeros(1, np.uint64)
    L.ksw_oracle_extend(len(query), query, len(target), target, m, mt.ctypes.data, o_del, e_del, o_ins, e_ins, w,
                        end_bonus, zdrop, h0, out.ctypes.data, cells.ctypes.data)
    return tuple(int(x) for x in out) + (int(cells[0]),)


def extend_batch(jobs, m: int, mat, o_del: int, e_del: int, o_ins: int, e_ins: int, zdrop: int):
    """jobs: (query, target, h0, w, end_bonus) tuples, run one after another on the calling thread (outside the GIL).
    Returns an (n, 6) int32 array of FIELDS and the (n,) uint64 cell counts."""
    L = _load()
    n = len(jobs)
    ql = np.fromiter((len(j[0]) for j in jobs), np.int64, n); tl = np.fromiter((len(j[1]) for j in jobs), np.int64, n)
    desc = np.zeros((n, 7), np.int64)
    desc[:, 0] = np.cumsum(ql) - ql; desc[:, 1] = ql; desc[:, 2] = np.cumsum(tl) - tl; desc[:, 3] = tl
    if n:
        desc[:, 4:] = np.array([j[2:5] for j in jobs], np.int64).reshape(n, 3)
    desc = desc.astype(np.int32)
    qb = np.frombuffer(b"".join(j[0] for j in jobs) or b"\0", np.uint8)
    tb = np.frombuffer(b"".join(j[1] for j in jobs) or b"\0", np.uint8)
    mt = np.ascontiguousarray(mat, dtype=np.int8)
    out = np.zeros((max(n, 1), 6), np.int32); cells = np.zeros(max(n, 1), np.uint64)
    L.ksw_oracle_extend_batch(n, qb.ctypes.data, tb.ctypes.data, desc.ctypes.data, m, mt.ctypes.data, o_del, e_del,
                              o_ins, e_ins, zdrop, out.ctypes.data, cells.ctypes.data)
    return out[:n], cells[:n]
