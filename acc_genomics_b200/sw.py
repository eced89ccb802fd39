"""ctypes binding of the Smith-Waterman library (include/smithwaterman_cuda.h): the aligner with backtrack and BWA-MEM's
seed extension, with seeded generators of haplotype-to-reference pairs and of extension jobs.  No fallback: a missing
library or GPU raises."""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from .engine import load_library

SW_OK = 0
SOFTCLIP, INDEL, LEADING_INDEL, IGNORE = 0, 1, 2, 3
DEFAULT_WEIGHTS = (200, -150, -260, -11)      # W_MATCH, W_MISMATCH, W_OPEN, W_EXTEND (htc-sw/host/common.h:15-18)
SW_EXPORTS = ["sw_create", "sw_destroy", "sw_last_error", "sw_align_batch", "sw_extend_batch", "sw_get_stats"]
EXTEND_FIELDS = ("score", "qle", "tle", "gtle", "gscore", "max_off")


def bwa_matrix(a: int = 1, b: int = 4, n: int = 1) -> np.ndarray:
    """bwa's 5 x 5 scoring matrix over A, C, G, T, N = 0..4: a on the diagonal, -b off it, -n against N (bwa_fill_scmat)."""
    mat = np.full((5, 5), -b, np.int8)
    np.fill_diagonal(mat, a)
    mat[4, :] = -n; mat[:, 4] = -n
    return mat.reshape(-1)


BWA_DEFAULTS = dict(m=5, mat=bwa_matrix(), o_del=6, e_del=1, o_ins=6, e_ins=1, zdrop=100)   # bwa mem's defaults
_OPS = {0: "M", 1: "I", 2: "D", 4: "S"}


class SwStats(C.Structure):
    _fields_ = [("pairs", C.c_uint64), ("cells", C.c_uint64), ("bytes_backtrack", C.c_uint64), ("kernel_launches", C.c_uint32),
                ("chunks", C.c_uint32), ("ms_kernel", C.c_float), ("ms_total", C.c_float)]


class SwError(RuntimeError):
    pass


def _lib():
    L = load_library()
    if not getattr(L, "_sw_ready", False):
        vp, u32 = C.c_void_p, C.c_uint32
        L.sw_create.argtypes = [C.c_int, C.POINTER(vp)]; L.sw_create.restype = C.c_int
        L.sw_destroy.argtypes = [vp]; L.sw_destroy.restype = None
        L.sw_last_error.argtypes = [vp]; L.sw_last_error.restype = C.c_char_p
        L.sw_align_batch.argtypes = [vp, u32, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u32, vp, vp, vp, vp]
        L.sw_align_batch.restype = C.c_int
        L.sw_extend_batch.argtypes = [vp, u32, vp, vp, vp, C.c_int, vp] + [C.c_int] * 5 + [vp]
        L.sw_extend_batch.restype = C.c_int
        L.sw_get_stats.argtypes = [vp, C.POINTER(SwStats)]; L.sw_get_stats.restype = C.c_int
        L._sw_ready = True
    return L


def cigar_string(elems) -> str:
    return "".join(f"{n}{_OPS.get(s, '?')}" for n, s in elems)


class SmithWaterman:
    """One GPU context (sw_ctx).  align(pairs) -> list of (alignment_offset, [(length, state), ...], score)."""

    def __init__(self, device: int = -1):
        self.lib = _lib()
        h = C.c_void_p()
        rc = self.lib.sw_create(device, C.byref(h))
        if rc != SW_OK:
            raise SwError(self.lib.sw_last_error(None).decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.sw_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def align(self, pairs: Sequence[tuple[bytes, bytes]], strategy: int = SOFTCLIP, weights=DEFAULT_WEIGHTS, cigar_cap: int = 64):
        n = len(pairs)
        # references are stored once each (the common case is one reference against many alternates)
        ref_pos, blob1, s1, l1 = {}, bytearray(), np.empty(n, np.uint32), np.empty(n, np.uint32)
        blob2, s2, l2 = bytearray(), np.empty(n, np.uint32), np.empty(n, np.uint32)
        for k, (r, a) in enumerate(pairs):
            if r not in ref_pos:
                ref_pos[r] = len(blob1); blob1 += r
            s1[k], l1[k] = ref_pos[r], len(r)
            s2[k], l2[k] = len(blob2), len(a); blob2 += a
        b1 = np.frombuffer(bytes(blob1) or b"\0", dtype=np.uint8); b2 = np.frombuffer(bytes(blob2) or b"\0", dtype=np.uint8)
        while True:
            cig = np.empty((max(n, 1), cigar_cap, 2), dtype=np.int32)
            ne = np.empty(max(n, 1), np.int32); off = np.empty(max(n, 1), np.int32); sc = np.empty(max(n, 1), np.int32)
            rc = self.lib.sw_align_batch(self.h, n, b1.ctypes.data, s1.ctypes.data, l1.ctypes.data, b2.ctypes.data, s2.ctypes.data,
                                         l2.ctypes.data, *weights, strategy, cigar_cap, cig.ctypes.data, ne.ctypes.data,
                                         off.ctypes.data, sc.ctypes.data)
            if rc != SW_OK:
                raise SwError(self.lib.sw_last_error(self.h).decode())
            if n == 0 or ne[:n].max() <= cigar_cap:
                break
            cigar_cap = int(ne[:n].max())             # a CIGAR did not fit: once more with room for the longest
        return [(int(off[k]), [(int(cig[k, e, 0]), int(cig[k, e, 1])) for e in range(ne[k])], int(sc[k])) for k in range(n)]

    def extend(self, jobs: Sequence[tuple[bytes, bytes, int, int, int]], mat, m: int, o_del: int, e_del: int, o_ins: int,
               e_ins: int, zdrop: int) -> np.ndarray:
        """BWA-MEM seed extension (ksw_extend2).  jobs: (query, target, h0, w, end_bonus), sequences as bytes < m (a left
        extension passes both reversed).  Returns an (n, 6) int32 array of EXTEND_FIELDS, one row per job."""
        n = len(jobs)
        ql = np.fromiter((len(j[0]) for j in jobs), np.int64, n); tl = np.fromiter((len(j[1]) for j in jobs), np.int64, n)
        desc = np.zeros((n, 7), np.int64)
        desc[:, 0] = np.cumsum(ql) - ql; desc[:, 1] = ql; desc[:, 2] = np.cumsum(tl) - tl; desc[:, 3] = tl
        if n:
            desc[:, 4:] = np.array([j[2:5] for j in jobs], np.int64)
        desc = desc.astype(np.uint32)                 # sw_extend_job_t: four uint32, three int32 (two's complement)
        qb = np.frombuffer(b"".join(j[0] for j in jobs) or b"\0", np.uint8)
        tb = np.frombuffer(b"".join(j[1] for j in jobs) or b"\0", np.uint8)
        mt = np.ascontiguousarray(np.asarray(mat, dtype=np.int8).reshape(-1))
        if mt.size < m * m:
            raise ValueError(f"the matrix has {mt.size} entries, m = {m} needs {m * m}")
        out = np.zeros((max(n, 1), 6), np.int32)
        rc = self.lib.sw_extend_batch(self.h, n, qb.ctypes.data, tb.ctypes.data, desc.ctypes.data, m, mt.ctypes.data,
                                      o_del, e_del, o_ins, e_ins, zdrop, out.ctypes.data)
        if rc != SW_OK:
            raise SwError(self.lib.sw_last_error(self.h).decode())
        return out[:n]

    def stats(self) -> dict:
        s = SwStats()
        self.lib.sw_get_stats(self.h, C.byref(s))
        return {f: getattr(s, f) for f, _ in s._fields_}


_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def haplotype_pairs(seed: int, n_pairs: int, ref_len: int | tuple[int, int] = (250, 500), per_ref: int = 16,
                    sub: float = 0.03, indel: float = 0.01, trim: float = 0.5):
    """(reference, alternate) pairs like GATK's haplotype-to-reference alignment: `per_ref` alternates per reference
    window, each the window with substitutions, short indels and sometimes trimmed ends (overhangs)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    while len(out) < n_pairs:
        L = int(rng.integers(ref_len[0], ref_len[1] + 1)) if isinstance(ref_len, tuple) else int(ref_len)
        ref = _ACGT[rng.integers(0, 4, L)]
        for _ in range(min(per_ref, n_pairs - len(out))):
            alt, k = [], 0
            while k < L:
                u = rng.random()
                if u < sub:
                    alt.append(int(_ACGT[rng.integers(0, 4)])); k += 1
                elif u < sub + indel:
                    alt.extend(_ACGT[rng.integers(0, 4, int(rng.integers(1, 12)))].tolist())
                elif u < sub + 2 * indel:
                    k += int(rng.integers(1, 12))
                else:
                    alt.append(int(ref[k])); k += 1
            a = np.array(alt if alt else [int(ref[0])], dtype=np.uint8)
            lo = int(rng.integers(0, 9)) if rng.random() < trim else 0
            hi = len(a) - (int(rng.integers(0, 9)) if rng.random() < trim else 0)
            a = a[lo:max(hi, lo + 1)]
            if len(a) == 0:
                a = ref[:1]
            out.append((ref.tobytes(), a.tobytes()))
    return out


def extension_jobs(seed: int, n: int, read_len: int = 150, w: int = 100, end_bonus: int = 5, sub: float = 0.02,
                   indel: float = 0.002, ref_len: int = 1 << 20, match: int = 1):
    """n BWA-MEM-like seed-extension jobs (query, target, h0, w, end_bonus), bases as 0..3.  Reads are taken from a
    random reference with substitutions and short indels; each gets a seed of 19..50 bases, and emits the reversed left
    extension (query = read before the seed, target = the reference before the seed's start) and the right one.  Each
    target is the matching reference stretch plus up to w extra bases, as bwa's mem_chain2aln bounds it; h0 is the
    seed's score (its length times `match`)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ref = rng.integers(0, 4, ref_len, dtype=np.uint8)
    out = []
    while len(out) < n:
        nr = max(64, (n - len(out)) // 2 + 1)
        # per read base: substitution, insertion (no reference base consumed) or a deletion of 1..5 bases before it
        u = rng.random((nr, read_len))
        ins = u < indel
        dele = (u >= indel) & (u < 2 * indel)
        subs = (u >= 2 * indel) & (u < 2 * indel + sub)
        adv = np.where(ins, 0, 1) + np.where(dele, rng.integers(1, 6, (nr, read_len)), 0)
        pos0 = rng.integers(2 * w + 64, ref_len - 3 * read_len - 2 * w - 64, nr)
        ridx = pos0[:, None] + np.cumsum(adv, axis=1) - adv[:, :1]       # reference position of each read base
        reads = ref[ridx]
        reads = np.where(subs, (reads + rng.integers(1, 4, (nr, read_len))) % 4, reads)
        reads = np.where(ins, rng.integers(0, 4, (nr, read_len)), reads).astype(np.uint8)
        slen = rng.integers(19, min(50, read_len) + 1, nr)
        qbeg = rng.integers(0, read_len - slen + 1)
        extra = rng.integers(0, w + 1, (nr, 2))
        for r in range(nr):
            qb, qe = int(qbeg[r]), int(qbeg[r] + slen[r])
            h0 = int(slen[r]) * match
            rb, re_ = int(ridx[r, qb]), int(ridx[r, qe - 1]) + 1
            if qb > 0 and len(out) < n:                        # left: both reversed
                t0 = rb - qb - int(extra[r, 0])
                out.append((reads[r, :qb][::-1].tobytes(), ref[t0:rb][::-1].tobytes(), h0, w, end_bonus))
            if qe < read_len and len(out) < n:
                t1 = re_ + (read_len - qe) + int(extra[r, 1])
                out.append((reads[r, qe:].tobytes(), ref[re_:t1].tobytes(), h0, w, end_bonus))
    return out
