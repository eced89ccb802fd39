"""ctypes binding of libpairhmm_b200.so (include/pairhmm_cuda.h) -- the same C ABI the C++ host layer
(pairhmm/client, pairhmm/task, pairhmm/host) links against.  Used by the tests and by bench.py.

There is no fallback of any kind here: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

import numpy as np

from .batch import Batch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PAIRHMM_B200_LIB") or os.path.join(_HERE, "libpairhmm_b200.so")   # override: tuning builds only

PMM_OK, PMM_ERR_INVALID, PMM_ERR_CUDA, PMM_ERR_NO_DEVICE, PMM_ERR_STATE = 0, 1, 2, 3, 4

EXPORTS = [
    "pmm_create", "pmm_destroy", "pmm_last_error", "pmm_device_count", "pmm_set_option",
    "pmm_forward_raw_serialized", "pmm_forward_log10", "pmm_forward_log10_serialized", "pmm_forward_log10_testcases",
    "pmm_stage_flat", "pmm_stage_serialized", "pmm_fetch_fallback", "pmm_launch", "pmm_join", "pmm_sync", "pmm_fetch_raw", "pmm_fetch_log10", "pmm_fetch_fallback_mask",
    "pmm_get_stats", "pmm_measure_fp32_peak", "pmm_measure_fp64_peak", "pmm_plan_flat", "pmm_host_table", "pmm_host_finish_log10",
    "pmm_pool_create", "pmm_pool_destroy", "pmm_pool_last_error", "pmm_pool_num_devices", "pmm_pool_submit_flat",
    "pmm_pool_wait", "pmm_pool_device_load", "pmm_pool_trace", "pmm_pool_get_trace", "pmm_get_timeline",
]


class PmmRegion(C.Structure):
    _fields_ = [("read_first", C.c_uint32), ("num_read", C.c_uint32), ("hap_first", C.c_uint32), ("num_hap", C.c_uint32)]


class PmmStats(C.Structure):
    _fields_ = [("pairs", C.c_uint64), ("cells", C.c_uint64), ("fallback_pairs", C.c_uint64), ("flush_pairs", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("kernel_launches", C.c_uint32),
                ("f32_tasks", C.c_uint32), ("ms_stage", C.c_float), ("ms_f32", C.c_float), ("ms_fallback", C.c_float),
                ("ms_fetch", C.c_float), ("recheck_pairs", C.c_uint64)]


class PmmTimeline(C.Structure):
    _fields_ = [("ref_host_s", C.c_double), ("kernels_start_s", C.c_double), ("f32_end_s", C.c_double), ("kernels_end_s", C.c_double)]


class PmmPoolTrace(C.Structure):
    _fields_ = [("device", C.c_int32), ("context", C.c_int32), ("regions", C.c_uint32),
                ("cells", C.c_uint64), ("pairs", C.c_uint64), ("t_take", C.c_double), ("t_staged", C.c_double),
                ("t_launched", C.c_double), ("t_fetched", C.c_double), ("d_start", C.c_double), ("d_f32_end", C.c_double),
                ("d_end", C.c_double)]


class PmmTaskInfo(C.Structure):
    _fields_ = [("read", C.c_uint32 * 4), ("out_base", C.c_uint32 * 4), ("hap_first", C.c_uint32), ("num_hap", C.c_uint32),
                ("num_read", C.c_uint32), ("rows_per_lane", C.c_uint32), ("lanes_per_read", C.c_uint32), ("striped", C.c_uint32)]


class PmmRead(C.Structure):
    _fields_ = [("len", C.c_int), ("_b", C.c_char_p), ("_q", C.c_char_p), ("_i", C.c_char_p), ("_d", C.c_char_p),
                ("_c", C.c_char_p)]


class PmmHap(C.Structure):
    _fields_ = [("len", C.c_int), ("_b", C.c_char_p)]


class PmmTestcase(C.Structure):      # same field order as `testcase`, /root/reference/pairhmm/xlnx/host/host_type.h:69-73
    _fields_ = [("rslen", C.c_int), ("haplen", C.c_int), ("q", C.c_char_p), ("i", C.c_char_p), ("d", C.c_char_p),
                ("c", C.c_char_p), ("hap", C.c_char_p), ("rs", C.c_char_p)]


class PmmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"pairhmm_cuda error {code}: {msg}")
        self.code = code


_lib = None


def load_library() -> C.CDLL:
    """Load the engine; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} is missing: build it with __graft_entry__.build(); "
                                    "there is no CPU fallback for the PairHMM engine")
        L = C.CDLL(LIB_PATH)
        vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
        L.pmm_create.argtypes = [C.c_int, C.POINTER(vp)]; L.pmm_create.restype = C.c_int
        L.pmm_destroy.argtypes = [vp]; L.pmm_destroy.restype = None
        L.pmm_last_error.argtypes = [vp]; L.pmm_last_error.restype = C.c_char_p
        L.pmm_device_count.argtypes = []; L.pmm_device_count.restype = C.c_int
        L.pmm_set_option.argtypes = [vp, C.c_char_p, C.c_char_p]; L.pmm_set_option.restype = C.c_int
        L.pmm_forward_raw_serialized.argtypes = [vp, vp, u64, vp, u64, vp, u64, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.pmm_forward_log10_serialized.argtypes = [vp, vp, u64, vp, u64, vp, u64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(u64)]
        L.pmm_forward_log10.argtypes = [vp, C.POINTER(PmmRead), C.c_int, C.POINTER(PmmHap), C.c_int, vp, C.POINTER(u64)]
        L.pmm_forward_log10_testcases.argtypes = [vp, C.POINTER(PmmTestcase), u64, vp, C.POINTER(u64)]
        L.pmm_stage_flat.argtypes = [vp, u32, vp, vp, vp, vp, vp, vp, u32, vp, vp, u32, vp]
        L.pmm_stage_serialized.argtypes = [vp, vp, u64, vp, u64, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.pmm_fetch_fallback.argtypes = [vp, vp, vp, u64, C.POINTER(u64)]
        L.pmm_launch.argtypes = [vp]; L.pmm_sync.argtypes = [vp]; L.pmm_join.argtypes = [vp]
        L.pmm_fetch_raw.argtypes = [vp, vp, u64]
        L.pmm_fetch_log10.argtypes = [vp, vp, u64, C.POINTER(u64)]
        L.pmm_fetch_fallback_mask.argtypes = [vp, vp, u64]
        L.pmm_get_stats.argtypes = [vp, C.POINTER(PmmStats)]
        L.pmm_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.pmm_measure_fp64_peak.argtypes = [vp, C.POINTER(C.c_double)]
        L.pmm_plan_flat.argtypes = [u32, vp, u32, vp, u32, vp, C.c_int, C.c_int, vp, u64, C.POINTER(u64)]
        L.pmm_host_table.argtypes = [C.c_int, vp, u64]
        L.pmm_host_finish_log10.argtypes = [vp, u64, vp, vp, u64, vp]
        L.pmm_pool_create.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp)]
        L.pmm_pool_destroy.argtypes = [vp]; L.pmm_pool_destroy.restype = None
        L.pmm_pool_last_error.argtypes = [vp]; L.pmm_pool_last_error.restype = C.c_char_p
        L.pmm_pool_num_devices.argtypes = [vp]
        L.pmm_pool_submit_flat.argtypes = [vp, u32, vp, vp, vp, vp, vp, vp, u32, vp, vp, u32, vp, vp, u64, C.POINTER(u64)]
        L.pmm_pool_wait.argtypes = [vp, u64, C.POINTER(u64), C.POINTER(C.c_int)]
        L.pmm_pool_device_load.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(u64), C.POINTER(u64)]
        L.pmm_pool_trace.argtypes = [vp, C.c_int]
        L.pmm_pool_get_trace.argtypes = [vp, vp, u64, C.POINTER(u64)]
        L.pmm_get_timeline.argtypes = [vp, C.POINTER(PmmTimeline)]
        for n in EXPORTS:
            if n not in ("pmm_destroy", "pmm_last_error", "pmm_pool_destroy", "pmm_pool_last_error"):
                getattr(L, n).restype = C.c_int
        _lib = L
    return _lib


def concat_regions(batches: Sequence[Batch]):
    """Flatten a list of regions into the multi-region layout of pmm_stage_flat."""
    ro, ho = [np.zeros(1, dtype=np.uint32)], [np.zeros(1, dtype=np.uint32)]
    regs = (PmmRegion * len(batches))()
    nr = nh = 0
    rb = hb = 0
    for k, b in enumerate(batches):
        regs[k] = PmmRegion(nr, b.num_read, nh, b.num_hap)
        ro.append(b.read_off[1:].astype(np.uint32) + np.uint32(rb)); ho.append(b.hap_off[1:].astype(np.uint32) + np.uint32(hb))
        nr += b.num_read; nh += b.num_hap; rb += int(b.read_off[-1]); hb += int(b.hap_off[-1])

    def cat(name):
        return np.ascontiguousarray(np.concatenate([getattr(b, name) for b in batches]), dtype=np.uint8)
    return dict(num_read=nr, read_off=np.ascontiguousarray(np.concatenate(ro)), rs=cat("rs"), q=cat("q"), i=cat("i"),
                d=cat("d"), c=cat("c"), num_hap=nh, hap_off=np.ascontiguousarray(np.concatenate(ho)), hap=cat("hap"),
                regions=regs, num_region=len(batches), pairs=sum(b.num_pairs for b in batches))


def host_table(which: int) -> np.ndarray:
    """Tables the engine uploads (host libm); see pmm_host_table in include/pairhmm_cuda.h.  No GPU needed."""
    L = load_library()
    dt, n = {0: (np.float32, 128), 1: (np.float32, 8256), 2: (np.float64, 128), 3: (np.float64, 8256),
             4: (np.float32, 1), 5: (np.float64, 1)}[which]
    out = np.zeros(n, dtype=dt)
    rc = L.pmm_host_table(which, out.ctypes.data, out.nbytes)
    if rc != PMM_OK:
        raise PmmError(rc, "pmm_host_table")
    return out


def plan(batches: Sequence[Batch] | Batch, sm_count: int = 148, tasks_per_warp: int = 16):
    """Host-only: the warp-tasks pmm_stage_flat would build.  Returns a list of dicts.  No GPU needed."""
    if isinstance(batches, Batch):
        batches = [batches]
    L = load_library()
    j = concat_regions(batches)
    n = C.c_uint64()
    args = (j["num_read"], j["read_off"].ctypes.data, j["num_hap"], j["hap_off"].ctypes.data, j["num_region"],
            C.cast(j["regions"], C.c_void_p), sm_count, tasks_per_warp)
    rc = L.pmm_plan_flat(*args, None, 0, C.byref(n))
    if rc != PMM_OK:
        raise PmmError(rc, L.pmm_last_error(None).decode())
    buf = (PmmTaskInfo * n.value)()
    rc = L.pmm_plan_flat(*args, C.cast(buf, C.c_void_p), n.value, C.byref(n))
    if rc != PMM_OK:
        raise PmmError(rc, L.pmm_last_error(None).decode())
    return [dict(read=list(t.read)[: t.num_read], out_base=list(t.out_base)[: t.num_read], hap_first=t.hap_first,
                 num_hap=t.num_hap, K=t.rows_per_lane, W=t.lanes_per_read, striped=bool(t.striped)) for t in buf]


class PairHMMEngine:
    """One GPU context (pmm_ctx).  Not thread-safe; one engine per host thread."""

    def __init__(self, device: int = -1):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.pmm_create(device, C.byref(h))
        if rc != PMM_OK:
            raise PmmError(rc, self.lib.pmm_last_error(None).decode())
        self.h = h
        self._job = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.pmm_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != PMM_OK:
            raise PmmError(rc, self.lib.pmm_last_error(self.h).decode())

    def set_option(self, key: str, value) -> None:
        self._ck(self.lib.pmm_set_option(self.h, key.encode(), str(value).encode()))

    # ---- staged path -----------------------------------------------------------------------------------
    def stage(self, batches: Sequence[Batch] | Batch):
        if isinstance(batches, Batch):
            batches = [batches]
        j = concat_regions(batches)
        self._job = j        # keeps the arrays alive; the library copies during the call anyway
        self._ck(self.lib.pmm_stage_flat(self.h, j["num_read"], j["read_off"].ctypes.data, j["rs"].ctypes.data,
                                         j["q"].ctypes.data, j["i"].ctypes.data, j["d"].ctypes.data, j["c"].ctypes.data,
                                         j["num_hap"], j["hap_off"].ctypes.data, j["hap"].ctypes.data,
                                         j["num_region"], C.cast(j["regions"], C.c_void_p)))
        return j

    def restage(self):
        """Repeat the last stage() from the already flattened host arrays (the e2e timing loop of bench.py)."""
        j = self._job
        self._ck(self.lib.pmm_stage_flat(self.h, j["num_read"], j["read_off"].ctypes.data, j["rs"].ctypes.data,
                                         j["q"].ctypes.data, j["i"].ctypes.data, j["d"].ctypes.data, j["c"].ctypes.data,
                                         j["num_hap"], j["hap_off"].ctypes.data, j["hap"].ctypes.data,
                                         j["num_region"], C.cast(j["regions"], C.c_void_p)))

    def launch(self):
        self._ck(self.lib.pmm_launch(self.h))

    def sync(self):
        self._ck(self.lib.pmm_sync(self.h))

    def join(self):
        """The launch stream waits for the last launch's double re-run (no host wait)."""
        self._ck(self.lib.pmm_join(self.h))

    def fetch_raw(self) -> np.ndarray:
        out = np.empty(self._job["pairs"], dtype=np.float32)
        self._ck(self.lib.pmm_fetch_raw(self.h, out.ctypes.data, out.size))
        return out

    def fetch_log10(self, out: np.ndarray | None = None):
        if out is None:
            out = np.empty(self._job["pairs"], dtype=np.float64)
        nfb = C.c_uint64()
        self._ck(self.lib.pmm_fetch_log10(self.h, out.ctypes.data, out.size, C.byref(nfb)))
        return out, int(nfb.value)

    def fetch_fallback_mask(self) -> np.ndarray:
        m = np.empty(self._job["pairs"], dtype=np.uint8)
        self._ck(self.lib.pmm_fetch_fallback_mask(self.h, m.ctypes.data, m.size))
        return m.astype(bool)

    def stats(self) -> dict:
        s = PmmStats()
        self._ck(self.lib.pmm_get_stats(self.h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in s._fields_}

    def measure_fp32_peak(self):
        r, mhz = C.c_double(), C.c_double()
        self._ck(self.lib.pmm_measure_fp32_peak(self.h, C.byref(r), C.byref(mhz)))
        return r.value, mhz.value

    def measure_fp64_peak(self) -> float:
        r = C.c_double()
        self._ck(self.lib.pmm_measure_fp64_peak(self.h, C.byref(r)))
        return r.value

    # ---- one-shot paths ---------------------------------------------------------------------------------
    def forward(self, b: Batch):
        """raw [R,H] float32, log10 [R,H] float64, fallback mask [R,H] -- one region through the staged path."""
        self.stage([b]); self.launch()
        raw = self.fetch_raw().reshape(b.num_read, b.num_hap)
        out, _ = self.fetch_log10()
        mask = self.fetch_fallback_mask().reshape(b.num_read, b.num_hap)
        return raw, out.reshape(b.num_read, b.num_hap), mask

    def forward_raw_serialized(self, reads_ser: bytes, haps_ser: bytes, capacity: int) -> np.ndarray:
        out = np.empty(capacity, dtype=np.float32)
        nr, nh = C.c_int(), C.c_int()
        self._ck(self.lib.pmm_forward_raw_serialized(self.h, reads_ser, len(reads_ser), haps_ser, len(haps_ser),
                                                     out.ctypes.data, capacity, C.byref(nr), C.byref(nh)))
        return out[: nr.value * nh.value].reshape(nr.value, nh.value)

    def forward_log10_serialized(self, reads_ser: bytes, haps_ser: bytes, capacity: int):
        out = np.empty(capacity, dtype=np.float64)
        nr, nh, nfb = C.c_int(), C.c_int(), C.c_uint64()
        self._ck(self.lib.pmm_forward_log10_serialized(self.h, reads_ser, len(reads_ser), haps_ser, len(haps_ser),
                                                       out.ctypes.data, capacity, C.byref(nr), C.byref(nh), C.byref(nfb)))
        return out[: nr.value * nh.value].reshape(nr.value, nh.value), int(nfb.value)

    def forward_log10_structs(self, b: Batch):
        """Through pmm_forward_log10 with read_t / hap_t arrays (the client-side entry)."""
        keep = []
        reads = (PmmRead * b.num_read)()
        for k in range(b.num_read):
            bs = [bytes(x) for x in b.read(k)]
            keep.append(bs)
            reads[k] = PmmRead(len(bs[0]), *bs)
        haps = (PmmHap * b.num_hap)()
        for k in range(b.num_hap):
            hb = bytes(b.haplotype(k)); keep.append(hb)
            haps[k] = PmmHap(len(hb), hb)
        out = np.empty(b.num_pairs, dtype=np.float64)
        nfb = C.c_uint64()
        self._ck(self.lib.pmm_forward_log10(self.h, reads, b.num_read, haps, b.num_hap, out.ctypes.data, C.byref(nfb)))
        return out.reshape(b.num_read, b.num_hap), int(nfb.value)


    def forward_log10_testcases(self, pairs):
        """Through pmm_forward_log10_testcases: `pairs` is a list of (read, hap) with read = the 5-tuple of bytes objects
        (bases, q, i, d, c) and hap = a bytes object; pairs that name the same objects share pointers, like GKL's JNI."""
        tc = (PmmTestcase * len(pairs))()
        for k, (r, h) in enumerate(pairs):
            tc[k] = PmmTestcase(len(r[0]), len(h), r[1], r[2], r[3], r[4], h, r[0])
        out = np.empty(len(pairs), dtype=np.float64)
        nfb = C.c_uint64()
        self._ck(self.lib.pmm_forward_log10_testcases(self.h, tc, len(pairs), out.ctypes.data, C.byref(nfb)))
        return out, int(nfb.value)


class PairHMMPool:
    """The multi-GPU work queue (pmm_pool_*): regions in, log10 likelihoods out, whole regions per GPU, no collective."""

    def __init__(self, devices: Sequence[int] | None = None, contexts_per_device: int = 2):
        self.lib = load_library()
        h = C.c_void_p()
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.pmm_pool_create(C.cast(arr, C.c_void_p), len(devices), contexts_per_device, C.byref(h))
        else:
            rc = self.lib.pmm_pool_create(None, 0, contexts_per_device, C.byref(h))
        if rc != PMM_OK:
            raise PmmError(rc, self.lib.pmm_pool_last_error(None).decode())
        self.h = h
        self._live = {}

    @property
    def num_devices(self) -> int:
        return self.lib.pmm_pool_num_devices(self.h)

    def submit(self, batches: Sequence[Batch] | Batch, out: np.ndarray | None = None, job: dict | None = None) -> int:
        """Queue one job (a list of regions).  Returns a ticket; the result array is returned by wait()."""
        if job is None:
            if isinstance(batches, Batch):
                batches = [batches]
            job = concat_regions(batches)
        if out is None:
            out = np.empty(job["pairs"], dtype=np.float64)
        t = C.c_uint64()
        rc = self.lib.pmm_pool_submit_flat(self.h, job["num_read"], job["read_off"].ctypes.data, job["rs"].ctypes.data,
                                           job["q"].ctypes.data, job["i"].ctypes.data, job["d"].ctypes.data,
                                           job["c"].ctypes.data, job["num_hap"], job["hap_off"].ctypes.data,
                                           job["hap"].ctypes.data, job["num_region"], C.cast(job["regions"], C.c_void_p),
                                           out.ctypes.data, out.size, C.byref(t))
        if rc != PMM_OK:
            raise PmmError(rc, self.lib.pmm_pool_last_error(self.h).decode())
        self._live[t.value] = (job, out)          # the library borrows these until wait()
        return t.value

    def wait(self, ticket: int):
        """-> (log10 likelihoods [pairs], number of fallback pairs, device index)."""
        nfb, dev = C.c_uint64(), C.c_int()
        rc = self.lib.pmm_pool_wait(self.h, ticket, C.byref(nfb), C.byref(dev))
        _, out = self._live.pop(ticket, (None, None))
        if rc != PMM_OK:
            raise PmmError(rc, self.lib.pmm_pool_last_error(self.h).decode())
        return out, int(nfb.value), int(dev.value)

    def trace(self, on: bool) -> None:
        """Start (and clear) or stop recording one timeline record per GPU job (pmm_pool_trace)."""
        self.lib.pmm_pool_trace(self.h, int(on))

    def get_trace(self) -> list:
        n = C.c_uint64()
        self.lib.pmm_pool_get_trace(self.h, None, 0, C.byref(n))
        buf = (PmmPoolTrace * max(1, n.value))()
        self.lib.pmm_pool_get_trace(self.h, C.cast(buf, C.c_void_p), n.value, C.byref(n))
        return [{f: getattr(buf[k], f) for f, _ in PmmPoolTrace._fields_} for k in range(n.value)]

    def device_load(self):
        res = []
        for s in range(self.num_devices):
            d, j, c = C.c_int(), C.c_uint64(), C.c_uint64()
            self.lib.pmm_pool_device_load(self.h, s, C.byref(d), C.byref(j), C.byref(c))
            res.append(dict(device=d.value, jobs=j.value, cells=c.value))
        return res

    def close(self):
        if getattr(self, "h", None):
            self.lib.pmm_pool_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
