"""TEST INFRASTRUCTURE ONLY -- parity unpinned.

ctypes loader for the C++ CPU oracle (oracle/parasuite_oracle.cpp).  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(REPO, "para-suite_b200"))
from parasuite_b200 import abi  # noqa: E402  (struct layouts only)

SO = os.path.join(HERE, "_build", "libparasuite_oracle.so")
_lib = None


def _stale() -> bool:
    src = os.path.join(HERE, "parasuite_oracle.cpp")
    hdr = os.path.join(REPO, "include", "parasuite_b200.h")
    return (not os.path.exists(SO)) or os.path.getmtime(SO) < max(os.path.getmtime(src), os.path.getmtime(hdr))


def build(force: bool = False) -> str:
    """Build the oracle if it is missing or older than its sources.  Safe when several processes call it at once (the
    ranks of one torchrun job on a fresh box): one builds under a file lock, the others wait and find it up to date; the
    Makefile writes under a temporary name and renames."""
    if not (force or _stale()):
        return SO
    import fcntl
    os.makedirs(os.path.join(HERE, "_build"), exist_ok=True)
    with open(os.path.join(HERE, "_build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or _stale():
                subprocess.check_call(["make", "-B", "-C", HERE], stdout=subprocess.DEVNULL)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return SO


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            build()
        lib = C.CDLL(SO)
        lib.or_profile_acc_len.restype = C.c_size_t
        lib.or_profile_acc_len.argtypes = [C.c_uint32, C.c_uint32]
        lib.or_profile_run.restype = C.c_int
        lib.or_profile_run.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch), C.c_uint32,
                                       C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p,
                                       C.POINTER(abi.ps_fault)]
        lib.or_pileup_run.restype = C.c_void_p
        lib.or_pileup_run.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch),
                                      C.POINTER(abi.ps_pileup_opts)]
        lib.or_pileup_counters.argtypes = [C.c_void_p, C.POINTER(abi.ps_pileup_counters)]
        lib.or_pileup_fault.argtypes = [C.c_void_p, C.POINTER(abi.ps_fault)]
        lib.or_pileup_copy.restype = C.c_int64
        lib.or_pileup_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
        lib.or_pileup_open.restype = C.c_int64
        lib.or_pileup_open.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        lib.or_pileup_free.argtypes = [C.c_void_p]
        lib.or_read_t2c_masks.restype = C.c_int
        lib.or_read_t2c_masks.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch), C.c_void_p]
        lib.or_pileup_head.restype = C.c_int64
        lib.or_pileup_head.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        lib.or_pileup_boundary_cov.restype = C.c_int64
        lib.or_pileup_boundary_cov.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_void_p, C.c_uint64]
        _lib = lib
    return _lib


def _i32(a: np.ndarray) -> np.ndarray:
    return (a.astype(np.int64) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)


def split_acc(acc: np.ndarray, max_len: int, infer_q: bool = False) -> dict:
    """Slice the int64 accumulator vector (layout in include/parasuite_b200.h) and apply Java int wrap."""
    m = max_len
    o = 0
    conv = acc[o:o + 16 * m]; o += 16 * m
    qsum = acc[o:o + 16]; o += 16
    qcnt = acc[o:o + 16]; o += 16
    ins = acc[o:o + m]; o += m
    dele = acc[o:o + m]; o += m
    ctr = acc[o:o + abi.PS_PC_COUNT]; o += abi.PS_PC_COUNT
    out = {
        "position_conversions": _i32(conv).reshape(m, 4, 4),
        "quality_per_mismatch": _i32(qsum).reshape(4, 4),
        "quality_per_mismatch_counts": _i32(qcnt).reshape(4, 4),
        "insertions_per_pos": ins.astype(np.float64),
        "deletions_per_pos": dele.astype(np.float64),
        "counters": _i32(ctr),
        "wide": acc.copy(),
    }
    if infer_q:
        out["quality_hist"] = acc[o:o + 256 * m].reshape(m, 256).copy()
    return out


class OracleFault(Exception):
    def __init__(self, code, ordinal):
        super().__init__(f"reference would throw: code {code} at record {ordinal}")
        self.code = code
        self.ordinal = ordinal


def profile_acc(ref, batch, max_len: int, infer_q: bool = False, threads: int = 1, first: int = 0, count=None,
                ordinal0: int = 0, acc: np.ndarray = None) -> np.ndarray:
    lib = load()
    n = lib.or_profile_acc_len(max_len, int(infer_q))
    if acc is None:
        acc = np.zeros(n, dtype=np.int64)
    rs = ref.as_struct()
    bs = batch.as_struct()
    if count is None:
        count = batch.n_reads - first
    fault = abi.ps_fault()
    st = lib.or_profile_run(C.byref(rs), C.byref(bs), max_len, int(infer_q), first, count, ordinal0, threads,
                            acc.ctypes.data, C.byref(fault))
    if st == abi.PS_ERR_REFERENCE_WOULD_THROW:
        raise OracleFault(fault.code, fault.read_ordinal)
    if st != 0:
        raise RuntimeError(f"oracle status {st}")
    return acc


def profile(ref, batch, max_len: int, infer_q: bool = False, threads: int = 1) -> dict:
    return split_acc(profile_acc(ref, batch, max_len, infer_q, threads), max_len, infer_q)


def pileup_count(ref, batch) -> int:
    """Run the T>C pileup loop and return only the number of closed clusters (timing legs of bench.py)."""
    lib = load()
    rs = ref.as_struct()
    bs = batch.as_struct()
    opts = abi.ps_pileup_opts(1, 0, 0, 0, 0, None)
    h = lib.or_pileup_run(C.byref(rs), C.byref(bs), C.byref(opts))
    try:
        ctr = abi.ps_pileup_counters()
        lib.or_pileup_counters(h, C.byref(ctr))
        return int(ctr.n_clusters)
    finally:
        lib.or_pileup_free(h)


def read_t2c_masks(ref, batch) -> np.ndarray:
    """uint64 per read: bit i = T>C at index i of the strand-oriented read (PileupClusters.java:637-661, no 51 limit,
    bits 0..61); 0 for records the pileup loop skips or would die on."""
    lib = load()
    rs = ref.as_struct()
    bs = batch.as_struct()
    out = np.zeros(batch.n_reads, dtype=np.uint64)
    st = lib.or_read_t2c_masks(C.byref(rs), C.byref(bs), out.ctypes.data)
    if st != 0:
        raise RuntimeError(f"oracle status {st}")
    return out


def pileup(ref, batch, first_running_id: int = 1, carry=None) -> dict:
    """carry=(contig, cluster_end): sharding emulation for the CPU tests of the halo merge (not reference
    behaviour); parity runs always pass the whole stream with carry=None."""
    lib = load()
    rs = ref.as_struct()
    bs = batch.as_struct()
    opts = abi.ps_pileup_opts(first_running_id, 0, 0, 0, 0, None)
    if carry is not None:
        opts.carry_valid, opts.carry_contig, opts.carry_cluster_end = 1, int(carry[0]), int(carry[1])
    h = lib.or_pileup_run(C.byref(rs), C.byref(bs), C.byref(opts))
    try:
        fault = abi.ps_fault()
        lib.or_pileup_fault(h, C.byref(fault))
        if fault.code:
            raise OracleFault(fault.code, fault.read_ordinal)
        ctr = abi.ps_pileup_counters()
        lib.or_pileup_counters(h, C.byref(ctr))
        clusters = np.zeros(ctr.n_clusters, dtype=abi.CLUSTER_DTYPE)
        sites = np.zeros(ctr.n_sites, dtype=abi.SITE_DTYPE)
        got = lib.or_pileup_copy(h, clusters.ctypes.data, ctr.n_clusters, sites.ctypes.data, ctr.n_sites)
        assert got == ctr.n_clusters
        open_c = np.zeros(1, dtype=abi.CLUSTER_DTYPE)
        open_s = np.zeros(4096, dtype=abi.SITE_DTYPE)
        k = lib.or_pileup_open(h, open_c.ctypes.data, open_s.ctypes.data, open_s.size)
        if k < 0:
            raise RuntimeError("open cluster has too many sites")
        head_c = np.zeros(1, dtype=abi.CLUSTER_DTYPE)
        head_s = np.zeros(4096, dtype=abi.SITE_DTYPE)
        kh = lib.or_pileup_head(h, head_c.ctypes.data, head_s.ctypes.data, head_s.size)
        cov = {}
        for which, name in ((0, "head_cov"), (1, "open_cov")):
            p0 = C.c_int32()
            ln = lib.or_pileup_boundary_cov(h, which, C.byref(p0), None, 0)
            a = np.zeros(max(int(ln), 0), dtype=np.uint32)
            if ln > 0:
                lib.or_pileup_boundary_cov(h, which, C.byref(p0), a.ctypes.data, a.size)
            cov[name] = (int(p0.value), a)
        return {
            "clusters": clusters, "sites": sites, **cov,
            "head_partial": head_c[0] if kh > 0 else None, "head_sites": head_s[:max(0, kh - 1)].copy(),
            "open_cluster": open_c[0] if k > 0 else None, "open_sites": open_s[:max(0, k - 1)].copy(),
            "counters": {f: getattr(ctr, f) for f, _ in abi.ps_pileup_counters._fields_},
        }
    finally:
        lib.or_pileup_free(h)
