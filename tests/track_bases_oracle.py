"""TEST INFRASTRUCTURE ONLY.

Two independent restatements of the track's per-position base counts (ps_track_opts.base_counts; the contract is the
header comment next to ps_track_batch_ex in include/parasuite_b200.h), beside the track restatements of
oracle/track_oracle.py, which they call for everything the option leaves as it is:

  * track_bases(records, genome, ...)        pure Python on py_oracle.Rec / Genome, including the bases.tsv text
  * track_bases_cpp(ref, batch, ...)         C++ (track_bases_oracle.cpp, over track_oracle.cpp's batch walk) on the
                                             same SoA batches and packed reference as the CUDA path

tests/test_track_bases_cpu.py checks that the two agree.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional

import numpy as np

import track_oracle as to
from parasuite_b200 import abi

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
SRC = os.path.join(HERE, "track_bases_oracle.cpp")
SO = os.path.join(REPO, "oracle", "_build", "libtrack_bases_oracle.so")
CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
_lib = None


def effective_mask(substitutions: int) -> int:
    """the twelve substitution bits that count: 0 selects all, diagonal bits are ignored"""
    return (substitutions or 0xFFFF) & ~0x8421


def track_bases(records, genome, contig_order: Optional[List[str]] = None, *, min_coverage: int = 1,
                min_events: int = 1, substitutions: int = 0) -> dict:
    """track_oracle.track with base counts: its dict plus "base_rows" (contig name, pos, strand, ref, cov, A, C, G, T,
    N), "base_totals" ((2, 4, 5) uint64) and files["bases.tsv"].  Raises what track() raises."""
    res = to.track(records, genome, contig_order)
    mask, mc, me = effective_mask(substitutions), max(1, min_coverage), max(1, min_events)
    counts = ({}, {})                  # (contig, pos) -> [A, C, G, T, N] in strand orientation
    refc = {}                          # (contig, pos) -> plus-strand reference code
    totals = np.zeros((2, 4, 5), dtype=np.uint64)
    visited: List[str] = []
    for r in records:
        if r.unmapped:
            continue
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):
            continue
        if r.rname not in visited:
            visited.append(r.rname)
        s = 1 if r.reverse else 0
        flip = 3 if s else 0
        seq = genome.contigs[r.rname]
        for rd1, rf1, n in r.alignment_blocks():
            for k in range(n):
                p = rf1 + k
                a = seq[p - 1]
                if a not in b"ACGTacgt":
                    continue
                a = CODE[ord(chr(a).upper())]
                refc[(r.rname, p)] = a
                b = r.seq[rd1 - 1 + k]
                col = CODE[b] ^ flip if b in CODE else 4
                counts[s].setdefault((r.rname, p), [0] * 5)[col] += 1
                totals[s, a ^ flip, col] += 1
    rows = []
    for c in visited:
        for p in sorted({p for s in (0, 1) for (cc, p) in counts[s] if cc == c}):
            for s in (0, 1):
                n = counts[s].get((c, p))
                if n is None:
                    continue
                a = refc[(c, p)] ^ (3 if s else 0)
                cov = sum(n)
                picked = sum(n[b] for b in range(4) if b != a and (mask >> (4 * a + b)) & 1)
                if cov >= mc and picked >= me:
                    rows.append((c, p, "+-"[s], "ACGT"[a], cov, *n))
    res["base_rows"] = rows
    res["base_totals"] = totals
    res["files"]["bases.tsv"] = "chrom\tpos\tstrand\tref\tcoverage\tA\tC\tG\tT\tN\n" + "".join(
        "\t".join(str(x) for x in row) + "\n" for row in rows)
    return res


def _stale() -> bool:
    deps = [SRC, to.SRC, os.path.join(REPO, "include", "parasuite_b200.h")]
    return (not os.path.exists(SO)) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in deps)


def build(force: bool = False) -> str:
    """Build the C++ restatement if it is missing or older than its sources (file lock, temporary name, rename)."""
    if not (force or _stale()):
        return SO
    import fcntl
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    with open(os.path.join(os.path.dirname(SO), ".track_bases_lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or _stale():
                tmp = f"{SO}.tmp.{os.getpid()}"
                subprocess.check_call([os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-Wall", "-Wextra", "-fPIC",
                                       "-shared", "-o", tmp, SRC])
                os.replace(tmp, SO)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return SO


def _load() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        lib = C.CDLL(SO)
        lib.or_track_run_ex.restype = C.c_void_p
        lib.or_track_run_ex.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch),
                                        C.POINTER(abi.ps_track_opts)]
        lib.or_track_ex_status.restype = C.c_int
        lib.or_track_ex_status.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_counters), C.POINTER(abi.ps_fault)]
        lib.or_track_ex_copy.restype = C.c_int64
        lib.or_track_ex_copy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        lib.or_track_base_totals.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_base_totals)]
        lib.or_track_free_ex.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def track_bases_cpp(ref, batch, *, min_coverage: int = 1, min_events: int = 1, substitutions: int = 0) -> dict:
    """track_oracle.track_cpp with base counts: its dict plus "base_rows" (abi.TRACK_BASE_ROW_DTYPE) and "base_totals"."""
    lib = _load()
    rs, bs = ref.as_struct(), batch.as_struct()
    opts = abi.ps_track_opts(1, min_coverage, min_events, substitutions)
    h = lib.or_track_run_ex(C.byref(rs), C.byref(bs), C.byref(opts))
    try:
        ctr, fault = abi.ps_track_counters(), abi.ps_fault()
        st = lib.or_track_ex_status(h, C.byref(ctr), C.byref(fault))
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED):
            raise to.TrackFault(fault.read_ordinal, fault.code)
        if st == abi.PS_ERR_UNSORTED:
            raise to.TrackUnsorted("records are not coordinate-sorted")
        out = {"counters": ctr.as_dict()}
        tot = abi.ps_track_base_totals()
        lib.or_track_base_totals(h, C.byref(tot))
        for which, name, dt, n in ((0, "runs_plus", abi.TRACK_RUN_DTYPE, ctr.n_runs[0]),
                                   (1, "runs_minus", abi.TRACK_RUN_DTYPE, ctr.n_runs[1]),
                                   (2, "sites", abi.TRACK_SITE_DTYPE, ctr.n_sites),
                                   (3, "base_rows", abi.TRACK_BASE_ROW_DTYPE, tot.n_rows)):
            a = np.zeros(n, dtype=dt)
            if n:
                lib.or_track_ex_copy(h, which, a.ctypes.data, n)
            out[name] = a
        out["base_totals"] = np.array(tot.bases, dtype=np.uint64).reshape(2, 4, 5)
        return out
    finally:
        lib.or_track_free_ex(h)
