"""TEST INFRASTRUCTURE ONLY.

Two independent restatements of the track's per-position deletion and insertion counts
(ps_track_indel_opts.indel_counts; the contract is the header comment next to ps_track_batch_ex2 in
include/parasuite_b200.h), beside the track restatements of oracle/track_oracle.py, which they call for everything the
option leaves as it is:

  * track_indels(records, genome, ...)       pure Python on py_oracle.Rec / Genome, including the indels.tsv text
  * track_indels_cpp(ref, batch, ...)        C++ (track_indels_oracle.cpp, over track_oracle.cpp's batch walk) on the
                                             same SoA batches and packed reference as the CUDA path

tests/test_track_indels_cpu.py checks that the two agree.
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
SRC = os.path.join(HERE, "track_indels_oracle.cpp")
SO = os.path.join(REPO, "oracle", "_build", "libtrack_indels_oracle.so")
CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
HEADER = "chrom\tpos\tstrand\tref\tcoverage\tdeletions\tinsertions\n"
TOTALS = ("deletion_ops", "deleted_bases", "insertion_ops", "inserted_bases", "unanchored_insertions")
_lib = None


def track_indels(records, genome, contig_order: Optional[List[str]] = None, *, min_depth: int = 1,
                 min_events: int = 1) -> dict:
    """track_oracle.track with indel counts: its dict plus "indel_rows" (contig name, pos, strand, ref letter, cov, del,
    ins), "indel_totals" (as Context.track returns them) and files["indels.tsv"].  Raises what track() raises."""
    res = to.track(records, genome, contig_order)
    md, me = max(1, min_depth), max(1, min_events)
    cov, dele, ins = ({}, {}), ({}, {}), ({}, {})       # (contig, pos) -> count, by strand
    tot = {k: [0, 0] for k in TOTALS}
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
        c, clen = r.rname, len(genome.contigs[r.rname])
        for _, rf1, n in r.alignment_blocks():
            for p in range(rf1, rf1 + n):
                cov[s][(c, p)] = cov[s].get((c, p), 0) + 1
        rf = r.pos                                      # the next reference position, 1-based
        for op, n in r.cigar:
            if op == "D" and n:
                tot["deletion_ops"][s] += 1
                for p in range(rf, min(rf + n, clen + 1)):
                    dele[s][(c, p)] = dele[s].get((c, p), 0) + 1
                    tot["deleted_bases"][s] += 1
            elif op == "I" and n:
                tot["insertion_ops"][s] += 1
                tot["inserted_bases"][s] += n
                if r.pos < rf <= clen + 1:              # anchor rf - 1: consumed before the I, on the contig
                    ins[s][(c, rf - 1)] = ins[s].get((c, rf - 1), 0) + 1
                else:
                    tot["unanchored_insertions"][s] += 1
            if op in "MDN=X":
                rf += n
    rows = []
    for c in visited:
        seq = genome.contigs[c]
        for p in sorted({p for s in (0, 1) for d in (dele[s], ins[s]) for (cc, p) in d if cc == c}):
            for s in (0, 1):
                d, i, v = dele[s].get((c, p), 0), ins[s].get((c, p), 0), cov[s].get((c, p), 0)
                if d + i >= me and v + d >= md:
                    a = seq[p - 1]
                    ref = "ACGT"[CODE[ord(chr(a).upper())] ^ (3 if s else 0)] if a in b"ACGTacgt" else "N"
                    rows.append((c, p, "+-"[s], ref, v, d, i))
    res["indel_rows"] = rows
    res["indel_totals"] = dict(tot, n_rows=len(rows))
    res["files"]["indels.tsv"] = HEADER + "".join("\t".join(str(x) for x in row) + "\n" for row in rows)
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
    with open(os.path.join(os.path.dirname(SO), ".track_indels_lock"), "w") as lock:
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
        lib.or_track_run_indels.restype = C.c_void_p
        lib.or_track_run_indels.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch),
                                            C.POINTER(abi.ps_track_indel_opts)]
        lib.or_track_indels_status.restype = C.c_int
        lib.or_track_indels_status.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_counters), C.POINTER(abi.ps_fault)]
        lib.or_track_indels_copy.restype = C.c_int64
        lib.or_track_indels_copy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        lib.or_track_indel_totals.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_indel_totals)]
        lib.or_track_free_indels.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def track_indels_cpp(ref, batch, *, min_depth: int = 1, min_events: int = 1) -> dict:
    """track_oracle.track_cpp with indel counts: its dict plus "indel_rows" (abi.TRACK_INDEL_ROW_DTYPE) and
    "indel_totals" (as Context.track returns them)."""
    lib = _load()
    rs, bs = ref.as_struct(), batch.as_struct()
    opts = abi.ps_track_indel_opts(1, min_depth, min_events, 0)
    h = lib.or_track_run_indels(C.byref(rs), C.byref(bs), C.byref(opts))
    try:
        ctr, fault = abi.ps_track_counters(), abi.ps_fault()
        st = lib.or_track_indels_status(h, C.byref(ctr), C.byref(fault))
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED):
            raise to.TrackFault(fault.read_ordinal, fault.code)
        if st == abi.PS_ERR_UNSORTED:
            raise to.TrackUnsorted("records are not coordinate-sorted")
        out = {"counters": ctr.as_dict()}
        tot = abi.ps_track_indel_totals()
        lib.or_track_indel_totals(h, C.byref(tot))
        for which, name, dt, n in ((0, "runs_plus", abi.TRACK_RUN_DTYPE, ctr.n_runs[0]),
                                   (1, "runs_minus", abi.TRACK_RUN_DTYPE, ctr.n_runs[1]),
                                   (2, "sites", abi.TRACK_SITE_DTYPE, ctr.n_sites),
                                   (3, "indel_rows", abi.TRACK_INDEL_ROW_DTYPE, tot.n_rows)):
            a = np.zeros(n, dtype=dt)
            if n:
                lib.or_track_indels_copy(h, which, a.ctypes.data, n)
            out[name] = a
        out["indel_totals"] = tot.as_dict()
        return out
    finally:
        lib.or_track_free_indels(h)
