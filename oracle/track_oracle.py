"""TEST INFRASTRUCTURE ONLY.

Two independent restatements of the per-position T>C conversion and coverage track (tool `track`; the Java toolkit has
no such tool, so its contract is the header comment of ps_track_batch in include/parasuite_b200.h):

  * track(records, genome)   pure Python on the objects htsjdk hands the Java loops (py_oracle.Rec / Genome), including
                             the texts of the three output files
  * track_cpp(ref, batch)    C++ (track_oracle.cpp) on the same SoA batches and packed reference as the CUDA path, for
                             large batches

tests/test_track_cpu.py checks that the two agree.  Only tests/, __graft_entry__ and tools/bench_track.py import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from typing import List, Optional

import numpy as np

from py_oracle import PS_FAULT_PAST_END, Genome, Rec, past_contig_end

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(REPO, "para-suite_b200"))
from parasuite_b200 import abi  # noqa: E402  (struct layouts only)

SRC = os.path.join(HERE, "track_oracle.cpp")
SO = os.path.join(HERE, "_build", "libtrack_oracle.so")
_lib = None



# ---- per-position T>C conversion and coverage track (tool `track`; no Java counterpart) --------------------------------
class TrackFault(Exception):
    """A record the pileup's loop would die on (or, codes 9 and 10, one the SoA cannot hold): code as ps_fault.code."""

    def __init__(self, ordinal: int, code: int):
        super().__init__(f"record {ordinal}: fault {code}")
        self.ordinal = ordinal
        self.code = code


class TrackUnsorted(Exception):
    pass


def track(records: List[Rec], genome: Genome, contig_order: Optional[List[str]] = None) -> dict:
    """The contract of ps_track_batch / ps_track_bam, record by record.

    Records: those the pileup's loop keeps (unmapped and (I or D)-with-N records skipped, duplicates kept), with its
    faults (1 reference range, 8 block range, 9 more than 255 CIGAR operations) and no 51-position limit.  Positions: the
    CIGAR walked on the genome (M = X read and reference, D N reference, I S read, H P nothing).  Flag 0x10: minus
    strand.  Coverage: every aligned base.  T>C: plus ref T / read C, minus ref A / read G, reference base ACGTacgt, read
    base ACGT.  contig_order: the names in the order the records follow (a file's header), default the genome's.
    Returns runs / sites / counters and the three file texts; a fault wins over unsortedness."""
    order = list(contig_order) if contig_order is not None else list(genome.contigs)
    rank = {c: i for i, c in enumerate(order)}
    cov = ({}, {})
    t2c = ({}, {})
    ctr = {"num_reads_processed": 0, "unmapped": 0, "skipped_due_indel": 0, "reads_counted": 0,
           "aligned_bases": [0, 0], "t2c_events": [0, 0]}
    visited: List[str] = []
    prev = None
    unsorted = False
    for ordinal, r in enumerate(records):
        ctr["num_reads_processed"] += 1
        if r.unmapped:
            ctr["unmapped"] += 1
            continue
        if len(r.cigar) > 255:
            raise TrackFault(ordinal, 9)
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):
            ctr["skipped_due_indel"] += 1
            continue
        if r.pos == 0 or r.rname not in genome.contigs:
            raise TrackFault(ordinal, 1)
        if past_contig_end(r, genome):
            raise TrackFault(ordinal, PS_FAULT_PAST_END)
        seq = genome.contigs[r.rname]
        for rd1, rf1, n in r.alignment_blocks():       # every block is fetched before a base is looked at
            if rd1 - 1 + n > len(r.seq):
                raise TrackFault(ordinal, 8)
            if rf1 - 1 + n > len(seq):
                raise TrackFault(ordinal, 1)
        key = (rank.get(r.rname, len(order)), r.pos)
        if prev is not None and key < prev:
            unsorted = True
        prev = key
        if not visited or visited[-1] != r.rname:
            visited.append(r.rname)
        s = 1 if r.reverse else 0
        ctr["reads_counted"] += 1
        for rd1, rf1, n in r.alignment_blocks():
            for k in range(n):
                p = rf1 + k
                cov[s][(r.rname, p)] = cov[s].get((r.rname, p), 0) + 1
                ctr["aligned_bases"][s] += 1
                a = seq[p - 1]
                b = r.seq[rd1 - 1 + k]
                if a not in b"ACGTacgt" or b not in b"ACGT":
                    continue
                a = chr(a).upper()
                if (s == 0 and a == "T" and b == ord("C")) or (s == 1 and a == "A" and b == ord("G")):
                    t2c[s][(r.rname, p)] = t2c[s].get((r.rname, p), 0) + 1
                    ctr["t2c_events"][s] += 1
    if unsorted:
        raise TrackUnsorted("records are not coordinate-sorted")
    seen = []
    for c in visited:
        if c not in seen:
            seen.append(c)
    runs = ([], [])
    for s in (0, 1):
        for c in seen:
            ps = sorted(p for (cc, p) in cov[s] if cc == c)
            for p in ps:
                v = cov[s][(c, p)]
                if runs[s] and runs[s][-1][0] == c and runs[s][-1][2] == p - 1 and runs[s][-1][3] == v:
                    runs[s][-1][2] = p
                else:
                    runs[s].append([c, p - 1, p, v])
    sites = []
    for c in seen:
        ps = sorted({p for s in (0, 1) for (cc, p) in t2c[s] if cc == c})
        for p in ps:
            for s in (0, 1):
                if (c, p) in t2c[s]:
                    sites.append((c, p, "+-"[s], t2c[s][(c, p)], cov[s][(c, p)]))
    runs = tuple([tuple(x) for x in rs] for rs in runs)
    ctr["n_runs"] = [len(runs[0]), len(runs[1])]
    ctr["n_sites"] = len(sites)
    files = {
        "plus.bedGraph": "".join(f"{c}\t{a}\t{b}\t{v}\n" for c, a, b, v in runs[0]),
        "minus.bedGraph": "".join(f"{c}\t{a}\t{b}\t{v}\n" for c, a, b, v in runs[1]),
        "t2c.tsv": "chrom\tpos\tstrand\tt2c\tcoverage\n" + "".join(f"{c}\t{p}\t{s}\t{t}\t{v}\n" for c, p, s, t, v in sites),
    }
    return {"runs_plus": runs[0], "runs_minus": runs[1], "sites": sites, "counters": ctr, "files": files}


def _stale() -> bool:
    hdr = os.path.join(REPO, "include", "parasuite_b200.h")
    return (not os.path.exists(SO)) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(hdr))


def build(force: bool = False) -> str:
    """Build the C++ restatement if it is missing or older than its sources, under a file lock (several processes may
    call this at once); written under a temporary name and renamed."""
    if not (force or _stale()):
        return SO
    import fcntl
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    with open(os.path.join(os.path.dirname(SO), ".track_lock"), "w") as lock:
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
        lib.or_track_run.restype = C.c_void_p
        lib.or_track_run.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch)]
        lib.or_track_status.restype = C.c_int
        lib.or_track_status.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_counters), C.POINTER(abi.ps_fault)]
        lib.or_track_copy.restype = C.c_int64
        lib.or_track_copy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        lib.or_track_free.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def track_cpp(ref, batch) -> dict:
    """The C++ restatement on one whole batch (contigs in FASTA order): {"runs_plus", "runs_minus", "sites",
    "counters"} as abi.TRACK_RUN_DTYPE / TRACK_SITE_DTYPE arrays.  Raises TrackFault and TrackUnsorted as track()."""
    lib = _load()
    rs, bs = ref.as_struct(), batch.as_struct()
    h = lib.or_track_run(C.byref(rs), C.byref(bs))
    try:
        ctr, fault = abi.ps_track_counters(), abi.ps_fault()
        st = lib.or_track_status(h, C.byref(ctr), C.byref(fault))
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED):
            raise TrackFault(fault.read_ordinal, fault.code)
        if st == abi.PS_ERR_UNSORTED:
            raise TrackUnsorted("records are not coordinate-sorted")
        out = {"counters": ctr.as_dict()}
        for which, name, dt, n in ((0, "runs_plus", abi.TRACK_RUN_DTYPE, ctr.n_runs[0]),
                                   (1, "runs_minus", abi.TRACK_RUN_DTYPE, ctr.n_runs[1]),
                                   (2, "sites", abi.TRACK_SITE_DTYPE, ctr.n_sites)):
            a = np.zeros(n, dtype=dt)
            if n:
                lib.or_track_copy(h, which, a.ctypes.data, n)
            out[name] = a
        return out
    finally:
        lib.or_track_free(h)
