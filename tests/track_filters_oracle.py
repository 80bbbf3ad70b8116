"""TEST INFRASTRUCTURE ONLY.

Two independent restatements of the track's read and base filters (ps_track_filter_opts; the contract is the header
comment next to ps_track_batch_ex3 in include/parasuite_b200.h), with the track's base counts and indel counts under
them.  They restate the track restatements of oracle/track_oracle.py, tests/track_bases_oracle.py and
tests/track_indels_oracle.py with the filters added, and leave those as they are:

  * track / track_bases / track_indels(records, genome, ..., **filters)   pure Python on Rec (py_oracle.Rec with the
                                                                           MAPQ) / Genome, including the file texts
  * track_cpp(ref, batch, bases=, indels=, **filters)                     C++ (track_filters_oracle.cpp, over
                                                                           track_oracle.cpp's batch walk) on the same SoA
                                                                           batches, aux arrays and packed reference as
                                                                           the CUDA path

filters: min_mapq, require_flags, exclude_flags, min_base_quality (0: off).  tests/test_track_filters_cpu.py checks that
the two agree.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

import py_oracle as po
import track_oracle as to
from parasuite_b200 import abi
from py_oracle import PS_FAULT_PAST_END, Genome, past_contig_end

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
SRC = os.path.join(HERE, "track_filters_oracle.cpp")
SO = os.path.join(REPO, "oracle", "_build", "libtrack_filters_oracle.so")
_lib = None


@dataclass
class Rec(po.Rec):
    """py_oracle.Rec with getMappingQuality()"""
    mapq: int = 255


def filtered(r: Rec, require_flags: int = 0, exclude_flags: int = 0, min_mapq: int = 0) -> int:
    """The track's record filter (ps_track_filter_opts): 0 kept, 1 dropped by a flag test, 2 for its MAPQ"""
    f = r.flag & 0xFFFF
    if (f & exclude_flags) or (f & require_flags) != require_flags:
        return 1
    return 2 if r.mapq < min_mapq else 0


def low_quality(r: Rec, i: int, min_base_quality: int) -> bool:
    """read base i is below min_base_quality (a record without qualities has none)"""
    return bool(min_base_quality) and len(r.qual) > 0 and r.qual[0] != 0xFF and r.qual[i] < min_base_quality


def track(records: List[Rec], genome: Genome, contig_order: Optional[List[str]] = None, *, min_mapq: int = 0,
          require_flags: int = 0, exclude_flags: int = 0, min_base_quality: int = 0) -> dict:
    """The contract of ps_track_batch / ps_track_bam, record by record.

    Records: those the pileup's loop keeps (unmapped and (I or D)-with-N records skipped, duplicates kept), with its
    faults (1 reference range, 8 block range, 9 more than 255 CIGAR operations) and no 51-position limit.  Positions: the
    CIGAR walked on the genome (M = X read and reference, D N reference, I S read, H P nothing).  Flag 0x10: minus
    strand.  Coverage: every aligned base.  T>C: plus ref T / read C, minus ref A / read G, reference base ACGTacgt, read
    base ACGT.  contig_order: the names in the order the records follow (a file's header), default the genome's.
    Returns runs / sites / counters and the three file texts; a fault wins over unsortedness.
    Filters (ps_track_filter_opts, all off at 0): a record that fails a flag or MAPQ test is absent (but a record past
    its contig's end is refused even so); a base below min_base_quality counts in "filter_counters" only, which the
    result has when any filter is set."""
    any_filter = bool(min_mapq or require_flags or exclude_flags or min_base_quality)
    fc = {"filtered_flags": 0, "filtered_mapq": 0, "low_quality_bases": [0, 0]}
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
        why = filtered(r, require_flags, exclude_flags, min_mapq)
        if why:
            if not r.unmapped and r.pos != 0 and len(r.cigar) <= 255 and past_contig_end(r, genome):
                raise to.TrackFault(ordinal, PS_FAULT_PAST_END)
            fc["filtered_flags" if why == 1 else "filtered_mapq"] += 1
            continue
        if r.unmapped:
            ctr["unmapped"] += 1
            continue
        if len(r.cigar) > 255:
            raise to.TrackFault(ordinal, 9)
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):
            ctr["skipped_due_indel"] += 1
            continue
        if r.pos == 0 or r.rname not in genome.contigs:
            raise to.TrackFault(ordinal, 1)
        if past_contig_end(r, genome):
            raise to.TrackFault(ordinal, PS_FAULT_PAST_END)
        seq = genome.contigs[r.rname]
        for rd1, rf1, n in r.alignment_blocks():       # every block is fetched before a base is looked at
            if rd1 - 1 + n > len(r.seq):
                raise to.TrackFault(ordinal, 8)
            if rf1 - 1 + n > len(seq):
                raise to.TrackFault(ordinal, 1)
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
                if low_quality(r, rd1 - 1 + k, min_base_quality):
                    fc["low_quality_bases"][s] += 1
                    continue
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
        raise to.TrackUnsorted("records are not coordinate-sorted")
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
    out = {"runs_plus": runs[0], "runs_minus": runs[1], "sites": sites, "counters": ctr, "files": files}
    if any_filter:
        out["filter_counters"] = fc
    return out


def effective_mask(substitutions: int) -> int:
    """the twelve substitution bits that count: 0 selects all, diagonal bits are ignored"""
    return (substitutions or 0xFFFF) & ~0x8421


def track_bases(records, genome, contig_order: Optional[List[str]] = None, *, min_coverage: int = 1,
                min_events: int = 1, substitutions: int = 0, **filters) -> dict:
    """track() with base counts: its dict plus "base_rows" (contig name, pos, strand, ref, cov, A, C, G, T,
    N), "base_totals" ((2, 4, 5) uint64) and files["bases.tsv"].  Raises what track() raises.  filters: track()'s
    (min_base_quality and the record filter)."""
    res = track(records, genome, contig_order, **filters)
    mbq = filters.get("min_base_quality", 0)
    rec_f = {k: filters.get(k, 0) for k in ("require_flags", "exclude_flags", "min_mapq")}
    mask, mc, me = effective_mask(substitutions), max(1, min_coverage), max(1, min_events)
    counts = ({}, {})                  # (contig, pos) -> [A, C, G, T, N] in strand orientation
    refc = {}                          # (contig, pos) -> plus-strand reference code
    totals = np.zeros((2, 4, 5), dtype=np.uint64)
    visited: List[str] = []
    for r in records:
        if filtered(r, **rec_f) or r.unmapped:
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
                if a not in b"ACGTacgt" or low_quality(r, rd1 - 1 + k, mbq):
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


CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
HEADER = "chrom\tpos\tstrand\tref\tcoverage\tdeletions\tinsertions\n"
TOTALS = ("deletion_ops", "deleted_bases", "insertion_ops", "inserted_bases", "unanchored_insertions")


def track_indels(records, genome, contig_order: Optional[List[str]] = None, *, min_depth: int = 1,
                 min_events: int = 1, **filters) -> dict:
    """track() with indel counts: its dict plus "indel_rows" (contig name, pos, strand, ref letter, cov, del,
    ins), "indel_totals" (as Context.track returns them) and files["indels.tsv"].  Raises what track() raises.
    filters: track()'s; indels are not filtered by base quality, the coverage is."""
    res = track(records, genome, contig_order, **filters)
    mbq = filters.get("min_base_quality", 0)
    rec_f = {k: filters.get(k, 0) for k in ("require_flags", "exclude_flags", "min_mapq")}
    md, me = max(1, min_depth), max(1, min_events)
    cov, dele, ins = ({}, {}), ({}, {}), ({}, {})       # (contig, pos) -> count, by strand
    tot = {k: [0, 0] for k in TOTALS}
    visited: List[str] = []
    for r in records:
        if filtered(r, **rec_f) or r.unmapped:
            continue
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):
            continue
        if r.rname not in visited:
            visited.append(r.rname)
        s = 1 if r.reverse else 0
        c, clen = r.rname, len(genome.contigs[r.rname])
        for rd1, rf1, n in r.alignment_blocks():
            for k, p in enumerate(range(rf1, rf1 + n)):
                if not low_quality(r, rd1 - 1 + k, mbq):
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
    with open(os.path.join(os.path.dirname(SO), ".track_filters_lock"), "w") as lock:
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
        lib.or_track_run_filtered.restype = C.c_void_p
        lib.or_track_run_filtered.argtypes = [C.POINTER(abi.ps_reference), C.POINTER(abi.ps_read_batch),
                                              C.POINTER(abi.ps_read_aux), C.POINTER(abi.ps_track_filter_opts),
                                              C.POINTER(abi.ps_track_opts), C.POINTER(abi.ps_track_indel_opts)]
        lib.or_track_filtered_status.restype = C.c_int
        lib.or_track_filtered_status.argtypes = [C.c_void_p, C.POINTER(abi.ps_track_counters), C.POINTER(abi.ps_fault),
                                                 C.POINTER(abi.ps_track_filter_counters),
                                                 C.POINTER(abi.ps_track_base_totals),
                                                 C.POINTER(abi.ps_track_indel_totals)]
        lib.or_track_filtered_copy.restype = C.c_int64
        lib.or_track_filtered_copy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        lib.or_track_filtered_free.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def track_cpp(ref, batch, *, bases: Optional[dict] = None, indels: Optional[dict] = None, min_mapq: int = 0,
              require_flags: int = 0, exclude_flags: int = 0, min_base_quality: int = 0) -> dict:
    """The C++ restatement on one whole batch (contigs in FASTA order): {"runs_plus", "runs_minus", "sites", "counters"}
    as track_oracle.track_cpp gives them, "filter_counters" (as Context.track gives them) when a filter is set, and with
    bases (the keywords min_coverage, min_events, substitutions of ps_track_opts) "base_rows" / "base_totals", with
    indels (min_depth, min_events) "indel_rows" / "indel_totals".  The record filter reads batch.sam_flags / batch.mapq.
    Raises track_oracle.TrackFault and TrackUnsorted as track() does."""
    lib = _load()
    rs, bs = ref.as_struct(), batch.as_struct()
    on = bool(min_mapq or require_flags or exclude_flags or min_base_quality)
    aux = batch.aux_struct() if on else None
    fo = abi.ps_track_filter_opts(min_mapq, require_flags, exclude_flags, min_base_quality) if on else None
    bo = None if bases is None else abi.ps_track_opts(1, bases.get("min_coverage", 1), bases.get("min_events", 1),
                                                       bases.get("substitutions", 0))
    io = None if indels is None else abi.ps_track_indel_opts(1, indels.get("min_depth", 1), indels.get("min_events", 1), 0)
    ref_ = (lambda x: C.byref(x) if x is not None else None)
    h = lib.or_track_run_filtered(C.byref(rs), C.byref(bs), ref_(aux), ref_(fo), ref_(bo), ref_(io))
    try:
        ctr, fault, fc = abi.ps_track_counters(), abi.ps_fault(), abi.ps_track_filter_counters()
        bt, it = abi.ps_track_base_totals(), abi.ps_track_indel_totals()
        st = lib.or_track_filtered_status(h, C.byref(ctr), C.byref(fault), C.byref(fc), C.byref(bt), C.byref(it))
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED):
            raise to.TrackFault(fault.read_ordinal, fault.code)
        if st == abi.PS_ERR_UNSORTED:
            raise to.TrackUnsorted("records are not coordinate-sorted")
        out = {"counters": ctr.as_dict()}
        items = [(0, "runs_plus", abi.TRACK_RUN_DTYPE, ctr.n_runs[0]), (1, "runs_minus", abi.TRACK_RUN_DTYPE, ctr.n_runs[1]),
                 (2, "sites", abi.TRACK_SITE_DTYPE, ctr.n_sites)]
        if bo is not None:
            items.append((3, "base_rows", abi.TRACK_BASE_ROW_DTYPE, bt.n_rows))
            out["base_totals"] = np.array(bt.bases, dtype=np.uint64).reshape(2, 4, 5)
        if io is not None:
            items.append((4, "indel_rows", abi.TRACK_INDEL_ROW_DTYPE, it.n_rows))
            out["indel_totals"] = it.as_dict()
        for which, name, dt, n in items:
            a = np.zeros(n, dtype=dt)
            if n:
                lib.or_track_filtered_copy(h, which, a.ctypes.data, n)
            out[name] = a
        if on:
            out["filter_counters"] = fc.as_dict()
        return out
    finally:
        lib.or_track_filtered_free(h)
