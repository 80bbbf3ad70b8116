"""The track's segments, compact space and window hand-offs at their limits, against the restatements and against the
shape each call should take.

One track call (track.cu) cuts the kept reads of a batch into SEGMENTS: a read opens one when its contig changes or it
starts more than one base past the running maximum end.  Segment s takes end - start + 2 slots of the compact space
(its bases and one slot for the -1 one past its end), M slots in all.  A window of the file tool (track_windows_run)
reports final rows only for the keys after the maximum end of the windows before (prev_end) and before its own last kept
start (the split); its head (first kept start .. prev_end) and its tail (split or prev_end + 1 .. its maximum end) come
back dense and wait in one pending region on the host, which hands positions to the writer once no later read can reach
them.  The writer joins runs that touch with equal coverage, so a run cut at a hand-off is one row.

Under PARASUITE_B200_DEBUG the library prints, per call, `[ps_track] segments S, compact M, reported R, head H, tail T`;
per window, in file order, `[ps_track_window] kept K, emitted E, pending P` (E: pending positions the window made final,
P: pending length after it); and per file `[ps_track_files] runs R+ R-, merged J+ J-, sites N` (J: runs joined by the
writer).  `shape` and `windows_model` predict every number from the records alone.

`Builder` writes its own contigs and records and names the paths each case is meant to reach; `paths_of` derives the
paths a case reaches from the model.  test_model_agrees_with_builder (no GPU) holds the two together and checks that the
Python and C++ restatements agree on every case; test_every_path_is_reached checks the union.  The GPU tests assert exact
equality with the restatements and the predicted lines: batches through host, device and misaligned views; windows
through one context, and through two contexts on one device (and on two devices where there are two), whose files must
be byte-identical."""
import random
import re

import numpy as np
import pytest

import py_oracle as po
import track_oracle as to
from helpers import to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi
from parasuite_b200.bamio import write_bam, write_fasta

CIGAR = re.compile(r"(\d+)([MIDNSHP=X])")
LOW = 0xFFFFFFFF


def ops(cigar):
    return [(int(n), op) for n, op in CIGAR.findall(cigar)]


def ref_span(cigar):
    return sum(n for n, op in ops(cigar) if op in "MDN=X")


# ---- builder ------------------------------------------------------------------------------------------------------
class Builder:
    """Records on contigs the builder writes.  A read copies the reference through its CIGAR (inserted and clipped bases
    are A), bar the positions where it is told to show a T>C (plus strand: reference T, read C; minus strand: reference
    A, read G); the reference base such an event needs is written into the contig when the case is made."""

    def __init__(self, lengths, seed=1, header=None):
        rng = np.random.default_rng(seed)
        self.names = [n for n, _ in lengths]
        self.seq = {n: bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes()) for n, ln in lengths}
        self.header = list(header) if header else list(self.names)
        self.reads = []              # (flag, contig, pos, cigar, events or None)
        self.need = {}
        self.intent = set()
        self.window = None           # records per window of the file tool (None: a batch case only)

    def read(self, contig, pos, cigar, rev=False, t2c=()):
        for p in t2c:
            base = "A" if rev else "T"
            assert self.need.setdefault((contig, p), base) == base, (contig, p)
        self.reads.append((16 if rev else 0, contig, pos, cigar, tuple(t2c)))
        return pos + ref_span(cigar) - 1

    def filler(self, k=1, skipped=False):
        """k records the track does not keep: unmapped (placed at the previous record, as mates are) or, skipped=True,
        mapped with I or D together with N."""
        _, c, p, _, _ = self.reads[-1] if self.reads else (0, self.header[0], 1, "", ())
        for _ in range(k):
            self.reads.append((0, c, p, "3M2I5N5M", None) if skipped else (4, c, p, "10M", None))

    def cut(self):
        """Unmapped fillers up to the next window boundary: the next record opens a window."""
        while len(self.reads) % self.window:
            self.filler()

    def make(self):
        seq = {n: bytearray(s) for n, s in self.seq.items()}
        for (c, p), base in self.need.items():
            seq[c][p - 1] = ord(base)
        recs = []
        for flag, c, pos, cigar, ev in self.reads:
            L = sum(n for n, op in ops(cigar) if op in "MIS=X")
            s = bytearray(b"A" * L)
            if ev is not None:
                rp, qp = pos, 0
                for n, op in ops(cigar):
                    if op in "M=X":
                        for k in range(n):
                            s[qp + k] = seq[c][rp + k - 1]
                        rp += n; qp += n
                    elif op in "SI":
                        qp += n
                    elif op in "DN":
                        rp += n
                for p in ev:
                    qp = aligned_offset(pos, cigar, p)
                    assert qp is not None, (pos, cigar, p)
                    s[qp] = ord("G" if flag & 16 else "C")
            recs.append(Record(flag, c, pos, cigar, bytes(s), bytes([30]) * L))
        return [(n, bytes(seq[n])) for n in self.names], recs


def aligned_offset(pos, cigar, p):
    rp, qp = pos, 0
    for n, op in ops(cigar):
        if op in "M=X":
            if rp <= p < rp + n:
                return qp + p - rp
            rp += n; qp += n
        elif op in "SI":
            qp += n
        elif op in "DN":
            rp += n
    return None


# ---- model --------------------------------------------------------------------------------------------------------
def kept_keys(recs, order):
    """(start key, end key) of the records the track keeps, in record order; keys (rank + 1) << 32 | 1-based position."""
    out = []
    for r in recs:
        if r.flag & 4:
            continue
        kinds = {op for _, op in ops(r.cigar)}
        if kinds & {"I", "D"} and "N" in kinds:
            continue
        hi = (order.index(r.rname) + 1) << 32
        out.append((hi | r.pos, hi | (r.pos + ref_span(r.cigar) - 1)))
    return out


def segments(items):
    """[start key, maximum end key] of every segment."""
    segs, run = [], 0
    for ks, ke in items:
        if not run or run >> 32 != ks >> 32 or (run & LOW) + 1 < (ks & LOW):
            segs.append([ks, ke])
        else:
            segs[-1][1] = max(segs[-1][1], ke)
        run = max(run, ke)
    return segs


def shape(items, prev_end=0, windowed=False):
    """(segments, M, reported, head, tail) of one call on the kept reads `items`."""
    if not items:
        return (0, 0, 0, 0, 0)
    segs = segments(items)
    lens = [e - s + 2 for s, e in segs]
    M = sum(lens)
    if not windowed:
        return (len(segs), M, M, 0, 0)

    def slots_below(key):           # compact slots whose key is < key (slot keys ascend)
        return sum(min(max(key - s, 0), n) for (s, _), n in zip(segs, lens))
    f, split, E = items[0][0], max(k for k, _ in items), max(e for _, e in items)
    reported = max(0, slots_below(split) - slots_below(prev_end + 1)) if prev_end else slots_below(split)
    head = prev_end - f + 1 if prev_end and prev_end >> 32 == f >> 32 and f <= prev_end else 0
    t0 = max(split, prev_end + 1)
    tail = E - t0 + 1 if t0 >> 32 == E >> 32 and t0 <= E else 0
    return (len(segs), M, reported, head, tail)


def runs_in(runs, order, lo, hi):
    """Runs (contig, start0, end0, cov) with a position whose key is in [lo, hi]."""
    n = 0
    if lo > hi:
        return 0
    for c, a, b, _ in runs:
        k = (order.index(c) + 1) << 32
        if k | (a + 1) <= hi and k | b >= lo:
            n += 1
    return n


def windows_model(recs, order, w, want):
    """Per window: (shape of its call or None without a call, (kept, emitted, pending)); and the files line
    (runs+, runs-, merged+, merged-, sites).  `want`: the Python restatement's result for the whole file."""
    calls, lines, blocks = [], [], []
    prev_end, p0, plen = 0, 0, 0
    for a in range(0, len(recs), w):
        items = kept_keys(recs[a:a + w], order)
        sh = shape(items, prev_end, True)
        calls.append(sh)
        if not items:
            lines.append((0, 0, plen))
            continue
        _, _, _, head, tail = sh
        split = max(k for k, _ in items)
        if plen:
            assert head == 0 or (items[0][0] >= p0 and items[0][0] + head <= p0 + plen), "head outside the pending region"
            k = (plen if split > p0 else 0) if split >> 32 != p0 >> 32 else min(max(split - p0, 0), plen)
        else:
            k = 0
        if k:
            blocks.append((p0, p0 + k - 1))
        p0, plen = p0 + k, plen - k
        blocks.append((prev_end + 1, split - 1))
        if tail:
            if not plen:
                p0 = max(split, prev_end + 1)
            plen += tail
        lines.append((len(items), k, plen))
        prev_end = max([prev_end] + [e for _, e in items])
    if plen:
        blocks.append((p0, p0 + plen - 1))
    pieces = [sum(runs_in(want[n], order, lo, hi) for lo, hi in blocks) for n in ("runs_plus", "runs_minus")]
    nr = [len(want["runs_plus"]), len(want["runs_minus"])]
    return calls, lines, (nr[0], nr[1], pieces[0] - nr[0], pieces[1] - nr[1], len(want["sites"]))


# ---- paths --------------------------------------------------------------------------------------------------------
BATCH_PATHS = {"join+1", "new+2", "max-from-back", "contig-adjacent", "cigar-edge-DN", "zero-op", "long-splice",
               "zero-span-inside", "zero-span-pos1", "zero-span-last", "short-contig", "ends-on-last-base",
               "deep", "minus-only", "no-t2c", "one-read", "no-segments", "zero-coverage-inside"}
WINDOW_PATHS = {"head", "first+1", "first+2", "empty-range", "empty-tail", "no-kept-window", "contig-change-pending",
                "writer-merge", "many-windows"}


def paths_of(case, contigs, recs, want, win=None):
    """The paths the case reaches, derived from the records, the restatement's rows and the model."""
    order = case.header
    lengths = dict((n, len(s)) for n, s in contigs)
    items = kept_keys(recs, order)
    kept = [r for r in recs if not r.flag & 4 and not ({"I", "D"} & {op for _, op in ops(r.cigar)}
                                                       and "N" in r.cigar)]
    got = set()
    run, run_from, prev = 0, None, None
    for j, (ks, ke) in enumerate(items):
        if run and run >> 32 == ks >> 32:
            d = (ks & LOW) - (run & LOW)
            if d in (1, 2):
                got.add("join+1" if d == 1 else "new+2")
                if run_from != j - 1:
                    got.add("max-from-back")
        if prev is not None and prev[1] >> 32 != ks >> 32:
            pr, r = kept[j - 1], kept[j]
            if (pr.pos + ref_span(pr.cigar) - 1 == lengths[pr.rname] and r.pos == 1
                    and case.names.index(r.rname) == case.names.index(pr.rname) + 1):
                got.add("contig-adjacent")
        if ke > run:
            run, run_from = ke, j
        prev = (ks, ke)
    segs = segments(items)
    for j, r in enumerate(kept):
        o = ops(r.cigar)
        if o[0][1] in "DN" or o[-1][1] in "DN":
            got.add("cigar-edge-DN")
        if any(n == 0 for n, _ in o):
            got.add("zero-op")
        if any(op == "N" and n >= 1000 for n, op in o):
            got.add("long-splice")
        if ref_span(r.cigar) == 0:
            ks, ke = items[j]
            if r.pos == 1:
                got.add("zero-span-pos1")
            if j == len(kept) - 1 and ks > max(e for _, e in items):
                got.add("zero-span-last")
            if any(s < ks and e >= ks for s, e in segs):
                got.add("zero-span-inside")
        if lengths[r.rname] < 16:
            got.add("short-contig")
        if ref_span(r.cigar) and r.pos + ref_span(r.cigar) - 1 == lengths[r.rname]:
            got.add("ends-on-last-base")
    if zero_inside(segs, want, order):
        got.add("zero-coverage-inside")
    if any(t > 65536 for _, _, _, t, _ in want["sites"]):
        got.add("deep")
    if kept and all(r.flag & 16 for r in kept):
        got.add("minus-only")
    if kept and not want["sites"]:
        got.add("no-t2c")
    if len(recs) == 1 and kept:
        got.add("one-read")
    if not segs:
        got.add("no-segments")
    if win:
        calls, lines, files = windows_model(recs, order, win, want)
        firsts = []
        prev_end = 0
        for a in range(0, len(recs), win):
            it = kept_keys(recs[a:a + win], order)
            if it and prev_end and it[0][0] >> 32 == prev_end >> 32:
                firsts.append((it[0][0] & LOW) - (prev_end & LOW))
            prev_end = max([prev_end] + [e for _, e in it])
        got |= {"first+1" for d in firsts if d == 1} | {"first+2" for d in firsts if d == 2}
        if any(c[3] for c in calls):
            got.add("head")
        if any(c[0] and c[2] == 0 for c in calls):
            got.add("empty-range")
        if any(c[0] and c[4] == 0 for c in calls):
            got.add("empty-tail")
        for i in range(1, len(lines) - 1):
            if lines[i][0] == 0 and lines[i - 1][2] and lines[i - 1][0]:
                got.add("no-kept-window")
        pend_key = pending_contigs(recs, order, win, lines)
        if pend_key:
            got.add("contig-change-pending")
        if files[2] or files[3]:
            got.add("writer-merge")
        if len(calls) >= 1000:
            got.add("many-windows")
    return got


def zero_inside(segs, want, order):
    """A position inside a segment that no read covers on either strand."""
    cov = set()
    for n in ("runs_plus", "runs_minus"):
        for c, a, b, _ in want[n]:
            k = (order.index(c) + 1) << 32
            cov.add((k | (a + 1), k | b))
    iv = sorted(cov)
    for s, e in segs:
        pos = s
        for a, b in iv:
            if b < pos or a > e:
                continue
            if a > pos:
                return True
            pos = max(pos, b + 1)
        if pos <= e:
            return True
    return False


def pending_contigs(recs, order, win, lines):
    """A window whose first kept read is on another contig than the pending region left open before it."""
    pend_contig = None
    for i, a in enumerate(range(0, len(recs), win)):
        it = kept_keys(recs[a:a + win], order)
        if it and pend_contig is not None and it[0][0] >> 32 != pend_contig and lines[i - 1][2]:
            return True
        if it:
            pend_contig = max(e for _, e in it) >> 32 if lines[i][2] else pend_contig
    return False


# ---- cases --------------------------------------------------------------------------------------------------------
def case_segment_edges():
    b = Builder([("chr1", 3000)], seed=11)
    b.intent |= {"join+1", "new+2", "max-from-back"}
    e = b.read("chr1", 100, "10M", t2c=[103])
    e = b.read("chr1", e + 1, "10M", rev=True)                   # at the running maximum end + 1: same segment
    e = b.read("chr1", e + 2, "10M")                             # + 2: a new segment
    e = b.read("chr1", 400, "100M", t2c=[450])                   # the maximum from a read further back
    b.read("chr1", 410, "10M")
    b.read("chr1", e + 1, "10M", t2c=[e + 3])                    # joins through the long read's end
    e = b.read("chr1", 800, "100M", rev=True)
    b.read("chr1", 810, "10M", rev=True)
    b.read("chr1", e + 2, "10M", rev=True)                       # opens a segment past the long read's end
    b.read("chr1", 2000, "5M")
    return b


def case_contig_edges(header=None):
    b = Builder([("chr1", 50), ("chr2", 40), ("chr3", 30)], seed=12, header=header)
    b.intent |= {"contig-adjacent", "ends-on-last-base"}
    for c in b.header:
        ln = len(b.seq[c])
        b.read(c, 1, "10M", rev=c == "chr2", t2c=[4])
        b.read(c, ln - 9, "10M", t2c=[ln])                        # ends on the contig's last base
    return b


def case_cigar_edges():
    b = Builder([("chr1", 2000)], seed=13)
    b.intent |= {"cigar-edge-DN", "zero-op", "zero-coverage-inside"}
    b.read("chr1", 100, "3D10M", t2c=[105])
    b.read("chr1", 105, "10M4N", rev=True)
    b.read("chr1", 110, "2N8M2D")
    b.read("chr1", 120, "0M10M", t2c=[122])
    b.read("chr1", 125, "5M0N5M")
    b.read("chr1", 130, "10M0M")
    b.read("chr1", 140, "2S6M3N")
    b.read("chr1", 300, "5N5M")                                   # a segment whose first positions nobody covers
    return b


def case_long_splices():
    b = Builder([("chr1", 400_000)], seed=14)
    b.intent |= {"long-splice", "zero-coverage-inside"}
    b.read("chr1", 1000, "20M200000N20M", t2c=[1005])
    b.read("chr1", 1010, "15M1000N15M", rev=True)
    for p in (5000, 60000, 150000, 200500):
        b.read("chr1", p, "25M", rev=p % 2 == 1)
    b.read("chr1", 201_030, "10M50000N10M", t2c=[201_032])
    b.read("chr1", 260_000, "12M")
    return b


def case_zero_span():
    b = Builder([("chr1", 500), ("chr2", 300)], seed=15)
    b.intent |= {"zero-span-pos1", "zero-span-inside", "zero-span-last"}
    b.read("chr1", 1, "5S5I")                                     # POS 1, no reference span
    b.read("chr1", 1, "20M", t2c=[3])
    b.read("chr1", 10, "4S6I")                                    # inside a segment
    b.read("chr1", 300, "30M", rev=True)
    b.read("chr1", 500, "3S2I")                                   # on the contig's last base
    b.read("chr2", 50, "30M", t2c=[60])
    b.read("chr2", 80, "5S5I")                                    # the last kept read: end < start
    return b


def case_short_contigs():
    b = Builder([("c1", 1), ("c5", 5), ("c15", 15), ("c16", 16), ("c40", 40)], seed=16)
    b.intent |= {"short-contig", "ends-on-last-base"}
    b.read("c1", 1, "1M")
    b.read("c5", 1, "5M", rev=True)
    b.read("c5", 3, "1S3M", t2c=[5])
    b.read("c15", 5, "11M", t2c=[15])
    b.read("c16", 1, "16M", rev=True, t2c=[16])
    b.read("c40", 31, "10M")
    return b


def case_deep():
    b = Builder([("chr1", 1000)], seed=17)
    b.intent |= {"deep"}
    for k in range(65_600):
        b.read("chr1", 100 + (k >= 32_800), "20M", t2c=[110])
    for k in range(65_600):
        b.read("chr1", 102, "20M", rev=True, t2c=[115])
    return b


def case_minus_only():
    b = Builder([("chr1", 2000)], seed=18)
    b.intent |= {"minus-only"}
    for p in range(10, 1500, 37):
        b.read("chr1", p, "30M", rev=True, t2c=[p + 7] if p % 2 else ())
    return b


def case_no_t2c():
    b = Builder([("chr1", 2000), ("chr2", 2000)], seed=19)
    b.intent |= {"no-t2c"}
    for c in ("chr1", "chr2"):
        for p in range(5, 1800, 53):
            b.read(c, p, "40M", rev=p % 3 == 0)
    return b


def case_one_read():
    b = Builder([("chr1", 200)], seed=20)
    b.intent |= {"one-read"}
    b.read("chr1", 50, "36M", t2c=[60])
    return b


def case_none_kept():
    b = Builder([("chr1", 200)], seed=21)
    b.intent |= {"no-segments"}
    b.read("chr1", 50, "36M")
    b.reads.pop()
    b.reads.append((0, "chr1", 10, "5M2I5N5M", None))
    b.filler(3)
    b.filler(2, skipped=True)
    return b


BATCH_CASES = {
    "segment-edges": case_segment_edges, "contig-edges": case_contig_edges, "cigar-edges": case_cigar_edges,
    "long-splices": case_long_splices, "zero-span": case_zero_span, "short-contigs": case_short_contigs,
    "deep": case_deep, "minus-only": case_minus_only, "no-t2c": case_no_t2c, "one-read": case_one_read,
    "none-kept": case_none_kept,
}


def win_head_and_firsts():
    b = Builder([("chr1", 5000)], seed=31)
    b.window = 4
    b.intent |= {"head", "first+1", "first+2"}
    e = b.read("chr1", 100, "50M", t2c=[120])
    b.cut()
    b.read("chr1", 120, "20M", rev=True)                          # head: 120 .. 149
    e = b.read("chr1", 130, "40M", t2c=[160])
    b.cut()
    e = b.read("chr1", e + 1, "10M")                              # prev_end + 1
    b.cut()
    e = b.read("chr1", e + 2, "10M", rev=True)                    # prev_end + 2
    b.read("chr1", e - 3, "4M")                                   # the tail starts at this split, not at the first read
    b.cut()
    return b


def win_inside_a_splice():
    b = Builder([("chr1", 100_000)], seed=32)
    b.window = 3
    b.intent |= {"empty-range", "empty-tail", "head"}
    b.read("chr1", 1000, "10M50000N10M", t2c=[1003])
    b.cut()
    b.read("chr1", 2000, "10M", t2c=[2004])                      # a whole window inside the splice
    b.read("chr1", 3000, "10M", rev=True)
    b.cut()
    b.read("chr1", 40000, "30M")
    b.cut()
    b.read("chr1", 60000, "10M")
    return b


def win_no_kept_between():
    b = Builder([("chr1", 2000), ("chr2", 2000)], seed=33)
    b.window = 5
    b.intent |= {"no-kept-window", "contig-change-pending"}
    b.read("chr1", 100, "30M")
    b.cut()
    b.filler(3)
    b.filler(2, skipped=True)                                     # a window with no kept read
    b.read("chr1", 120, "30M")
    b.cut()
    b.read("chr1", 1990, "11M", t2c=[1995])                      # the pending region is open on chr1 ...
    b.cut()
    b.read("chr2", 1, "10M", rev=True)                            # ... when chr2 starts
    b.read("chr2", 5, "10M", rev=True)
    return b


def win_run_over_windows():
    b = Builder([("chr1", 5000)], seed=34)
    b.window = 1
    b.intent |= {"writer-merge", "first+1"}
    p = 100
    for _ in range(40):                                          # one run of coverage 1 over 40 windows
        p = b.read("chr1", p, "10M") + 1
    for _ in range(30):                                          # and one of coverage 2 on the minus strand
        b.read("chr1", p, "10M", rev=True)
        b.read("chr1", p, "10M", rev=True)
        p += 10
    return b


def win_many_in_splice():
    b = Builder([("chr1", 300_000)], seed=35)
    b.window = 7
    b.intent |= {"many-windows", "head", "empty-range"}
    rng = random.Random(35)
    b.read("chr1", 1000, "20M200000N20M", t2c=[1004])
    b.cut()
    p = 1100
    for _ in range(2500):
        k = rng.randint(1, 7)
        for _ in range(k):
            p += rng.randint(0, 40)
            b.read("chr1", p, f"{rng.randint(10, 60)}M", rev=rng.random() < 0.5)
        b.cut()
    return b


WINDOW_CASES = {
    "head-and-firsts": win_head_and_firsts, "inside-a-splice": win_inside_a_splice,
    "no-kept-between": win_no_kept_between, "run-over-windows": win_run_over_windows,
    "many-in-splice": win_many_in_splice,
    "contig-edges-header": lambda: windowed(case_contig_edges(["chr2", "chr1", "chr3"]), 1),
}
for _name, _fn in BATCH_CASES.items():
    if _name != "deep":
        WINDOW_CASES[f"{_name}-w1"] = (lambda fn: lambda: windowed(fn(), 1))(_fn)
WINDOW_CASES["deep-w4093"] = lambda: windowed(case_deep(), 4093)


def windowed(b, w):
    b.window = w
    b.intent = set()
    return b


_made = {}


def made(name):
    """(builder, contigs, records, Python restatement's result), cached."""
    if name not in _made:
        b = (BATCH_CASES.get(name) or WINDOW_CASES[name])()
        contigs, recs = b.make()
        want = to.track(to_py(recs), po.Genome(dict(contigs)), b.header)
        _made[name] = (b, contigs, recs, want)
    return _made[name]


def reached(name):
    b, contigs, recs, want = made(name)
    return paths_of(b, contigs, recs, want, b.window)


# ---- no GPU -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(BATCH_CASES) + list(WINDOW_CASES))
def test_model_agrees_with_builder(name):
    """The paths the builder meant are the paths the model derives; both restatements agree on the case."""
    b, contigs, recs, want = made(name)
    got = reached(name)
    assert b.intent <= got, (name, b.intent - got)
    if b.header == b.names:
        from test_track_cpu import _same
        ref = PackedReference.from_contigs(contigs)
        _same(want, to.track_cpp(ref, ReadBatch.from_records(recs, ref)), b.names)


def test_every_path_is_reached():
    got = set()
    for name in list(BATCH_CASES) + list(WINDOW_CASES):
        got |= reached(name)
    assert BATCH_PATHS <= got, BATCH_PATHS - got
    assert WINDOW_PATHS <= got, WINDOW_PATHS - got


def test_model_on_hand_derived_calls():
    """The model at the segment rule's edge and on the hand-off formulas, by hand."""
    k = lambda p: (1 << 32) | p
    assert shape([(k(1), k(10)), (k(11), k(20))]) == (1, 21, 21, 0, 0)
    assert shape([(k(1), k(10)), (k(12), k(20))]) == (2, 11 + 10, 21, 0, 0)
    assert shape([(k(1), k(0))]) == (1, 1, 1, 0, 0)                        # zero span at POS 1
    # prev_end 15: head 5 .. 15, reported (15, 20) = 16 .. 19, tail 20 .. 30
    assert shape([(k(5), k(30)), (k(20), k(25))], k(15), True) == (1, 27, 4, 11, 11)
    # a window inside an earlier splice: nothing reported, no tail
    assert shape([(k(20), k(29)), (k(40), k(49))], k(100), True) == (2, 22, 0, 81, 0)


# ---- GPU ----------------------------------------------------------------------------------------------------------
TRACK_LINE = re.compile(r"\[ps_track\] segments (\d+), compact (\d+), reported (\d+), head (\d+), tail (\d+)")
WINDOW_LINE = re.compile(r"\[ps_track_window\] kept (\d+), emitted (\d+), pending (\d+)")
FILES_LINE = re.compile(r"\[ps_track_files\] runs (\d+) (\d+), merged (\d+) (\d+), sites (\d+)")


def _ints(rx, text):
    return [tuple(int(x) for x in m) for m in rx.findall(text)]


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture
def debug(monkeypatch, capfd):
    """debug(fn): fn() and the stderr it printed (PARASUITE_B200_DEBUG is looked up on every call)."""
    monkeypatch.setenv("PARASUITE_B200_DEBUG", "1")

    def run(fn):
        capfd.readouterr()
        out = fn()
        return out, capfd.readouterr().err
    return run


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BATCH_CASES))
def test_batch_cases(ctx, debug, name):
    from test_gpu_bitparallel_edges import views
    from test_gpu_track import _equal
    b, contigs, recs, _ = made(name)
    ref = PackedReference.from_contigs(contigs)
    batch = ReadBatch.from_records(recs, ref)
    exp = to.track_cpp(ref, batch)
    want = shape(kept_keys(recs, b.names))
    ctx.upload_reference(ref)
    for how, view in views(batch):
        got, err = debug(lambda: ctx.track(view))
        _equal(got, exp, f"{name} {how}")
        assert _ints(TRACK_LINE, err) == [want], (name, how, err)


def _texts(prefix):
    return {k: open(f"{prefix}.{k}").read() for k in ("plus.bedGraph", "minus.bedGraph", "t2c.tsv")}


def _files(tmp_path, name):
    b, contigs, recs, want = made(name)
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / "reads.bam")
    write_fasta(fa, contigs)
    lengths = dict(contigs)
    write_bam(path, [(c, len(lengths[c])) for c in b.header], recs)
    return b, fa, path, recs, want


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WINDOW_CASES))
def test_window_cases(tmp_path, monkeypatch, debug, name):
    """One context: the files equal the Python restatement's, every call and window prints what the model predicts."""
    from parasuite_b200.runtime import Context
    b, fa, path, recs, want = _files(tmp_path, name)
    calls, lines, files = windows_model(recs, b.header, b.window, want)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(b.window))
    c = Context(0)
    try:
        c.load_fasta(fa)
        ctr, err = debug(lambda: c.track_bam(path, str(tmp_path / "one")))
    finally:
        c.close()
    assert _texts(tmp_path / "one") == want["files"]
    assert ctr["n_runs"] == want["counters"]["n_runs"] and ctr["n_sites"] == want["counters"]["n_sites"]
    assert _ints(TRACK_LINE, err) == calls, name
    assert _ints(WINDOW_LINE, err) == lines, name
    assert _ints(FILES_LINE, err) == [files], name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WINDOW_CASES))
def test_window_cases_on_several_contexts(tmp_path, monkeypatch, name):
    """Windows round-robin over two contexts on one device (and over two devices where there are two): the same
    bytes as the restatement, hence as one context."""
    import torch
    from parasuite_b200.runtime import MultiContext
    b, fa, path, recs, want = _files(tmp_path, name)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(b.window))
    sets = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() > 1 else [])
    for devs in sets:
        m = MultiContext(devs)
        try:
            m.load_fasta(fa)
            m.track_bam(path, str(tmp_path / "multi"))
        finally:
            m.close()
        assert _texts(tmp_path / "multi") == want["files"], devs


# ---- entry points -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_compact_pinned_and_uploaded_views(ctx, debug):
    """The compact host form (one flag byte per read, 16-bit starts) through ps_track_batch, and an uploaded view
    through ps_track_batch_device on a stream of its own: both equal the C++ restatement and print the model's line.
    (The second call waits for the staging copy's event; a missing wait could still pass by timing, so the wait itself
    is not pinned here.)"""
    import torch
    from parasuite_b200.runtime import PinnedBatch
    from test_gpu_track import _equal
    b = Builder([("chr1", 300_000), ("chr2", 200_000)], seed=41)
    rng = random.Random(41)
    for c, ln in (("chr1", 300_000), ("chr2", 200_000)):
        p = 1
        while p < ln - 100:
            b.read(c, p, "36M", rev=rng.random() < 0.5, t2c=[p + 5] if rng.random() < 0.3 else ())
            p += rng.choice((1, 2, 3, 7, 36, 37, 38, 200))
    contigs, recs = b.make()
    ref = PackedReference.from_contigs(contigs)
    batch = ReadBatch.from_records(recs, ref)
    exp = to.track_cpp(ref, batch)
    want = [shape(kept_keys(recs, b.names))]
    ctx.upload_reference(ref)
    pb = PinnedBatch(batch, compact=True)
    assert pb.compact and pb.compact_start
    got, err = debug(lambda: ctx.track(pb))
    _equal(got, exp, "compact pinned")
    assert _ints(TRACK_LINE, err) == want
    s = torch.cuda.Stream()
    view = ctx.upload(pb)
    got, err = debug(lambda: ctx.track(view, stream=s.cuda_stream))
    _equal(got, exp, "uploaded view on its own stream")
    assert _ints(TRACK_LINE, err) == want


def test_renderer_matches_the_restatement():
    """render() of track_cpp's rows gives the Python restatement's file texts (on a prefix of the scale records)."""
    contigs, recs = scale_records(20_000)
    ref = PackedReference.from_contigs(contigs)
    want = to.track(to_py(recs), po.Genome(dict(contigs)))["files"]
    assert render(to.track_cpp(ref, ReadBatch.from_records(recs, ref)), [n for n, _ in contigs]) == want


# ---- records past a contig's end ----------------------------------------------------------------------------------
# A mapped record that consumes no reference (5S5I) at POS > its contig's length has no offset on its contig.  The
# pileup, clust and track refuse it by name (PS_ERR_UNSUPPORTED, PS_FAULT_PAST_END, its ordinal); the profile keeps the
# JVM's fault: the empty fetch at POS = length + 1 dies on refSequenceForRead[0], a fetch further out in htsjdk.
PAST = [("chr1", 38), ("chr2", 60)]


def past_end_case(where):
    """(contigs, records, ordinal of the past-end record, profile fault code)."""
    rng = np.random.default_rng(5)
    contigs = [(n, np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes()) for n, ln in PAST]
    seq = dict(contigs)
    ok = lambda c, p: Record(0, c, p, "8M", seq[c][p - 1:p + 7], bytes([30]) * 8)
    zero = lambda c, p: Record(0, c, p, "5S5I", b"ACGTACGTAC", bytes([30]) * 10)
    if where == "last-contig":                   # chr2 POS 61: one past the genome
        return contigs, [ok("chr1", 3), ok("chr2", 10), zero("chr2", 61)], 2, abi.PS_THROW_EMPTY_REF
    if where == "middle-contig":                 # chr1 POS 39, then chr2:1
        return contigs, [ok("chr1", 3), zero("chr1", 39), ok("chr2", 1)], 1, abi.PS_THROW_EMPTY_REF
    if where == "further-out":                   # chr1 POS 43 (the fetch itself throws), then chr2:1
        return contigs, [ok("chr1", 3), zero("chr1", 43), ok("chr2", 1), zero("chr2", 70)], 1, abi.PS_THROW_REF_RANGE
    if where == "earlier-fault":                 # a record before it that the JVM dies on keeps its fault
        return contigs, [ok("chr1", 3), Record(0, "chrUn", 5, "8M", b"A" * 8, bytes([30]) * 8), zero("chr1", 39)], 1, None
    raise ValueError(where)


PAST_CASES = ["last-contig", "middle-contig", "further-out", "earlier-fault"]


@pytest.mark.parametrize("where", PAST_CASES)
def test_past_end_restatements_and_batches(where):
    """from_records marks the first such record and keeps it on its own contig; both restatements of every tool agree."""
    import oracle_lib
    contigs, recs, k, prof = past_end_case(where)
    ref = PackedReference.from_contigs(contigs)
    b = ReadBatch.from_records(recs, ref)
    g = po.Genome(dict(contigs))
    first = next(i for i, r in enumerate(recs) if r.cigar == "5S5I")
    assert b.past_end == first + 1
    ci = [n for n, _ in PAST].index(recs[first].rname)
    assert int(b.ref_start[first]) == int(ref.contig_off[ci + 1]) - 1
    track_fault = (abi.PS_FAULT_PAST_END if where != "earlier-fault" else abi.PS_THROW_REF_RANGE, k)
    with pytest.raises(to.TrackFault) as e:
        to.track(to_py(recs), g)
    assert (e.value.code, e.value.ordinal) == track_fault
    with pytest.raises(to.TrackFault) as e:
        to.track_cpp(ref, b)
    assert (e.value.code, e.value.ordinal) == track_fault
    with pytest.raises(oracle_lib.OracleFault) as e:
        oracle_lib.pileup(ref, b)
    assert (e.value.code, e.value.ordinal) == track_fault
    if where == "earlier-fault":
        with pytest.raises(po.ReferenceWouldThrow) as e:
            po.pileup(to_py(recs), g, po.SnpDb([]), 1)
        assert e.value.ordinal == k
        return
    with pytest.raises(po.PastContigEnd) as e:
        po.pileup(to_py(recs), g, po.SnpDb([]), 1)
    assert e.value.ordinal == k
    with pytest.raises(po.ReferenceWouldThrow) as e:
        po.profile(to_py(recs), g, 64)
    assert e.value.ordinal == k and ("empty" in e.value.what) == (prof == abi.PS_THROW_EMPTY_REF)
    with pytest.raises(oracle_lib.OracleFault) as e:
        oracle_lib.profile(ref, b, 64)
    assert (e.value.code, e.value.ordinal) == (prof, k)


def test_past_end_slices():
    from parasuite_b200.sharding import slice_batch
    contigs, recs, k, _ = past_end_case("further-out")
    ref = PackedReference.from_contigs(contigs)
    b = ReadBatch.from_records(recs, ref)
    assert slice_batch(b, 0, 4).past_end == 2 and slice_batch(b, 1, 4).past_end == 1
    assert slice_batch(b, 0, 1).past_end == 0 and slice_batch(b, 2, 4).past_end == 0


@pytest.mark.gpu
@pytest.mark.parametrize("where", PAST_CASES)
def test_past_end_every_tool(tmp_path, where):
    """Every tool, batch (host and device) and file: the same status and fault as the restatements."""
    from parasuite_b200.runtime import Context, DeviceBatch
    contigs, recs, k, prof = past_end_case(where)
    ref = PackedReference.from_contigs(contigs)
    b = ReadBatch.from_records(recs, ref)
    refused = (abi.PS_ERR_UNSUPPORTED, (abi.PS_FAULT_PAST_END, k))
    if where == "earlier-fault":
        refused = prof_want = (abi.PS_ERR_REFERENCE_WOULD_THROW, (abi.PS_THROW_REF_RANGE, k))
    else:
        prof_want = (abi.PS_ERR_REFERENCE_WOULD_THROW, (prof, k))

    def outcome(fn):
        with pytest.raises(abi.PsError) as e:
            fn()
        return e.value.status, tuple(e.value.fault)
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / "reads.bam")
    write_fasta(fa, contigs)
    write_bam(path, PAST, recs)
    c = Context(0)
    try:
        c.upload_reference(ref)
        for view in (b, DeviceBatch(b, "cuda:0")):
            assert outcome(lambda: c.track(view)) == refused
            assert outcome(lambda: c.pileup(view)) == refused
        assert outcome(lambda: c.profile(b, 64)) == prof_want
        c.load_fasta(fa)
        assert outcome(lambda: c.track_bam(path, str(tmp_path / "t"))) == refused
        assert outcome(lambda: c.pileup_bam(path)) == refused
        assert outcome(lambda: c.clust_bam(path, str(tmp_path / "clust"))) == refused
        assert outcome(lambda: c.profile_bam(path, 64)) == prof_want
    finally:
        c.close()


# ---- scale --------------------------------------------------------------------------------------------------------
def scale_records(n=1_000_000, seed=77):
    """n sorted records on three 4 Mb contigs: lengths 18-64, 5 % N-spliced (50 b - 50 kb), 2 % with I or D, both
    strands, read bases at random (T>C events wherever a C or G meets a reference T or A)."""
    rng = np.random.default_rng(seed)
    names, ln = ["chrA", "chrB", "chrC"], 4_000_000
    contigs = [(c, np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes()) for c in names]
    L = rng.integers(18, 65, n)
    kind = rng.random(n)
    gap = rng.integers(50, 50_001, n)
    a = (L * rng.uniform(0.2, 0.8, n)).astype(np.int64).clip(1, L - 2)
    cig = []
    for i in range(n):
        li, ai = int(L[i]), int(a[i])
        if kind[i] < 0.05:
            cig.append(f"{ai}M{int(gap[i])}N{li - ai}M")
        elif kind[i] < 0.06:
            cig.append(f"{ai}M1I{li - ai - 1}M")
        elif kind[i] < 0.07:
            cig.append(f"{ai}M2D{li - ai}M")
        else:
            cig.append(f"{li}M")
    span = np.array([ref_span(c) for c in cig])
    contig = rng.integers(0, 3, n)
    pos = rng.integers(1, ln - 60_000, n)
    order = np.lexsort((pos, contig))
    seqs = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(L.sum()))].tobytes()
    starts = np.concatenate(([0], np.cumsum(L)))
    rev = rng.random(n) < 0.5
    recs = [Record(16 if rev[i] else 0, names[contig[i]], int(pos[i]), cig[i], seqs[starts[i]:starts[i + 1]],
                   bytes([30]) * int(L[i])) for i in order]
    assert int(span.max()) < 60_000
    return contigs, recs


def render(res, names):
    """The three file texts of track_bam from a whole-input result (rows are maximal runs and sites in file order)."""
    runs = ["".join(f"{names[int(x['contig'])]}\t{int(x['start0'])}\t{int(x['end0'])}\t{int(x['cov'])}\n" for x in res[k])
            for k in ("runs_plus", "runs_minus")]
    sites = "".join(f"{names[int(x['contig'])]}\t{int(x['pos'])}\t{'+-'[int(x['strand'])]}\t{int(x['t2c'])}\t{int(x['cov'])}\n"
                    for x in res["sites"])
    return {"plus.bedGraph": runs[0], "minus.bedGraph": runs[1], "t2c.tsv": "chrom\tpos\tstrand\tt2c\tcoverage\n" + sites}


@pytest.mark.gpu
def test_million_ragged_records(ctx, tmp_path, monkeypatch):
    """1 M ragged, spliced, gapped records on three contigs: the batch against track_cpp, and the file tool at windows
    of 10^9, 65 536 and 4 093 records against the texts rendered from it."""
    from parasuite_b200.runtime import Context
    from test_gpu_track import _equal
    contigs, recs = scale_records()
    ref = PackedReference.from_contigs(contigs)
    batch = ReadBatch.from_records(recs, ref)
    exp = to.track_cpp(ref, batch)
    ctx.upload_reference(ref)
    _equal(ctx.track(batch), exp, "1M batch")
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / "reads.bam")
    write_fasta(fa, contigs)
    write_bam(path, [(n, len(s)) for n, s in contigs], recs)
    want = render(exp, [n for n, _ in contigs])
    c = Context(0)
    try:
        c.load_fasta(fa)
        for w in (10 ** 9, 65_536, 4_093):
            monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(w))
            c.track_bam(path, str(tmp_path / "o"))
            assert _texts(tmp_path / "o") == want, w
    finally:
        c.close()
