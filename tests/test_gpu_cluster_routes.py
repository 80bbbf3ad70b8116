"""The four routes of pl_cluster_kernel at their limits, against the oracle and against the route each cluster should
take.

For each cluster slot the kernel picks one of four ways to compute the same record and sites:
  1 block pass with shared tables: not slot 0, at most CB_CHUNK reads in the slot's read range (unkept reads included),
    every T>C position in the 64 positions from the opener's start, at most CB_SITES distinct positions;
  2 warp routine, ballot form: at most 32 reads in the slot, events less than PL_WINDOW positions apart;
  3 warp routine, streaming sweep over a ring of PL_RING positions;
  4 window loop, one pass per PL_WINDOW positions, when the sweep gives up (the first pending read does not fit the
    ring, or starts go backwards below the ring's first position).
The library counts its warp-routine work and prints it to stderr under PARASUITE_B200_DEBUG: (sweep entries, sweep
give-ups, window passes).  A slot with events adds (0, 0, 0) on routes 1 and 2, (1, 0, 0) on route 3 and
(1, 1, (ev_max - ev_min) // 128 + 1) on route 4; a slot without events adds nothing.

`Builder` lays out clusters on a reference it writes itself and records the route it meant each cluster to take;
`predict` restates the kernel's choice (and the sweep's ring) from the batch, the oracle's T>C masks and the oracle's
cluster slots.  test_model_agrees_with_builder (no GPU) holds the two together on every batch of this file; every GPU
case then asserts oracle parity and the predicted counters through every view that reaches a different instantiation
of pl_cluster_kernel<NW, MK>: host and device batches (NW = 0 .. 4 by the read length), the misaligned device view
(generic decode, NW = 0) and the pileup fed by the profile's mask words (MK)."""
import re
from dataclasses import dataclass, field

import numpy as np
import pytest

from parasuite_b200 import PackedReference, ReadBatch, Record, abi

CB_CHUNK, CB_SITES, PL_WINDOW, PL_RING = 1024, 6, 128, 256
NONE, BLOCK, BALLOT, SWEEP, WINDOWS = 0, 1, 2, 3, 4
ROUTE_NAMES = {NONE: "no events", BLOCK: "block pass", BALLOT: "ballot form", SWEEP: "sweep", WINDOWS: "window loop"}
CIGAR = re.compile(r"(\d+)([MIDNSHP=X])")


# ---- cluster builder ----------------------------------------------------------------------------------------------
class Builder:
    """Reads on one contig whose bases the builder writes: a read copies the reference, bar the positions where it is
    told to show a T>C (plus strand: reference T, read C; minus strand: reference A, read G in the forward view).  The
    reference base such an event needs is written into the contig when the batch is made."""

    def __init__(self, length=400_000, seed=1):
        rng = np.random.default_rng(seed)
        self.seq = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, length)].tobytes())
        self.reads = []          # (flag, pos, cigar, {read offset: base})
        self.intent = []         # (read index of the opener, route meant for its cluster)
        self.need = {}           # position -> reference base its events need
        self.t_end = 0           # running maximum end of the kept reads

    @staticmethod
    def blocks(start, cigar):
        """[(reference position, read offset)] of the aligned bases, in forward order."""
        out, rp, qp = [], start, 0
        for n, op in CIGAR.findall(cigar):
            n = int(n)
            if op in "M=X":
                out += [(rp + k, qp + k) for k in range(n)]
                rp += n; qp += n
            elif op in "SI":
                qp += n
            elif op in "DN":
                rp += n
        return out

    @staticmethod
    def index(start, rev, cigar, p):
        """Strand-oriented index of position p in the read, or None where the read does not align p."""
        b = Builder.blocks(start, cigar)
        j = next((k for k, (rp, _) in enumerate(b) if rp == p), None)
        return None if j is None else (len(b) - 1 - j if rev else j)

    def opens(self, route):
        self.intent.append((len(self.reads), route))

    def read(self, start, rev, cigar, events=()):
        b = self.blocks(start, cigar)
        at = dict(b)
        ev = {}
        for p in events:
            i = self.index(start, rev, cigar, p)
            assert i is not None and i < 51, (start, cigar, p, i)       # index 51 and up kills the JVM
            base = "A" if rev else "T"
            assert self.need.setdefault(p, base) == base, f"position {p} needs both strands' base"
            ev[at[p]] = "G" if rev else "C"
        ref_len = sum(int(n) for n, op in CIGAR.findall(cigar) if op in "MDN=X")
        self.reads.append((16 if rev else 0, start, cigar, ev))
        self.t_end = max(self.t_end, start + ref_len - 1)

    def unmapped(self, cigar):
        """A filler the pileup does not keep: unmapped (placed at the previous read, as mates are)."""
        self.reads.append((4, self.reads[-1][1], cigar, None))

    def skipped(self, cigar="10M2D5N26M"):
        """A filler the pileup skips: I or D together with N (skippedDueIndel)."""
        self.reads.append((0, self.reads[-1][1], cigar, None))

    def gap(self, n=20):
        """A start that opens a new cluster."""
        return self.t_end + n

    def make(self):
        seq = bytearray(self.seq)
        for p, base in self.need.items():
            seq[p - 1] = ord(base)
        recs = []
        for flag, pos, cigar, ev in self.reads:
            L = sum(int(n) for n, op in CIGAR.findall(cigar) if op in "MIS=X")
            if ev is None:
                s = bytearray(b"A" * L)
            else:
                s = bytearray(b"A" * L)
                for rp, qp in self.blocks(pos, cigar):
                    s[qp] = seq[rp - 1]
                for qp, base in ev.items():
                    s[qp] = ord(base)
            recs.append(Record(flag, "chr1", pos, cigar, bytes(s), bytes([30]) * L))
        ref = PackedReference.from_contigs([("chr1", bytes(seq))])
        return ref, ReadBatch.from_records(recs, ref)


def cluster(b, route, reads, sites, thin=3):
    """One cluster.  reads: (start, rev) or (start, rev, cigar), the opener first, or "U" / "S" for an unmapped / skipped
    filler; sites {position: strand}: a read of that strand that aligns the position at an index below 51 shows the
    T>C there, bar every `thin`-th such read (so that T>C counts stay below coverage).  Every site gets an event."""
    b.opens(route)
    got = dict.fromkeys(sites, 0)
    for k, rd in enumerate(reads):
        if rd in ("U", "S"):
            (b.unmapped if rd == "U" else b.skipped)(b.cigar if rd == "U" else "10M2D5N26M")
            continue
        start, rev = rd[0], rd[1]
        cigar = rd[2] if len(rd) > 2 else b.cigar
        ev = []
        for p, srev in sites.items():
            i = Builder.index(start, rev, cigar, p) if srev == rev else None
            if i is not None and i < 51 and (got[p] == 0 or (k + p) % thin):
                ev.append(p)
                got[p] += 1
        b.read(start, rev, cigar, ev)
    assert all(got.values()), got


def chain(base, n, span, opener_rev=False):
    """n reads whose starts run from base to base + span, strands alternating from the opener's; the first two and
    the last two share a start, so that both strands reach both ends."""
    st = np.round(np.linspace(base, base + span, n - 2)).astype(int)
    st = np.concatenate(([base], st, [base + span]))
    return [(int(s), bool(opener_rev) ^ (k % 2 == 1)) for k, s in enumerate(st)]


def new_builder(L, **kw):
    b = Builder(**kw)
    b.cigar = f"{L}M"
    return b


# ---- route model --------------------------------------------------------------------------------------------------
@dataclass
class Table:
    kept: list
    start: list
    lo: list
    hi: list
    rev: list
    pos: list = field(default_factory=list)       # event positions of every read


def read_table(ref, batch, masks):
    """Per read: kept, start, checkPosition interval (plus: [start, start + alen - 1], minus: [end - alen + 1, end]),
    strand and T>C positions (oracle masks: bit i = strand-oriented index i)."""
    n = batch.n_reads
    meta = np.asarray(batch.meta[:n]).astype(np.int64)
    flags, ncig = meta >> 24, (meta >> 16) & 0xFF
    off = np.concatenate(([0], np.cumsum(ncig)))
    cig = np.asarray(batch.cigar).astype(np.int64).tolist()
    g0 = np.asarray(batch.ref_start[:n]).astype(np.int64).tolist()
    coff = ref.contig_off.astype(np.int64)
    t = Table([], [], [], [], [])
    for r in range(n):
        ops = [(c & 15, c >> 4) for c in cig[off[r]:off[r + 1]]]
        has_id, has_n = any(o in (1, 2) for o, _ in ops), any(o == 3 for o, _ in ops)
        kept = not (int(flags[r]) & (abi.PS_RF_UNMAPPED | abi.PS_RF_POS_ZERO | abi.PS_RF_CIGAR_OVERFLOW)) \
            and not (has_id and has_n)
        R = sum(n_ for o, n_ in ops if o in (0, 2, 3, 7, 8))
        alen = sum(n_ for o, n_ in ops if o in (0, 7, 8))
        c = int(np.searchsorted(coff, g0[r], side="right")) - 1
        start = g0[r] - int(coff[c]) + 1
        end = start + R - 1
        rev = bool(int(flags[r]) & abi.PS_RF_REVERSE)
        lo, hi = (end - alen + 1, end) if rev else (start, start + alen - 1)
        m = int(masks[r]) if kept else 0
        idx = [i for i in range(64) if (m >> i) & 1]
        t.kept.append(kept); t.start.append(start); t.lo.append(lo); t.hi.append(hi); t.rev.append(rev)
        t.pos.append([hi - i if rev else lo + i for i in idx])
    return t


def key_set_fits(t, r, base):
    """t2c_positions: every T>C position of read r in [base, base + 64); a plus read also needs 0 <= lo - base <= 63
    (the shift), a minus read -63 <= hi - base - 63 <= 63."""
    if t.rev[r]:
        ok = -63 <= t.hi[r] - base - 63 <= 63
    else:
        ok = 0 <= t.lo[r] - base <= 63
    return ok and all(0 <= p - base <= 63 for p in t.pos[r])


def sweep_gives_up(t, f, fe):
    """The sweep's loop over batches of 32 reads of [f, fe): pending reads, the ring's first position wlo, the fit
    test of the first pending read and the deferral of the reads from the first misfit on."""
    started, wlo = False, 0
    for q in range(f, fe, 32):
        pending = [r for r in range(q, min(q + 32, fe)) if t.kept[r]]
        while pending:
            bstart = min(t.start[r] for r in pending)
            if not started:
                wlo, started = bstart, True
            if bstart < wlo:
                return True                               # starts went backwards
            wlo = bstart
            fits = [t.hi[r] + 2 - wlo <= PL_RING and t.lo[r] >= wlo for r in pending]
            if not fits[0]:
                return True                               # the first pending read does not fit the ring
            pending = pending[fits.index(False):] if False in fits else []
    return False


def slot_route(t, slot, f, fe):
    """(route, counters added, site slots reserved) of the slot holding reads [f, fe)."""
    pos = [p for r in range(f, fe) if t.kept[r] for p in t.pos[r]]
    if not pos:
        return NONE, (0, 0, 0), 0
    if slot != 0 and fe - f <= CB_CHUNK:
        base = t.start[f]                                 # the opener
        keys = set(pos)
        if all(key_set_fits(t, r, base) for r in range(f, fe) if t.kept[r] and t.pos[r]) and len(keys) <= CB_SITES:
            return BLOCK, (0, 0, 0), len(keys)
    lo, hi = min(pos), max(pos)
    reserved = min(len(pos), hi - lo + 1)
    if fe - f <= 32 and hi - lo < PL_WINDOW:
        return BALLOT, (0, 0, 0), reserved
    if not sweep_gives_up(t, f, fe):
        return SWEEP, (1, 0, 0), reserved
    return WINDOWS, (1, 1, (hi - lo) // PL_WINDOW + 1), reserved


def slot_starts(exp):
    """First reads of the oracle's clusters (slots 1 ..), the open one included."""
    f = [int(x) for x in exp["clusters"]["first_read"]]
    return f + ([int(exp["open_cluster"]["first_read"])] if exp["open_cluster"] is not None else [])


def predict(t, firsts, a, b):
    """Routes of the slots of the call over reads [a, b) of the table (a shard, or the whole batch), the counters the
    call must print and the site slots it reserves.  Slot 0 holds the reads in front of the first opener."""
    bounds = [a] + [f for f in firsts if a <= f < b] + [b]
    routes, dbg, reserved = [], [0, 0, 0], 0
    for s in range(len(bounds) - 1):
        route, add, res = slot_route(t, s, bounds[s], bounds[s + 1])
        routes.append((bounds[s], route))
        dbg = [x + y for x, y in zip(dbg, add)]
        reserved += res
    return routes, tuple(dbg), reserved


# ---- cases ----------------------------------------------------------------------------------------------------------
UNIFORM_LENGTHS = [16, 17, 36, 51, 64]          # NW = 1, 2, 3, 4, 4; at 64 events stay below index 51
SITE_OFFSETS = [0, 63, 30, 10, 50, 20, 40]      # bit 0 and bit 63 of the key set first


def site_strands(base, offsets, opener_rev, L):
    """{position: strand} of sites at base + offsets: the opener's strand first, then alternating.  Reads start at base
    or later, so a minus read longer than 51 holds base + o at an index of at least L - 1 - o: plus there below o = 13."""
    return {base + o: False if L > 51 and o < 13 else bool(opener_rev) ^ (j % 2 == 1) for j, o in enumerate(offsets)}


def case_distinct_sites(L):
    """(a) 1 .. 7 distinct T>C positions, 40 reads each, plus and minus openers: 6 take the block pass, 7 the sweep."""
    b = new_builder(L)
    base = 1000
    span = max(64 - L, 16)           # the last reads reach base + 63; at L = 64 plus reads reach it below index 51
    for opener_rev in (False, True):
        for k in range(1, 8):
            cluster(b, BLOCK if k <= CB_SITES else SWEEP, chain(base, 40, span, opener_rev),
                    site_strands(base, SITE_OFFSETS[:k], opener_rev, L))
            base = b.gap()
    return b


def case_key_span(L, generic=False):
    """(b) The farthest event at base + 63 (block pass) or base + 64 (falls back), from plus reads (a plus read starting
    right there, and one 13 bases before it) and from minus reads (hi - ib with ib = 0 and ib = 13), under plus and minus
    openers.  The generic variant adds a minus read aligned on one base at the opener's start (d = -63) to every
    cluster, and a cluster whose only stray event comes from a minus read with hi = base + 126 (d = 63)."""
    b = new_builder(L)
    base = 1000
    for opener_rev in (False, True):
        for src_rev in (False, True):
            for far in (63, 64):
                p = base + far
                specials = [(p, False), (p - 13, False)] if not src_rev else [(p - L + 1, True), (p + 13 - L + 1, True)]
                reach = max(s + L - 1 for s, _ in specials)
                reads = chain(base, 40, max(16, reach + 6 - L - base), opener_rev)
                sites = {base + 20: opener_rev, p: src_rev}
                if generic:
                    reads.append((base, True, f"{L - 1}S1M"))
                    sites[base] = True
                    if base + 20 in sites and opener_rev:
                        sites[base + 20] = True
                reads = reads[:1] + sorted(reads[1:] + specials, key=lambda x: x[0])
                cluster(b, BLOCK if far == 63 else SWEEP, reads, sites, thin=1000)
                base = b.gap()
    if generic:
        reads = chain(base, 40, 111, False) + [(base + 126 - L + 1, True)]
        cluster(b, SWEEP, sorted(reads, key=lambda x: x[0]), {base + 5: False, base + 126: True}, thin=1000)
    return b


def small(b, n=3, sites=1):
    """A small block-pass cluster at the next free start."""
    base = b.gap()
    cluster(b, BLOCK, chain(base, max(n, 4), 4), {base + 2 + 3 * k: k % 2 == 1 for k in range(sites)})


def big(b, n, route, fillers=(), span=20, sites=3):
    """n reads in the slot's read range (fillers at the given read ranks count among them) over `span` positions."""
    base = b.gap()
    kept = chain(base, n - len(fillers), span)
    reads = []
    for rd in kept:
        while len(reads) in fillers:
            reads.append("U" if len(reads) % 2 else b.filler)
        reads.append(rd)
    cluster(b, route, reads, {base + 3 + 7 * k: k % 2 == 1 for k in range(sites)})


def case_reads_per_slot(L, generic=False):
    """(c) 1024 reads (block pass), with fillers among them too; 1025 reads in the middle of a block (ncomp == 0, the
    sweep); two groups of 512 overlapping by 5 (one 1024-read cluster) or by 4 (two clusters); four clusters of 256
    filling one chunk, clusters of 257 crossing chunk edges.  The generic variant's fillers are skipped reads."""
    b = new_builder(L)
    b.filler = "S" if generic else "U"
    big(b, 1024, BLOCK)
    big(b, 1024, BLOCK, fillers=set(range(100, 1024, 9)))
    for _ in range(10):
        small(b)
    big(b, 1025, SWEEP)
    big(b, 1025, SWEEP, fillers=set(range(5, 1025, 50)))
    for _ in range(10):
        small(b)
    for overlap in (5, 4):
        base = b.gap()
        a = [(base, k % 2 == 1) for k in range(512)]
        nxt = base + L - 1 - overlap
        bb = [(nxt, k % 2 == 0) for k in range(512)]
        sites = {base + 2: False, nxt + L - 3: True}
        if overlap == 5:
            cluster(b, BLOCK, a + bb, sites)
        else:
            cluster(b, BLOCK, a, {base + 2: False})
            cluster(b, BLOCK, bb, {nxt + L - 3: True})
    for n in (256, 256, 256, 256, 257, 257, 257, 257, 257):
        big(b, n, BLOCK)
    return b


def case_block_edges():
    """(c) 64 * 3 + 1 slots (slot 0 is empty): clusters the block pass cannot take at the first and the last slot of
    every block of pl_cluster_kernel -- 63, 64, 127, 128, 191, 192 -- sweep and ballot form alternately."""
    b = new_builder(17)
    b.filler = "U"
    for slot in range(1, 193):
        if slot in (63, 128, 192):
            base = b.gap()
            cluster(b, SWEEP, chain(base, 40, 40), {base + 7 * k: k % 2 == 1 for k in range(7)})
        elif slot in (64, 127, 191):
            base = b.gap()
            cluster(b, BALLOT, chain(base, 8, 30), {base + 5 * k: k % 2 == 1 for k in range(7)})
        else:
            small(b, n=4, sites=1 + slot % 3)
    return b


def case_ballot_vs_sweep(L, generic=False):
    """(d) 7 sites in a slot of 32 reads (the ballot form) or 33 (the sweep), fillers counted; events 127 positions
    apart (ballot form) or 128 (the sweep), in 28 reads and 2 fillers.  One site sits at the end of the last reads (pos == hi)."""
    b = new_builder(L)
    filler = "S" if generic else "U"
    span = max(64 - L, 16)
    for n, route in ((32, BALLOT), (33, SWEEP)):
        for opener_rev in (False, True):
            base = b.gap()
            reads = chain(base, n - 4, span, opener_rev)
            reads = reads[:3] + [filler, "U"] + reads[3:10] + [filler, "U"] + reads[10:]
            cluster(b, route, reads, site_strands(base, SITE_OFFSETS, opener_rev, L))
    for apart, route in ((127, BALLOT), (128, SWEEP)):
        for opener_rev in (False, True):
            base = b.gap()
            reads = chain(base, 28, apart + 1 - L + 12, opener_rev) + [filler, "U"]
            far = base + apart
            cluster(b, route, reads, {base + 1: False, far: True} if L > 51 else {base: opener_rev, far: True})
    return b


def case_sweep(L):
    """(e) One chain of reads over more than 10 x 256 positions (the ring wraps again and again), events at the ring's
    slot edges 0 / 255 and a few in between."""
    b = new_builder(L)
    base, span = 2048, 11 * 256 + 8
    sites = {}
    for k in range(11):
        for o in (0, 255, 128):
            sites[base + 256 * k + o] = (k + o) % 2 == 1
    cluster(b, SWEEP, chain(base, span // 4, span, False), sites, thin=2)
    return b


def case_ring_fit():
    """(e) The first pending read against the ring: a plus read of alen 255 fits, 256 misses by one; a minus read of
    reference span R = 255 (20M215N20M) fits, R = 256 misses; a read that does not fit behind the first pending one is
    deferred and taken after the flush.  A miss gives up into the window loop."""
    b = new_builder(36)
    for alen, route in ((255, SWEEP), (256, WINDOWS)):
        base = b.gap()
        reads = [(base, False, f"{alen}M")] + chain(base + 4, 39, 150)
        cluster(b, route, sorted(reads, key=lambda x: x[0]), {base + 3: False, base + 40: True, base + 150: False})
    for R, route in ((255, SWEEP), (256, WINDOWS)):
        base = b.gap()
        opener = (base, True, f"20M{R - 40}N20M")
        reads = [opener] + chain(base + 2, 39, 200)
        cluster(b, route, sorted(reads, key=lambda x: x[0]), {base + R - 1: True, base + R - 10: True,
                                                              base + 30: False})
    # deferral: the second read of the first batch reaches 261 - 10 positions past the ring's start
    base = b.gap()
    reads = [(base, False), (base + 10, False, "250M")] + chain(base + 12, 38, 200)
    cluster(b, SWEEP, sorted(reads, key=lambda x: x[0]), {base + 2: False, base + 50: False, base + 230: True})
    return b


def case_window_loop(generic):
    """(f) Give-up clusters with events 127, 128, 255 and 256 apart (1, 2, 2, 3 window passes), with events at
    w0 + 127 and w0 + 128.  Generic: the give-up comes from an opener of alen 256 that starts before each window and
    ends after it.  Uniform (36M): from a read at rank 32 that starts before the first read of its slot (starts go
    backwards); two more clusters go backwards without a give-up -- inside one batch of 32, and across batches but not
    below the ring's first position."""
    b = new_builder(36)
    for span in (127, 128, 255, 256):
        base = b.gap()
        if generic:
            reads = [(base, False, "256M")] + chain(base + 3, 45, span + 5, True)
        else:
            ch = chain(base + 4, 45, span + 5, True)
            reads = ch[:32] + [(base, False)] + ch[32:]
        sites = {base + 4: True, base + 4 + span: False}
        if span >= 128:
            sites.update({base + 4 + 127: True, base + 4 + 128: False})
        cluster(b, WINDOWS, reads, sites, thin=4)
    if not generic:
        base = b.gap()
        ch = chain(base + 4, 45, 100)
        cluster(b, SWEEP, ch[:20] + [(base, True)] + ch[20:], {base + 4: False, base + 90: True})
        base = b.gap()
        ch = chain(base, 45, 100)         # the first batch's first start is base; rank 32 starts above it
        cluster(b, SWEEP, ch[:32] + [(base + 2, True)] + ch[32:], {base + 3: False, base + 90: True})
    return b


def case_shard_cuts():
    """(g) Small clusters around a route-1-shaped cluster (100 reads, 3 sites), a 7-site cluster (100 reads) and a
    1025-read cluster; the tests cut the batch inside each of the three."""
    b = new_builder(36)
    b.filler = "U"
    for _ in range(5):
        small(b)
    big(b, 100, BLOCK)
    for _ in range(5):
        small(b)
    big(b, 100, SWEEP, sites=7, span=28)
    for _ in range(5):
        small(b)
    big(b, 1025, SWEEP)
    for _ in range(5):
        small(b)
    return b


def case_site_capacity():
    """(h) 5310 reads dense in T>C: 150 seven-site clusters of 33 reads whose events spread over 61 positions (the warp
    routine reserves min(t2c, ev_max - ev_min + 1) slots each) and 30 block-pass clusters of 6 sites."""
    b = new_builder(36)
    for k in range(150):
        base = b.gap()
        cluster(b, SWEEP, chain(base, 33, 28), {base + o: j % 2 == 1 for j, o in enumerate((0, 10, 20, 30, 40, 50, 60))},
                thin=1000)
        if k % 5 == 0:
            base = b.gap()
            cluster(b, BLOCK, chain(base, 12, 20), {base + o: j % 2 == 1 for j, o in enumerate((0, 4, 8, 20, 30, 40))},
                    thin=1000)
    return b


CASES = {}
for _L in UNIFORM_LENGTHS:
    CASES[f"a-distinct-sites-L{_L}"] = (case_distinct_sites, _L)
for _L in (16, 36, 64):
    CASES[f"b-key-span-L{_L}"] = (case_key_span, _L)
CASES["b-key-span-generic"] = (case_key_span, 16, True)
CASES["c-reads-per-slot-L36"] = (case_reads_per_slot, 36)
CASES["c-reads-per-slot-generic"] = (case_reads_per_slot, 36, True)
CASES["c-block-edges-L17"] = (case_block_edges,)
for _L in (17, 51):
    CASES[f"d-ballot-vs-sweep-L{_L}"] = (case_ballot_vs_sweep, _L)
CASES["d-ballot-vs-sweep-generic"] = (case_ballot_vs_sweep, 36, True)
for _L in (36, 64):
    CASES[f"e-sweep-chain-L{_L}"] = (case_sweep, _L)
CASES["e-ring-fit"] = (case_ring_fit,)
CASES["f-window-loop-L36"] = (case_window_loop, False)
CASES["f-window-loop-generic"] = (case_window_loop, True)
CASES["g-shard-cuts"] = (case_shard_cuts,)
CASES["h-site-capacity"] = (case_site_capacity,)

_MADE = {}


def make_case(name):
    """(ref, batch, builder) of a case, made once per session."""
    if name not in _MADE:
        fn, *args = CASES[name]
        b = fn(*args)
        _MADE[name] = (*b.make(), b)
    return _MADE[name]


def model(oracle, ref, batch, exp):
    return read_table(ref, batch, oracle.read_t2c_masks(ref, batch)), slot_starts(exp)


# ---- the model against the builder (no GPU) -------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_model_agrees_with_builder(oracle, name):
    """Every cluster the builder laid out opens where it meant (the oracle's slots) and the model sends it down the
    route the builder meant; the whole file reaches every route."""
    ref, batch, b = make_case(name)
    exp = oracle.pileup(ref, batch)
    t, firsts = model(oracle, ref, batch, exp)
    routes, dbg, reserved = predict(t, firsts, 0, batch.n_reads)
    assert routes[0] == (0, NONE)                      # nothing in front of the first opener
    got = routes[1:]
    assert [f for f, _ in got] == [f for f, _ in b.intent], f"{name}: clusters open elsewhere than laid out"
    wrong = [(f, ROUTE_NAMES[r], ROUTE_NAMES[w]) for (f, r), (_, w) in zip(got, b.intent) if r != w]
    assert not wrong, f"{name}: (opener, model, builder) {wrong[:5]}"
    if name == "h-site-capacity":
        assert reserved > max(1024, batch.n_reads // 4), reserved


def test_every_route_is_reached():
    seen = {route for name in CASES for _, route in make_case(name)[2].intent}
    assert seen == {BLOCK, BALLOT, SWEEP, WINDOWS}


# ---- running on the GPU -------------------------------------------------------------------------------------------
DEBUG_LINE = re.compile(r"\[ps_pileup\] warp-routine site passes (\d+), sweep give-ups (\d+), window passes (\d+)")


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture
def debug(monkeypatch, capfd):
    """debug(fn): fn() and the counters the one pileup call inside it printed (PARASUITE_B200_DEBUG is looked up on
    every call)."""
    monkeypatch.setenv("PARASUITE_B200_DEBUG", "1")

    def run(fn):
        capfd.readouterr()
        out = fn()
        lines = DEBUG_LINE.findall(capfd.readouterr().err)
        assert len(lines) == 1, lines
        return out, tuple(int(x) for x in lines[0])
    return run


def mask_fed(ctx, batch, carry=None):
    """The profile with mask words, then the pileup fed by them (pl_cluster_kernel<NW, true>)."""
    import torch
    from parasuite_b200.runtime import DeviceBatch
    d = DeviceBatch(batch, "cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    ctx.profile_begin(max(51, batch.uniform_len), emit_t2c_masks=True)
    ctx.profile_batch_device(d, st)
    masks = ctx.profile_masks()
    assert masks is not None
    with ctx.pileup_run(d, carry=carry, stream=st, masks=masks) as h:
        pile = h.fetch()
    ctx.profile_end()
    return pile


def views(ctx, batch, carry=None):
    from parasuite_b200.runtime import DeviceBatch
    from test_gpu_bitparallel_edges import misaligned
    out = [("host", lambda: ctx.pileup(batch, carry=carry)),
           ("device", lambda: ctx.pileup(DeviceBatch(batch, "cuda:0"), carry=carry)),
           ("misaligned", lambda: ctx.pileup(misaligned(batch), carry=carry))]
    if batch.uniform_ncigar == 1 and 1 <= batch.uniform_len <= 62:     # longer reads get no mask words
        out.append(("mask-fed", lambda: mask_fed(ctx, batch, carry)))
    return out


def check_views(ctx, debug, batch, exp, want, what, carry=None):
    from test_gpu_pileup import assert_pileup_equal
    for how, run in views(ctx, batch, carry):
        got, printed = debug(run)
        assert_pileup_equal(got, exp, f"{what} {how}")
        assert printed == want, (what, how, printed, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in CASES if n[0] in "abcdef"])
def test_routes(ctx, oracle, debug, name):
    """(a) - (f): every view against the oracle, and the counters the model predicts."""
    ref, batch, _ = make_case(name)
    exp = oracle.pileup(ref, batch)
    t, firsts = model(oracle, ref, batch, exp)
    _, want, _ = predict(t, firsts, 0, batch.n_reads)
    ctx.upload_reference(ref)
    check_views(ctx, debug, batch, exp, want, name)


def big_openers(b, at_least=100):
    """(opener, reads in the slot) of the builder's clusters of at least `at_least` reads, in batch order."""
    firsts = [f for f, _ in b.intent] + [len(b.reads)]
    return [(f, e - f) for f, e in zip(firsts[:-1], firsts[1:]) if e - f >= at_least]


@pytest.mark.gpu
@pytest.mark.parametrize("which,into", [(0, 40), (1, 40), (2, 500)], ids=["block-shaped", "seven-sites", "1025-reads"])
def test_slot_zero_after_a_cut(ctx, oracle, debug, which, into):
    """(g) Two shards cut `into` reads inside a cluster: the second shard's head slot (slot 0, the reads that continue the
    first shard's open cluster) goes to the warp routine whatever its shape, the first shard's open part takes its own
    route; merged, the shards give the whole stream."""
    from parasuite_b200.sharding import merge_pileup_shards, slice_batch
    from test_gpu_pileup import assert_pileup_equal
    ref, batch, b = make_case("g-shard-cuts")
    whole = oracle.pileup(ref, batch)
    t, firsts = model(oracle, ref, batch, whole)
    opener, size = big_openers(b)[which]
    cut = opener + into
    parts = [(0, cut), (cut, batch.n_reads)]
    shards = [slice_batch(batch, lo, hi) for lo, hi in parts]
    plans = [predict(t, firsts, lo, hi) for lo, hi in parts]
    assert plans[1][0][0] == (cut, SWEEP), plans[1][0][0]            # the head slot: more than 32 reads, events
    ctx.upload_reference(ref)
    for how, _ in views(ctx, shards[0]):
        results, carry = [], None
        for shard, (routes, want, _) in zip(shards, plans):
            got, printed = debug(dict(views(ctx, shard, carry))[how])
            assert printed == want, (which, how, printed, want)
            results.append(got)
            carry = merge_pileup_shards.carry_after(results, carry)
        assert_pileup_equal(merge_pileup_shards(results, [0, cut]), whole, f"cut {cut} ({size}-read cluster) {how}")


@pytest.mark.gpu
def test_site_capacity_retry(oracle, debug):
    """(h) A fresh context and a batch whose reserved site slots (the block pass: its sites; the warp routine:
    min(t2c, ev_max - ev_min + 1)) exceed the first-guess capacity max(1024, n / 4): the call runs again with room for
    them and equals the oracle; the next calls on the context too."""
    from parasuite_b200.runtime import Context, DeviceBatch
    from test_gpu_pileup import assert_pileup_equal
    ref, batch, _ = make_case("h-site-capacity")
    exp = oracle.pileup(ref, batch)
    t, firsts = model(oracle, ref, batch, exp)
    _, want, reserved = predict(t, firsts, 0, batch.n_reads)
    assert reserved > max(1024, batch.n_reads // 4) > len(exp["sites"]), (reserved, len(exp["sites"]))
    fresh = Context(0)
    try:
        fresh.upload_reference(ref)
        for what, run in (("first call", lambda: fresh.pileup(batch)), ("second call", lambda: fresh.pileup(batch)),
                          ("device", lambda: fresh.pileup(DeviceBatch(batch, "cuda:0")))):
            got, printed = debug(run)
            assert_pileup_equal(got, exp, f"site capacity {what}")
            assert printed == want, (what, printed, want)
    finally:
        fresh.close()
