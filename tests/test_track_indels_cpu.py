"""CPU: the track's per-position deletion and insertion counts (ps_track_indel_opts.indel_counts).  The Python and C++
restatements against each other on random records of every CIGAR kind under several thresholds, hand-derived rows for
single records, the invariants that tie the totals to the rows, the contig end, the struct layouts and the keywords of
the Python binding."""
import ctypes as C
import random

import numpy as np
import pytest

import py_oracle as po
import track_indels_oracle as ti
import track_oracle as to
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi
from parasuite_b200.runtime import track_indel_opts

# (min_depth, min_events)
SETTINGS = [(1, 1), (0, 0), (3, 1), (1, 2), (8, 3), (10 ** 6, 1)]


def indel_cigar(rng: random.Random):
    """A CIGAR rich in indels: leading H / S / I / D, runs of I and D, I right after D, zero-length ops, =/X blocks,
    trailing D and I.  Returns (text, read length)."""
    ops = []
    if rng.random() < 0.1:
        ops.append(("H", rng.randint(1, 4)))
    if rng.random() < 0.25:
        ops.append(("S", rng.randint(1, 4)))
    if rng.random() < 0.12:
        ops.append(("I", rng.randint(1, 3)))        # no anchor
    if rng.random() < 0.08:
        ops.append(("D", rng.randint(1, 4)))        # the read starts with a deletion
    for _ in range(rng.randint(1, 4)):
        ops.append((rng.choice("MMM=X"), rng.randint(1, 30)))
        r = rng.random()
        if r < 0.22:
            ops.append(("I", rng.randint(1, 5)))
        elif r < 0.44:
            ops.append(("D", rng.randint(1, 8)))
        elif r < 0.50:
            ops.append(("D", rng.randint(1, 3)))
            ops.append(("I", rng.randint(1, 3)))    # anchored on the deleted base
        elif r < 0.55:
            ops.append(("I", rng.randint(1, 3)))
            ops.append(("I", rng.randint(1, 3)))    # two events, one anchor
        elif r < 0.60:
            ops.append((rng.choice("ID"), 0))
    ops.append((rng.choice("MM=X"), rng.randint(1, 20)))
    r = rng.random()
    if r < 0.08:
        ops.append(("D", rng.randint(1, 5)))
    elif r < 0.16:
        ops.append(("I", rng.randint(1, 4)))
    if rng.random() < 0.2:
        ops.append(("S", rng.randint(1, 4)))
    if rng.random() < 0.05:
        ops.append(("H", 2))
    L = sum(n for op, n in ops if op in "MIS=X")
    return "".join(f"{n}{op}" for op, n in ops), L


def indel_records(rng: random.Random, contigs, n, err=0.05, splice_frac=0.05):
    """n sorted records with indel_cigar CIGARs (a few with N, some of those also with an indel: skipped), bases from
    the reference with errors, on both strands"""
    recs = []
    for _ in range(n):
        name, seq = contigs[rng.randrange(len(contigs))]
        if rng.random() < splice_frac:
            a, b = rng.randint(5, 20), rng.randint(5, 20)
            text, L = (f"{a}M{rng.randint(1, 40)}N{b}M", a + b) if rng.random() < 0.5 else \
                (f"{a}M1I{rng.randint(1, 40)}N{b}M", a + b + 1)
        else:
            text, L = indel_cigar(rng)
        span = sum(k for op, k in po.parse_cigar(text) if op in "MDN=X")
        if span + 2 >= len(seq):
            continue
        pos = rng.randint(1, len(seq) - span)
        rd = bytearray()
        rf = pos
        for op, k in po.parse_cigar(text):
            if op in "M=X":
                for j in range(k):
                    b = seq[rf - 1 + j]
                    b = b if b in b"ACGT" else ord("ACGT"[j % 4])
                    rd.append(rng.choice(b"ACGT") if rng.random() < err else (b & ~0x20 if b >= 97 else b))
                rf += k
            elif op in "IS":
                rd += bytes(rng.choice(b"ACGT") for _ in range(k))
            elif op in "DN":
                rf += k
        assert len(rd) == L
        recs.append(Record(16 if rng.random() < 0.5 else 0, name, pos, text, bytes(rd), bytes([30] * L)))
    order = {c: i for i, (c, _) in enumerate(contigs)}
    recs.sort(key=lambda r: (order[r.rname], r.pos))
    return recs


def clean(recs, contigs, order=None):
    """drop the records the track faults on (order: the contig order the records follow, default the genome's)"""
    g = po.Genome(dict(contigs))
    while True:
        try:
            to.track(to_py(recs), g, order)
            return recs
        except to.TrackFault as e:
            recs = recs[:e.ordinal] + recs[e.ordinal + 1:]


def span_past_end_allowed(batch):
    """The batch with PS_RF_REF_RANGE cleared on every record.  Both producers set it for a record whose reference span
    runs past its contig's end (htsjdk's fetch of the whole span would throw), so the track faults on such a record; a
    batch made otherwise reaches the track with the flag clear, and its D ops can then run past the contig's end while
    every alignment block stays on the contig.  The Python restatement checks the blocks only, like the track."""
    meta = np.asarray(batch.meta)
    meta &= np.uint32(~(abi.PS_RF_REF_RANGE << 24) & 0xFFFFFFFF)
    return batch


def rows_of(cpp, names):
    """indel rows of track_indels_cpp as the Python restatement's tuples"""
    return [(names[int(x["contig"])], int(x["pos"]), "+-"[int(x["strand"])], "ACGTN"[int(x["ref"])], int(x["cov"]),
             int(x["del"]), int(x["ins"])) for x in cpp["indel_rows"]]


def _case(seed):
    rng = random.Random(9900 + seed)
    contigs = random_genome(rng, n_contigs=3, length=600, n_frac=0.05, lower_frac=0.2)
    recs = indel_records(rng, contigs, 400)
    recs += random_records(rng, contigs, 200, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 90),
                           err=0.08, flags_special=0.05)
    order = {c: i for i, (c, _) in enumerate(contigs)}
    recs = [r for r in recs if r.pos > 0 or r.flag & 4]
    recs.sort(key=lambda r: (order.get(r.rname, 99), r.pos))
    recs = clean(recs, contigs)
    return contigs, po.Genome(dict(contigs)), PackedReference.from_contigs(contigs), recs


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("setting", range(len(SETTINGS)))
def test_python_and_cpp_restatements_agree(seed, setting):
    md, me = SETTINGS[setting]
    contigs, g, ref, recs = _case(seed)
    names = [c for c, _ in contigs]
    py = ti.track_indels(to_py(recs), g, min_depth=md, min_events=me)
    cpp = ti.track_indels_cpp(ref, ReadBatch.from_records(recs, ref), min_depth=md, min_events=me)
    assert rows_of(cpp, names) == py["indel_rows"]
    assert cpp["indel_totals"] == py["indel_totals"]
    assert ti.HEADER + "".join("\t".join(map(str, r)) + "\n" for r in rows_of(cpp, names)) == py["files"]["indels.tsv"]
    plain = to.track_cpp(ref, ReadBatch.from_records(recs, ref))
    for k in ("runs_plus", "runs_minus", "sites"):
        assert np.array_equal(plain[k], cpp[k]), k
    assert plain["counters"] == cpp["counters"]
    if setting == 0:
        assert len(py["indel_rows"]) > 50 and min(py["indel_totals"]["unanchored_insertions"]) > 0
    if md == 10 ** 6:
        assert py["indel_rows"] == []


@pytest.mark.parametrize("seed", range(4))
def test_invariants(seed):
    contigs, g, ref, recs = _case(seed)
    cpp = ti.track_indels_cpp(ref, ReadBatch.from_records(recs, ref))
    tot, rows = cpp["indel_totals"], cpp["indel_rows"]
    for s in (0, 1):
        r = rows[rows["strand"] == s]
        assert int(r["del"].sum()) == tot["deleted_bases"][s]
        assert int(r["ins"].sum()) == tot["insertion_ops"][s] - tot["unanchored_insertions"][s]
        assert tot["deletion_ops"][s] <= tot["deleted_bases"][s] and tot["insertion_ops"][s] <= tot["inserted_bases"][s]
    assert ((rows["del"] + rows["ins"]) > 0).all()
    # the coverage of a row is the strand's coverage there
    cov = {}
    for s, name in ((0, "runs_plus"), (1, "runs_minus")):
        for r in cpp[name]:
            for p in range(int(r["start0"]), int(r["end0"])):
                cov[(int(r["contig"]), p + 1, s)] = int(r["cov"])
    assert all(cov.get((int(x["contig"]), int(x["pos"]), int(x["strand"])), 0) == int(x["cov"]) for x in rows)
    # thresholds only remove rows
    full = set(map(tuple, rows_of(cpp, [c for c, _ in contigs])))
    for md, me in SETTINGS:
        sub = ti.track_indels(to_py(recs), g, min_depth=md, min_events=me)["indel_rows"]
        assert set(sub) <= full
        assert all(r[5] + r[6] >= max(1, me) and r[4] + r[5] >= max(1, md) for r in sub)
        assert sub == [r for r in rows_of(cpp, [c for c, _ in contigs]) if r[5] + r[6] >= max(1, me) and
                       r[4] + r[5] >= max(1, md)]


# ---- hand-derived rows --------------------------------------------------------------------------------------------
SEQ = b"ACGTTGCAAC" b"GGTACCATGA" b"NCTAGGATCC" b"TTAGCAGTCA"      # 40 bases, position 21 is N
ZERO = {k: [0, 0] for k in ti.TOTALS}


def _one(cigar, pos=1, flag=0, **kw):
    """one record on chr1 = SEQ through both restatements: (rows, totals)"""
    contigs = [("chr1", SEQ), ("chr2", b"ACGT" * 10)]
    L = sum(n for op, n in po.parse_cigar(cigar) if op in "MIS=X")
    rec = Record(flag, "chr1", pos, cigar, b"A" * L, bytes([30] * L))
    ref = PackedReference.from_contigs(contigs)
    py = ti.track_indels(to_py([rec]), po.Genome(dict(contigs)), **kw)
    cpp = ti.track_indels_cpp(ref, span_past_end_allowed(ReadBatch.from_records([rec], ref)), **kw)
    assert rows_of(cpp, ["chr1", "chr2"]) == py["indel_rows"]
    assert cpp["indel_totals"] == py["indel_totals"]
    return py["indel_rows"], py["indel_totals"]


def _tot(**kw):
    t = {k: list(v) for k, v in ZERO.items()}
    for k, v in kw.items():
        t[k] = v
    return t


HAND = [
    # cigar, pos, flag, rows, totals (n_rows added)
    ("3M2D3M", 1, 0, [("chr1", 4, "+", "T", 0, 1, 0), ("chr1", 5, "+", "T", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[2, 0])),
    ("3M2I3M", 1, 0, [("chr1", 3, "+", "G", 1, 0, 1)], _tot(insertion_ops=[1, 0], inserted_bases=[2, 0])),
    ("2S3I5M", 1, 0, [], _tot(insertion_ops=[1, 0], inserted_bases=[3, 0], unanchored_insertions=[1, 0])),
    ("3I5M", 4, 0, [], _tot(insertion_ops=[1, 0], inserted_bases=[3, 0], unanchored_insertions=[1, 0])),
    ("2H2S3I5M", 4, 0, [], _tot(insertion_ops=[1, 0], inserted_bases=[3, 0], unanchored_insertions=[1, 0])),
    ("2D4M", 1, 0, [("chr1", 1, "+", "A", 0, 1, 0), ("chr1", 2, "+", "C", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[2, 0])),
    ("4M2D", 1, 0, [("chr1", 5, "+", "T", 0, 1, 0), ("chr1", 6, "+", "G", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[2, 0])),
    ("3M1D2I3M", 1, 0, [("chr1", 4, "+", "T", 0, 1, 1)],
     _tot(deletion_ops=[1, 0], deleted_bases=[1, 0], insertion_ops=[1, 0], inserted_bases=[2, 0])),
    ("3M3I2I3M", 1, 0, [("chr1", 3, "+", "G", 1, 0, 2)], _tot(insertion_ops=[2, 0], inserted_bases=[5, 0])),
    ("3M0D0I3M", 1, 0, [], _tot()),
    ("3M0I2D0D3M", 1, 0, [("chr1", 4, "+", "T", 0, 1, 0), ("chr1", 5, "+", "T", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[2, 0])),
    ("3M2D3M", 1, 16, [("chr1", 4, "-", "A", 0, 1, 0), ("chr1", 5, "-", "A", 0, 1, 0)],
     _tot(deletion_ops=[0, 1], deleted_bases=[0, 2])),
    ("3M2I3M", 1, 16, [("chr1", 3, "-", "C", 1, 0, 1)], _tot(insertion_ops=[0, 1], inserted_bases=[0, 2])),
    ("18M3D2M", 1, 0, [("chr1", 19, "+", "G", 0, 1, 0), ("chr1", 20, "+", "A", 0, 1, 0), ("chr1", 21, "+", "N", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[3, 0])),
    ("18M3D2M", 1, 16, [("chr1", 19, "-", "C", 0, 1, 0), ("chr1", 20, "-", "T", 0, 1, 0), ("chr1", 21, "-", "N", 0, 1, 0)],
     _tot(deletion_ops=[0, 1], deleted_bases=[0, 3])),
    ("20M1I2M", 1, 0, [("chr1", 20, "+", "A", 1, 0, 1)], _tot(insertion_ops=[1, 0], inserted_bases=[1, 0])),
    ("5M2I", 1, 0, [("chr1", 5, "+", "T", 1, 0, 1)], _tot(insertion_ops=[1, 0], inserted_bases=[2, 0])),
    # past the contig end: the M block ends on the last base, the deletion runs past it
    ("10M5D", 31, 0, [], _tot(deletion_ops=[1, 0])),
    ("10M5D2I", 31, 0, [], _tot(deletion_ops=[1, 0], insertion_ops=[1, 0], inserted_bases=[2, 0],
                                unanchored_insertions=[1, 0])),
    ("8M5D", 31, 0, [("chr1", 39, "+", "C", 0, 1, 0), ("chr1", 40, "+", "A", 0, 1, 0)],
     _tot(deletion_ops=[1, 0], deleted_bases=[2, 0])),
    ("10M2I", 31, 0, [("chr1", 40, "+", "A", 1, 0, 1)], _tot(insertion_ops=[1, 0], inserted_bases=[2, 0])),
    ("9M1D2I", 31, 16, [("chr1", 40, "-", "T", 0, 1, 1)],
     _tot(deletion_ops=[0, 1], deleted_bases=[0, 1], insertion_ops=[0, 1], inserted_bases=[0, 2])),
]


@pytest.mark.parametrize("case", range(len(HAND)), ids=[f"{c[0]}@{c[1]}{'-' if c[2] else '+'}" for c in HAND])
def test_hand_derived(case):
    cigar, pos, flag, rows, tot = HAND[case]
    got_rows, got_tot = _one(cigar, pos, flag)
    assert got_rows == rows
    assert got_tot == dict(tot, n_rows=len(rows))


def test_thresholds_on_one_position():
    # 3M1D2I3M: pos 4 has cov 0, del 1, ins 1
    assert _one("3M1D2I3M", min_events=2)[0] == [("chr1", 4, "+", "T", 0, 1, 1)]
    assert _one("3M1D2I3M", min_events=3)[0] == []
    assert _one("3M1D2I3M", min_depth=1)[0] == [("chr1", 4, "+", "T", 0, 1, 1)]
    assert _one("3M1D2I3M", min_depth=2)[0] == []
    # 3M2I3M: pos 3 has cov 1, ins 1: a row needs cov + del >= min_depth, so depth 2 drops it
    assert _one("3M2I3M", min_depth=1)[0] == [("chr1", 3, "+", "G", 1, 0, 1)]
    assert _one("3M2I3M", min_depth=2)[0] == []
    assert _one("3M2I3M", min_depth=0, min_events=0)[0] == [("chr1", 3, "+", "G", 1, 0, 1)]
    # the totals do not depend on the thresholds
    assert _one("3M1D2I3M", min_events=3)[1] == _one("3M1D2I3M")[1] | {"n_rows": 0}


def test_splice_with_indel_is_skipped():
    rows, tot = _one("3M2D3M10N4M")
    assert rows == [] and tot == dict(_tot(), n_rows=0)
    rows, tot = _one("3M10N4M")
    assert rows == [] and tot == dict(_tot(), n_rows=0)


def test_faults_and_unsorted():
    contigs, g, ref, recs = _case(0)
    bad = list(recs)
    bad.insert(3, bad[-1])
    with pytest.raises(to.TrackUnsorted):
        ti.track_indels_cpp(ref, ReadBatch.from_records(bad, ref))
    with pytest.raises(to.TrackUnsorted):
        ti.track_indels(to_py(bad), g)


def test_abi_layouts_and_keywords():
    assert C.sizeof(abi.ps_track_indel_opts) == 16
    assert C.sizeof(abi.ps_track_indel_row) == 24 == np.dtype(abi.TRACK_INDEL_ROW_DTYPE).itemsize
    assert C.sizeof(abi.ps_track_indel_totals) == 88
    assert C.sizeof(abi.ps_track_opts) == 16
    for f, _ in abi.ps_track_indel_row._fields_:
        assert getattr(abi.ps_track_indel_row, f).offset == np.dtype(abi.TRACK_INDEL_ROW_DTYPE).fields[f][1], f
    assert track_indel_opts(False, 5, 5) is None
    o = track_indel_opts(True, 3, 2)
    assert (o.indel_counts, o.min_depth, o.min_events, o.reserved) == (1, 3, 2, 0)
    with pytest.raises(ValueError):
        track_indel_opts(True, -1, 1)
    assert abi.PS_ABI_VERSION == 7

