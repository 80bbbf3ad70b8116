"""The track's read and base filters without a GPU: struct layouts, option validation, FLAG and MAPQ through the
batcher (BAM bytes and SAM text) against ReadBatch.from_records, the Python and C++ restatements under every filter,
and the record filter as a pre-filter of the records."""
import ctypes as C
import random
import struct

import numpy as np
import pytest

import py_oracle as po
import track_filters_oracle as tfo
import track_oracle as to
from parasuite_b200 import PackedReference, ReadBatch, Record, abi
from parasuite_b200.bamio import BamBatcher, PackedFasta, encode_bam_record, write_bam, write_fasta, write_sam
from parasuite_b200.runtime import track_filter_opts

FILTERS = ("min_mapq", "require_flags", "exclude_flags", "min_base_quality")


def to_py(records):
    """Record -> py_oracle.Rec with the MAPQ (255 when the record has none)"""
    out = []
    for r in records:
        q = bytes(r.qual)
        if len(q) == 0 or q[0] == 0xFF:
            q = b""
        out.append(tfo.Rec(r.flag, r.rname, r.pos, po.parse_cigar(r.cigar), bytes(r.seq), q,
                          255 if r.mapq is None else r.mapq))
    return out


def genome_of(contigs):
    return po.Genome({n: s.encode() for n, s in contigs})


def random_records(rng, contigs, n, ragged=True, indels=True):
    """sorted records with random flags (secondary, QC-fail, duplicate, supplementary, reverse, unmapped), MAPQ and
    qualities, some without qualities"""
    recs = []
    for name, seq in contigs:
        pos = 1
        for _ in range(n):
            pos += rng.randrange(0, 4)
            L = rng.choice((20, 36, 50)) if ragged else 36
            if pos + L + 5 > len(seq):
                break
            r = rng.random()
            if indels and r < 0.2:
                a = rng.randrange(3, L - 3)
                cig = f"{a}M{rng.randrange(1, 4)}D{L - a}M"
            elif indels and r < 0.35:
                a = rng.randrange(3, L - 3)
                cig = f"{a}M2I{L - a - 2}M"
            elif r < 0.45:
                cig = f"2S{L - 2}M"
            else:
                cig = f"{L}M"
            flag = rng.choice((0, 0x10)) | (rng.random() < 0.4 and rng.choice((0x100, 0x200, 0x400, 0x800)) or 0)
            if rng.random() < 0.03:
                flag |= 0x4
            bases = "".join(rng.choice("ACGTTC") if rng.random() < 0.3 else seq[pos - 1 + k] for k in range(L))
            qual = b"" if rng.random() < 0.05 else bytes(rng.choice((2, 10, 19, 20, 21, 37)) for _ in range(L))
            mapq = rng.choice((None, 0, 1, 9, 10, 30, 60, 255))
            recs.append(Record(flag, name, pos, cig, bases.encode(), qual, mapq))
    return recs


CONTIGS = [("chr1", "".join(random.Random(1).choice("ACGT") for _ in range(3000))),
           ("chr2", "".join(random.Random(2).choice("ACGTN") for _ in range(2000)))]

FILTER_CASES = [
    {},
    {"min_mapq": 10},
    {"exclude_flags": 0x904},
    {"require_flags": 0x10},
    {"exclude_flags": 0x400, "require_flags": 0x10, "min_mapq": 1},
    {"min_base_quality": 20},
    {"min_base_quality": 1},
    {"min_base_quality": 255},
    {"min_base_quality": 21, "min_mapq": 30, "exclude_flags": 0x900},
]


# ---- layouts and options ------------------------------------------------------------------------------------------
def test_struct_layouts():
    assert C.sizeof(abi.ps_track_filter_opts) == 32
    assert C.sizeof(abi.ps_track_filter_counters) == 32
    assert C.sizeof(abi.ps_read_aux) == 16
    assert abi.ps_track_filter_opts.min_base_quality.offset == 12
    assert abi.ps_track_filter_counters.low_quality_bases.offset == 16


def test_filter_options_validation():
    assert track_filter_opts(0, 0, 0, 0) is None
    o = track_filter_opts(255, 0xFFFF, 0x904, 255)
    assert (o.min_mapq, o.require_flags, o.exclude_flags, o.min_base_quality) == (255, 0xFFFF, 0x904, 255)
    assert list(o.reserved) == [0] * 4
    for bad in ((256, 0, 0, 0), (-1, 0, 0, 0), (0, 0x10000, 0, 0), (0, 0, 0x10000, 0), (0, 0, -4, 0), (0, 0, 0, 256),
                (0, 0, 0, -1)):
        with pytest.raises(ValueError):
            track_filter_opts(*bad)


# ---- FLAG and MAPQ through the batcher ------------------------------------------------------------------------------
def _flag_records():
    recs = []
    flags = (0, 0x100, 0x200, 0x400, 0x800, 0x10 | 0x100, 0x4, 0x200 | 0x800)
    mapqs = (0, 1, 60, 255, None)
    pos = 1
    for i, (f, q) in enumerate((f, q) for f in flags for q in mapqs):
        pos += i % 3
        recs.append(Record(f, "chr1", pos, "30M", CONTIGS[0][1][pos - 1:pos + 29].encode(), bytes([30] * 30), q))
    return recs


def test_bam_record_bytes_carry_mapq_and_flag():
    rec = Record(0x900 | 0x10, "chr1", 5, "4M", b"ACGT", b"\x1e" * 4, 60)
    raw = encode_bam_record(rec, {"chr1": 0})
    assert raw[4 + 9] == 60                                     # MAPQ: byte 9 of the record after block_size
    assert struct.unpack_from("<H", raw, 4 + 14)[0] == 0x910    # FLAG
    assert encode_bam_record(Record(0, "chr1", 5, "4M", b"ACGT", b"\x1e" * 4), {"chr1": 0})[4 + 9] == 255


@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_batcher_carries_flag_and_mapq(tmp_path, fmt):
    recs = _flag_records()
    fa = str(tmp_path / "g.fa")
    write_fasta(fa, [(n, s.encode()) for n, s in CONTIGS])
    path = str(tmp_path / f"r.{fmt}")
    lens = [(n, len(s)) for n, s in CONTIGS]
    (write_bam if fmt == "bam" else write_sam)(path, lens, recs)
    pf = PackedFasta(fa)
    got = list(BamBatcher(path, pf, max_batch_reads=7, threads=2))
    flags = np.concatenate([b.sam_flags for b in got])
    mapq = np.concatenate([b.mapq for b in got])
    want = ReadBatch.from_records(recs, pf.reference())
    assert np.array_equal(flags, want.sam_flags)
    assert np.array_equal(flags, [r.flag for r in recs])
    # SAM text without a MAPQ column value keeps the writer's "30"; BAM without one, 255
    none_q = 255 if fmt == "bam" else 30
    assert list(mapq) == [none_q if r.mapq is None else r.mapq for r in recs]
    assert np.array_equal(want.mapq, [255 if r.mapq is None else r.mapq for r in recs])
    assert {0, 1, 60, 255} <= set(int(x) for x in mapq)


# ---- the two restatements agree -------------------------------------------------------------------------------------
def _cpp_vs_py(res_c, res_p, names):
    for s, k in ((0, "runs_plus"), (1, "runs_minus")):
        got = [(names[x["contig"]], int(x["start0"]), int(x["end0"]), int(x["cov"])) for x in res_c[k]]
        assert got == [tuple(r) for r in res_p[k]], k
    got = [(names[x["contig"]], int(x["pos"]), "+-"[x["strand"]], int(x["t2c"]), int(x["cov"])) for x in res_c["sites"]]
    assert got == list(res_p["sites"])
    for f in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events"):
        assert res_c["counters"][f] == res_p["counters"][f], f


@pytest.mark.parametrize("case", range(len(FILTER_CASES)))
@pytest.mark.parametrize("seed", [3, 4])
def test_oracles_agree_under_filters(case, seed):
    flt = FILTER_CASES[case]
    rng = random.Random(seed)
    recs = random_records(rng, CONTIGS, 150)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    batch = ReadBatch.from_records(recs, ref)
    g = genome_of(CONTIGS)
    py, cc = tfo.track(to_py(recs), g, **flt), tfo.track_cpp(ref, batch, **flt)
    _cpp_vs_py(cc, py, ref.names)
    assert ("filter_counters" in cc) == bool(flt) == ("filter_counters" in py)
    if flt:
        assert cc["filter_counters"] == py["filter_counters"]
        c, fc = cc["counters"], cc["filter_counters"]
        assert c["num_reads_processed"] == (fc["filtered_flags"] + fc["filtered_mapq"] + c["unmapped"] +
                                            c["skipped_due_indel"] + c["reads_counted"])
    # aligned bases are what the runs hold
    for s, k in ((0, "runs_plus"), (1, "runs_minus")):
        assert cc["counters"]["aligned_bases"][s] == int(((cc[k]["end0"] - cc[k]["start0"]).astype(np.int64) *
                                                          cc[k]["cov"]).sum())
    # base counts and indel counts under the same filters
    pb, cb = tfo.track_bases(to_py(recs), g, **flt), tfo.track_cpp(ref, batch, bases={}, **flt)
    got = [(ref.names[x["contig"]], int(x["pos"]), "+-"[x["strand"]], "ACGT"[x["ref"]], int(x["cov"]),
            *map(int, x["n"])) for x in cb["base_rows"]]
    assert got == list(pb["base_rows"])
    assert np.array_equal(cb["base_totals"], pb["base_totals"])
    for s in (0, 1):
        assert int(cb["base_totals"][s][3][1]) == cc["counters"]["t2c_events"][s]
    pi, ci = tfo.track_indels(to_py(recs), g, **flt), tfo.track_cpp(ref, batch, indels={}, **flt)
    got = [(ref.names[x["contig"]], int(x["pos"]), "+-"[x["strand"]], "ACGTN"[x["ref"]], int(x["cov"]), int(x["del"]),
            int(x["ins"])) for x in ci["indel_rows"]]
    assert got == list(pi["indel_rows"])


def test_base_quality_threshold_edges():
    """a base exactly at the threshold passes; q = 1 drops only Q0; q = 255 drops every base of a read with
    qualities; a read without qualities keeps every base"""
    seq = CONTIGS[0][1]
    quals = bytes([0, 1, 19, 20, 21, 40, 0, 20])
    recs = [Record(0, "chr1", 10, "8M", seq[9:17].encode(), quals),
            Record(0x10, "chr1", 12, "8M", seq[11:19].encode(), b"")]
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    batch = ReadBatch.from_records(recs, ref)
    for q, low in ((20, 4), (21, 6), (1, 2), (255, 8), (0, 0)):
        res = tfo.track_cpp(ref, batch, min_base_quality=q)
        assert res["counters"]["aligned_bases"] == [8 - low, 8], q
        if q:
            assert res["filter_counters"]["low_quality_bases"] == [low, 0]
        assert res["counters"]["fast_path_reads"] == 0


@pytest.mark.parametrize("flt", [{"min_mapq": 10}, {"exclude_flags": 0x904}, {"require_flags": 0x10, "min_mapq": 1}])
def test_record_filter_is_a_prefilter(flt):
    """the record filter equals the call on the records it keeps; fault ordinals map back"""
    rng = random.Random(9)
    recs = random_records(rng, CONTIGS, 120)
    # a kept-order break and a fault that only filtered records carry
    bad = Record(0x100, "chr1", 2900, "500M", b"A" * 500, bytes([30] * 500), 0)       # past the contig: would fault
    recs.insert(len(recs) // 3, bad)
    back = Record(0x900, "chr1", 1, "10M", CONTIGS[0][1][:10].encode(), bytes([30] * 10), 0)   # out of order
    recs.insert(len(recs) // 2, back)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    g = genome_of(CONTIGS)
    keep = [r for r in recs if not tfo.filtered(to_py([r])[0], flt.get("require_flags", 0), flt.get("exclude_flags", 0),
                                                  flt.get("min_mapq", 0))]
    assert bad not in keep and back not in keep
    a = tfo.track_cpp(ref, ReadBatch.from_records(recs, ref), **flt)
    b = tfo.track_cpp(ref, ReadBatch.from_records(keep, ref))
    for k in ("runs_plus", "runs_minus", "sites"):
        assert np.array_equal(a[k], b[k]), k
    ca, cb = dict(a["counters"]), dict(b["counters"])
    fc = a["filter_counters"]
    assert ca.pop("num_reads_processed") == cb.pop("num_reads_processed") + fc["filtered_flags"] + fc["filtered_mapq"]
    assert ca == cb
    assert tfo.track(to_py(recs), g, **flt)["files"] == tfo.track(to_py(keep), g)["files"]
    # a fault among the kept records: its ordinal in the full batch
    faulty = Record(0x10, "chr1", 2990, "50M", b"A" * 50, bytes([30] * 50), 60)
    full = recs[:10] + [faulty] + recs[10:]
    kept = [r for r in full if r in keep or r is faulty]
    with pytest.raises(to.TrackFault) as e1:
        tfo.track_cpp(ref, ReadBatch.from_records(full, ref), **flt)
    with pytest.raises(to.TrackFault) as e2:
        tfo.track_cpp(ref, ReadBatch.from_records(kept, ref))
    assert e1.value.code == e2.value.code
    assert e1.value.ordinal == full.index(faulty) and e2.value.ordinal == kept.index(faulty)


def test_past_end_record_faults_even_when_filtered():
    seq = CONTIGS[0][1]
    recs = [Record(0, "chr1", 5, "10M", seq[4:14].encode(), bytes([30] * 10), 60),
            Record(0x100, "chr1", len(seq) + 3, "5S", b"ACGTA", bytes([30] * 5), 60)]
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    batch = ReadBatch.from_records(recs, ref)
    assert batch.past_end == 2
    for impl in (lambda: tfo.track_cpp(ref, batch, exclude_flags=0x100),
                 lambda: tfo.track(to_py(recs), genome_of(CONTIGS), exclude_flags=0x100)):
        with pytest.raises(to.TrackFault) as e:
            impl()
        assert (e.value.code, e.value.ordinal) == (po.PS_FAULT_PAST_END, 1)
