"""GPU: the track's per-position deletion and insertion counts (ps_track_indel_opts.indel_counts) against the
restatements of tests/track_indels_oracle.py, bit for bit: batches through the host, device and misaligned views,
random and ragged batches of every CIGAR kind, config 5 (150-nt reads with indels and soft clips) at 1 M reads, config 2
(no indel at all), more than 65 536 events at one position, a deletion of tens of kb, contig ends, thresholds, faults,
and the file tool at several window sizes on one and two contexts.  With the option off, or beside base counts, the
track's other outputs are unchanged."""
import ctypes as C
import random

import numpy as np
import pytest

import py_oracle as po
import track_bases_oracle as tb
import track_indels_oracle as ti
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi, synth
from parasuite_b200.bamio import write_bam, write_fasta, write_sam
from test_contig_order_cpu import HEADER, header_sq, permuted_records
from test_track_indels_cpu import clean, indel_records, span_past_end_allowed

pytestmark = pytest.mark.gpu

ZERO = {k: [0, 0] for k in ti.TOTALS}


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


def misaligned(batch):
    """a DeviceBatch whose bases2 starts one byte into its allocation: the track reads it base by base"""
    import torch
    from parasuite_b200.runtime import DeviceBatch
    d = DeviceBatch(batch, "cuda:0")
    src = d._t["bases2"]
    buf = torch.zeros(src.numel() + 4, dtype=torch.uint8, device=src.device)
    buf[1:1 + src.numel()] = src
    torch.cuda.synchronize()
    d._t["bases2"] = buf
    d.struct.bases2 = buf.data_ptr() + 1
    return d


def views(batch):
    from parasuite_b200.runtime import DeviceBatch
    return [("host", batch), ("device", DeviceBatch(batch, "cuda:0")), ("misaligned", misaligned(batch))]


def same_track(got, exp, what):
    for k in ("runs_plus", "runs_minus", "sites"):
        assert got[k].dtype == exp[k].dtype and np.array_equal(got[k], exp[k]), (what, k)
    for k in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events",
              "n_runs", "n_sites"):
        assert got["counters"][k] == exp["counters"][k], (what, k)


def check(ctx, ref, batch, what, **kw):
    """every view against track_indels_cpp"""
    exp = ti.track_indels_cpp(ref, batch, **kw)
    ctx.upload_reference(ref)
    for how, v in views(batch):
        got = ctx.track(v, indel_counts=True, min_indel_depth=kw.get("min_depth", 1),
                        min_indel_events=kw.get("min_events", 1))
        same_track(got, exp, (what, how))
        assert got["indel_rows"].dtype == exp["indel_rows"].dtype
        assert np.array_equal(got["indel_rows"], exp["indel_rows"]), \
            (what, how, got["indel_rows"].size, exp["indel_rows"].size)
        assert got["indel_totals"] == exp["indel_totals"], (what, how)
    return exp


def _genome_case(seed, n=3000, length=5000, n_contigs=3):
    rng = random.Random(seed)
    contigs = random_genome(rng, n_contigs=n_contigs, length=length, n_frac=0.02, lower_frac=0.1)
    recs = indel_records(rng, contigs, n)
    recs += random_records(rng, contigs, n // 3, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 150),
                           err=0.05, flags_special=0.03)
    order = {c: i for i, (c, _) in enumerate(contigs)}
    recs = [r for r in recs if r.pos > 0 or r.flag & 4]
    recs.sort(key=lambda r: (order.get(r.rname, 99), r.pos))
    return rng, contigs, clean(recs, contigs)


# ---- 1. the option off, and beside base counts ---------------------------------------------------------------------
def test_option_off_and_beside(ctx):
    rng, contigs, recs = _genome_case(7100)
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    plain = ctx.track(b)
    on = ctx.track(b, indel_counts=True)
    assert set(plain) == {"runs_plus", "runs_minus", "sites", "counters"}
    same_track(on, plain, "beside")
    assert on["counters"] == plain["counters"] and on["indel_rows"].size > 0
    bases = ctx.track(b, base_counts=True, min_events=2)
    both = ctx.track(b, base_counts=True, min_events=2, indel_counts=True, min_indel_events=2)
    same_track(both, plain, "both")
    assert np.array_equal(both["base_rows"], bases["base_rows"]) and np.array_equal(both["base_totals"], bases["base_totals"])
    two = ctx.track(b, indel_counts=True, min_indel_events=2)
    assert np.array_equal(both["indel_rows"], two["indel_rows"]) and both["indel_totals"] == two["indel_totals"]
    lib = ctx.lib
    s = b.as_struct()
    for opts in (None, abi.ps_track_indel_opts(0, 5, 5, 0)):       # _ex2 with the option off is the plain call
        h = C.c_void_p()
        assert lib.ps_track_batch_ex2(ctx.h, C.byref(s), None, C.byref(opts) if opts else None, C.byref(h)) == abi.PS_OK
        ctr = abi.ps_track_counters()
        lib.ps_track_counters_get(h, C.byref(ctr))
        assert ctr.as_dict() == plain["counters"]
        assert lib.ps_track_indel_rows(h, 0, None, 0) == abi.PS_ERR_STATE
        assert lib.ps_track_indel_totals_get(h, C.byref(abi.ps_track_indel_totals())) == abi.PS_ERR_STATE
        lib.ps_track_close(h)
    bad = abi.ps_track_indel_opts(1, 1, 1, 1)
    for call in (lambda h: lib.ps_track_batch_ex2(ctx.h, C.byref(s), None, C.byref(bad), C.byref(h)),
                 lambda h: lib.ps_track_batch_device_ex2(ctx.h, C.byref(s), None, C.byref(bad), None, C.byref(h))):
        h = C.c_void_p()
        assert call(h) == abi.PS_ERR_INVALID_ARG and not h.value
    assert lib.ps_track_bam_ex2(ctx.h, b"none.bam", b"none", None, C.byref(bad), None, None, None, None) == \
        abi.PS_ERR_INVALID_ARG


# ---- 2. batches against the C++ restatement ------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(3))
def test_random_batches_all_cigar_kinds(ctx, seed):
    rng, contigs, recs = _genome_case(7200 + seed)
    ref = PackedReference.from_contigs(contigs)
    exp = check(ctx, ref, ReadBatch.from_records(recs, ref), f"random {seed}")
    t = exp["indel_totals"]
    assert exp["indel_rows"].size > 100 and min(t["unanchored_insertions"]) > 0 and min(t["deletion_ops"]) > 0


def test_ragged_and_uniform(ctx):
    rng = random.Random(7300)
    contigs = random_genome(rng, n_contigs=2, length=8000, n_frac=0.01, lower_frac=0.1)
    ref = PackedReference.from_contigs(contigs)
    ragged = clean(random_records(rng, contigs, 6000, kinds=("M", "indel", "clip"), Lrange=(18, 90), err=0.05), contigs)
    check(ctx, ref, ReadBatch.from_records(ragged, ref), "ragged")
    uni = clean(random_records(rng, contigs, 6000, kinds=("M", "M", "indel"), Lrange=(36, 36), err=0.05), contigs)
    b = ReadBatch.from_records(uni, ref)
    assert b.uniform_len == 36
    check(ctx, ref, b, "uniform")


def test_more_than_65536_events_at_one_position(ctx):
    """70 000 reads on each strand delete position 61 and insert after it"""
    contigs = [("chr1", b"ACGTACGTAC" * 20)]
    n = 70_000
    recs = []
    for flag in (0, 16):
        recs += [Record(flag, "chr1", 51, "10M1D2I8M", b"A" * 20, bytes([30] * 20)) for _ in range(n)]
    recs.sort(key=lambda r: r.pos)
    ref = PackedReference.from_contigs(contigs)
    exp = check(ctx, ref, ReadBatch.from_records(recs, ref), "65536")
    rows = exp["indel_rows"]
    for s in (0, 1):
        hit = rows[(rows["pos"] == 61) & (rows["strand"] == s)]
        assert hit.size == 1 and int(hit["del"][0]) == n and int(hit["ins"][0]) == n
    assert exp["indel_totals"]["deleted_bases"] == [n, n]


def test_long_deletion_inside_one_read(ctx):
    """a 40 kb deletion inside one read, under reads that cover part of it"""
    rng = random.Random(7400)
    contigs = [("chr1", bytes(rng.choice(b"ACGT") for _ in range(100_000))), ("chr2", b"ACGT" * 100)]
    recs = [Record(0, "chr1", 1000, "20M40000D20M", b"A" * 40, bytes([30] * 40)),
            Record(16, "chr1", 1005, "10M25000D3I10M", b"A" * 23, bytes([30] * 23))]
    recs += [Record(rng.choice((0, 16)), "chr1", p, "30M", b"C" * 30, bytes([30] * 30))
             for p in sorted(rng.randint(1100, 41000) for _ in range(500))]
    recs.sort(key=lambda r: r.pos)
    ref = PackedReference.from_contigs(contigs)
    exp = check(ctx, ref, ReadBatch.from_records(recs, ref), "40 kb")
    assert exp["indel_totals"]["deleted_bases"] == [40_000, 25_000]
    assert exp["indel_rows"].size == 65_000          # the insertion sits on a deleted base of the minus strand


def test_contig_ends(ctx):
    """10M5D with its M block ending on the contig's last base, a trailing 2I after it, and shorter cases, on a contig
    followed by another: nothing is counted past the contig's end"""
    rng = random.Random(7500)
    contigs = [(f"chr{k + 1}", bytes(rng.choice(b"ACGT") for _ in range(200 + 13 * k))) for k in range(3)]
    recs = []
    for name, seq in contigs:
        n = len(seq)
        for cig, p, flag in (("5M3D5M", 1, 0), ("2D8M", 1, 16), ("10M5D", n - 9, 0), ("10M5D2I", n - 9, 16),
                             ("8M5D", n - 9, 0), ("10M2I", n - 9, 0), ("9M1D2I", n - 9, 16), ("10M1I", n - 9, 16),
                             ("4M3D", n - 6, 0)):
            L = sum(k for op, k in po.parse_cigar(cig) if op in "MIS=X")
            recs.append(Record(flag, name, p, cig, bytes(rng.choice(b"ACGT") for _ in range(L)), bytes([30] * L)))
        recs += [Record(rng.choice((0, 16)), name, p, "20M", b"G" * 20, bytes([30] * 20))
                 for p in sorted(rng.randint(1, n - 19) for _ in range(40))]
    order = {c: i for i, (c, _) in enumerate(contigs)}
    recs.sort(key=lambda r: (order[r.rname], r.pos))
    ref = PackedReference.from_contigs(contigs)
    b = span_past_end_allowed(ReadBatch.from_records(recs, ref))
    py = ti.track_indels(to_py(recs), po.Genome(dict(contigs)))
    exp = check(ctx, ref, b, "contig ends")
    assert exp["indel_totals"] == {k: py["indel_totals"][k] for k in exp["indel_totals"]}
    rows = exp["indel_rows"]
    for c, (_, seq) in enumerate(contigs):
        r = rows[rows["contig"] == c]
        assert int(r["pos"].max()) == len(seq) and int(r["pos"].min()) == 1
    assert exp["indel_totals"]["unanchored_insertions"] == [0, 3]


def test_thresholds(ctx):
    rng, contigs, recs = _genome_case(7600, n=4000, length=2000, n_contigs=2)
    ref = PackedReference.from_contigs(contigs)
    b = ReadBatch.from_records(recs, ref)
    sizes = []
    for md, me in ((0, 0), (1, 1), (5, 1), (1, 2), (20, 2), (60, 3), (10 ** 6, 1)):
        sizes.append(check(ctx, ref, b, (md, me), min_depth=md, min_events=me)["indel_rows"].size)
    assert sizes[0] == sizes[1] > 0 and sizes[1] >= sizes[2] >= sizes[4] and sizes[1] >= sizes[3] and sizes[-1] == 0


# ---- 3. config 5 and config 2 at 1 M reads -------------------------------------------------------------------------
def test_config5_million(ctx):
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(0x5EED0001, [10_000_000])
    b = synth.synth_reads(ref, 1_000_000, 150, seed=0x5EED0002, mode=1)
    ctx.upload_reference(ref)
    exp = ti.track_indels_cpp(ref, b)
    got = ctx.track(DeviceBatch(b, "cuda:0"), indel_counts=True)
    same_track(got, exp, "config 5")
    assert np.array_equal(got["indel_rows"], exp["indel_rows"]) and got["indel_totals"] == exp["indel_totals"]
    t = got["indel_totals"]
    assert min(t["deletion_ops"]) > 0 and min(t["insertion_ops"]) > 0 and got["indel_rows"].size > 1000
    for s in (0, 1):
        r = got["indel_rows"][got["indel_rows"]["strand"] == s]
        assert int(r["del"].sum()) == t["deleted_bases"][s]
        assert int(r["ins"].sum()) == t["insertion_ops"][s] - t["unanchored_insertions"][s]


def test_config2_no_indels(ctx):
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(0x5EED0001, [10_000_000])
    b = synth.synth_reads(ref, 1_000_000, 36, seed=0x5EED0002)
    ctx.upload_reference(ref)
    d = DeviceBatch(b, "cuda:0")
    plain = ctx.track(d)
    got = ctx.track(d, indel_counts=True)
    same_track(got, plain, "config 2")
    assert got["counters"] == plain["counters"]
    assert got["indel_rows"].size == 0 and got["indel_totals"] == dict(ZERO, n_rows=0)


# ---- 4. faults -----------------------------------------------------------------------------------------------------
def _outcome(fn):
    try:
        return ("ok", fn())
    except abi.PsError as e:
        return (e.status, e.fault)


def test_faults_match_the_plain_track(ctx):
    rng = random.Random(7700)
    contigs = random_genome(rng, n_contigs=2, length=3000, n_frac=0.0, lower_frac=0.0)
    recs = clean(indel_records(rng, contigs, 400), contigs)
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    name, seq = contigs[0]
    cases = {
        "block range": recs[:200] + [Record(0, name, recs[199].pos, "40M", b"A" * 30, bytes([30] * 30))] + recs[200:],
        "ref range": recs[:100] + [Record(0, "chrUn", 5, "30M", b"A" * 30, bytes([30] * 30))] + recs[100:],
        "cigar ops": recs[:150] + [Record(0, name, recs[150].pos, "1M1I" * 130 + "10M", b"A" * 270, bytes([30] * 270))]
        + recs[150:],
        "past end": [r for r in recs if r.rname == name] + [Record(0, name, len(seq) + 1, "5S5I", b"ACGTACGTAC",
                                                                   bytes([30] * 10))],
        "span past end": [r for r in recs if r.rname == name] + [Record(0, name, len(seq) - 9, "10M5D", b"A" * 10,
                                                                        bytes([30] * 10))],
        "unsorted": recs[:50] + [recs[300]] + recs[50:],
    }
    for what, rs in cases.items():
        b = ReadBatch.from_records(rs, ref)
        for how, v in views(b):
            plain = _outcome(lambda: ctx.track(v))
            ind = _outcome(lambda: ctx.track(v, indel_counts=True, base_counts=True))
            assert plain[0] != "ok" and plain == ind, (what, how, plain, ind)
        h = C.c_void_p()
        s = b.as_struct()
        opts = abi.ps_track_indel_opts(1, 1, 1, 0)
        st = ctx.lib.ps_track_batch_ex2(ctx.h, C.byref(s), None, C.byref(opts), C.byref(h))
        assert st != abi.PS_OK
        if h.value:
            assert ctx.lib.ps_track_indel_rows(h, 0, None, 0) == 0
            tot = abi.ps_track_indel_totals()
            assert ctx.lib.ps_track_indel_totals_get(h, C.byref(tot)) == abi.PS_OK
            assert tot.as_dict() == dict(ZERO, n_rows=0)
            ctx.lib.ps_track_close(h)


# ---- 5. the file tool ----------------------------------------------------------------------------------------------
FILES = ("plus.bedGraph", "minus.bedGraph", "t2c.tsv")


def _texts(prefix, extra=()):
    return {k: open(f"{prefix}.{k}").read() for k in FILES + tuple(extra)}


def _file_case(tmp_path, fmt):
    contigs, recs = permuted_records(66, n=600, kinds=("M", "clip", "indel"))
    rng = random.Random(7800)
    present = [contigs[c] for c in HEADER]
    recs += indel_records(rng, present, 1200)
    hpos = {contigs[c][0]: h for h, c in enumerate(HEADER)}
    recs.sort(key=lambda r: (hpos[r.rname], r.pos))
    recs = clean(recs, contigs, [contigs[c][0] for c in HEADER])
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / f"reads.{fmt}")
    write_fasta(fa, contigs)
    (write_bam if fmt == "bam" else write_sam)(path, header_sq(contigs), recs)
    return contigs, recs, fa, path, [contigs[c][0] for c in HEADER]


@pytest.mark.parametrize("window", [10 ** 9, 700, 97, 1])
@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_track_bam_files(tmp_path, monkeypatch, window, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs, fa, path, order = _file_case(tmp_path, fmt)
    want = ti.track_indels(to_py(recs), po.Genome(dict(contigs)), order, min_events=1)
    want_bases = tb.track_bases(to_py(recs), po.Genome(dict(contigs)), order)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
    c = Context(0)
    try:
        c.load_fasta(fa)
        plain = c.track_bam(path, str(tmp_path / "plain"))
        ctr = c.track_bam(path, str(tmp_path / "out"), indel_counts=True)
        both = c.track_bam(path, str(tmp_path / "both"), indel_counts=True, base_counts=True)
    finally:
        c.close()
    assert _texts(tmp_path / "out", ("indels.tsv",)) == {k: want["files"][k] for k in FILES + ("indels.tsv",)}
    assert _texts(tmp_path / "plain") == {k: want["files"][k] for k in FILES}
    assert not (tmp_path / "out.bases.tsv").exists() and not (tmp_path / "plain.indels.tsv").exists()
    assert _texts(tmp_path / "both", ("indels.tsv", "bases.tsv")) == \
        dict(_texts(tmp_path / "out", ("indels.tsv",)), **{"bases.tsv": want_bases["files"]["bases.tsv"]})
    assert {k: v for k, v in ctr.items() if k != "indel_totals"} == plain
    assert ctr["indel_totals"] == want["indel_totals"] and ctr["indel_totals"]["n_rows"] > 100
    assert both["indel_totals"] == ctr["indel_totals"]
    assert np.array_equal(both["base_totals"], want_bases["base_totals"])


def test_two_contexts(tmp_path, monkeypatch):
    import torch
    from parasuite_b200.runtime import Context, MultiContext
    contigs, recs, fa, path, order = _file_case(tmp_path, "bam")
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", "211")
    c = Context(0)
    try:
        c.load_fasta(fa)
        one = c.track_bam(path, str(tmp_path / "one"), indel_counts=True, min_indel_events=2, min_indel_depth=3)
    finally:
        c.close()
    want = ti.track_indels(to_py(recs), po.Genome(dict(contigs)), order, min_events=2, min_depth=3)
    assert _texts(tmp_path / "one", ("indels.tsv",))["indels.tsv"] == want["files"]["indels.tsv"]
    devs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() > 1 else [])
    for d in devs:
        m = MultiContext(d)
        try:
            m.load_fasta(fa)
            ctr = m.track_bam(path, str(tmp_path / "m"), indel_counts=True, min_indel_events=2, min_indel_depth=3)
        finally:
            m.close()
        assert _texts(tmp_path / "m", ("indels.tsv",)) == _texts(tmp_path / "one", ("indels.tsv",)), d
        assert ctr == one, d
