"""GPU: the track's read and base filters (ps_track_filter_opts) against the restatements, bit for bit, through the
host, device and misaligned views, alone and beside base counts and indel counts: every arm of the bit-parallel path
with low-quality bases at the word edges, the record filter against the pre-filtered batch, option errors, all-zero
options, the file tool at three window sizes on one and two contexts, and one config-2-sized batch."""
import ctypes as C
import random

import numpy as np
import pytest

import py_oracle as po
import track_filters_oracle as tfo
import track_oracle as to
from parasuite_b200 import PackedReference, ReadBatch, Record, abi, synth
from parasuite_b200.bamio import write_bam, write_fasta, write_sam
from test_track_filters_cpu import CONTIGS, genome_of, random_records, to_py

pytestmark = pytest.mark.gpu

RECORD_FILTER = {"min_mapq": 10, "exclude_flags": 0x904}
FULL_FILTER = {"min_mapq": 10, "exclude_flags": 0x904, "min_base_quality": 20}


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


def misaligned(batch):
    """a DeviceBatch whose bases2 and qual start one byte into their allocations: the per-base path"""
    import torch
    from parasuite_b200.runtime import DeviceBatch
    d = DeviceBatch(batch, "cuda:0")
    for f in ("bases2", "qual"):
        src = d._t[f]
        buf = torch.zeros(src.numel() + 4, dtype=torch.uint8, device=src.device)
        buf[1:1 + src.numel()] = src
        d._t[f] = buf
        setattr(d.struct, f, buf.data_ptr() + 1)
    torch.cuda.synchronize()
    return d


def views(batch):
    from parasuite_b200.runtime import DeviceBatch
    return [("host", batch), ("device", DeviceBatch(batch, "cuda:0")), ("misaligned", misaligned(batch))]


def _same(got, exp, what, keys=("runs_plus", "runs_minus", "sites")):
    for k in keys:
        assert got[k].dtype == exp[k].dtype and np.array_equal(got[k], exp[k]), (what, k)
    for k in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events",
              "n_runs", "n_sites"):
        assert got["counters"][k] == exp["counters"][k], (what, k)


def check(ctx, ref, batch, what, flt, fast=False):
    """every view, alone and with base counts, indel counts and both, against the C++ restatements"""
    exp = tfo.track_cpp(ref, batch, **flt)
    eb = tfo.track_cpp(ref, batch, bases={}, **flt)
    ei = tfo.track_cpp(ref, batch, indels={}, **flt)
    ctx.upload_reference(ref)
    for how, v in views(batch):
        # the base filter keeps every read on its arm: the same call without it takes as many bit-parallel reads
        unfiltered = ctx.track(v, **{k: x for k, x in flt.items() if k != "min_base_quality"})["counters"]["fast_path_reads"]
        for opt in ({}, {"base_counts": True}, {"indel_counts": True}, {"base_counts": True, "indel_counts": True}):
            got = ctx.track(v, **opt, **flt)
            w = (what, how, tuple(opt))
            _same(got, exp, w)
            assert got["filter_counters"] == exp["filter_counters"], w
            assert got["counters"]["fast_path_reads"] == unfiltered, w
            if fast and how != "misaligned":
                assert unfiltered > 0, w
            if opt.get("base_counts"):
                assert np.array_equal(got["base_rows"], eb["base_rows"]), w
                assert np.array_equal(got["base_totals"], eb["base_totals"]), w
                for s in (0, 1):
                    assert int(got["base_totals"][s, 3, 1]) == got["counters"]["t2c_events"][s], w
            if opt.get("indel_counts"):
                assert np.array_equal(got["indel_rows"], ei["indel_rows"]), w
                assert got["indel_totals"] == ei["indel_totals"], w
        c, fc = got["counters"], got["filter_counters"]
        assert c["num_reads_processed"] == (fc["filtered_flags"] + fc["filtered_mapq"] + c["unmapped"] +
                                            c["skipped_due_indel"] + c["reads_counted"])
        for s, k in ((0, "runs_plus"), (1, "runs_minus")):
            r = got[k]
            assert c["aligned_bases"][s] == int(((r["end0"] - r["start0"]).astype(np.int64) * r["cov"]).sum())
    return exp


# ---- 1. the bit-parallel arm ----------------------------------------------------------------------------------------
def _uniform_case(L, seed):
    rng = random.Random(seed)
    name, seq = CONTIGS[0]
    edges = [p for p in (0, 15, 16, 31, 32, 63, L - 1) if p < L]
    recs, pos = [], 1
    for i in range(1200):
        pos += rng.randrange(0, 3)
        if pos + L > len(seq):
            break
        q = [30] * L
        kind = i % 7
        if kind == 0:
            for p in edges:
                q[p] = 5
        elif kind == 1:
            q = [5] * L                                         # all low
        elif kind == 2:
            q = [5 if k % 2 == 0 else 30 for k in range(L)]     # alternating: the most runs
        elif kind == 3:
            q = [rng.choice((19, 20, 21)) for _ in range(L)]    # at the threshold
        elif kind == 4:
            for p in rng.sample(range(L), 3):
                q[p] = 0
        qual = b"" if kind == 5 and i % 2 else bytes(q)         # some reads without qualities
        bases = "".join(rng.choice("CGAT") if rng.random() < 0.2 else seq[pos - 1 + k] for k in range(L))
        flag = rng.choice((0, 0x10)) | (0x100 if i % 11 == 0 else 0)
        recs.append(Record(flag, name, pos, f"{L}M", bases.encode(), qual, rng.choice((None, 0, 5, 10, 60))))
    return recs


@pytest.mark.parametrize("L", [36, 50, 64])
@pytest.mark.parametrize("flt", [{"min_base_quality": 20}, FULL_FILTER])
def test_fast_arm(ctx, L, flt):
    recs = _uniform_case(L, 100 + L)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    batch = ReadBatch.from_records(recs, ref)
    assert batch.uniform_len == L and batch.uniform_ncigar == 1
    exp = check(ctx, ref, batch, f"L={L}", flt, fast=True)
    assert exp["filter_counters"]["low_quality_bases"][0] > 0 and exp["filter_counters"]["low_quality_bases"][1] > 0


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("flt", [{"min_base_quality": 20}, {"min_base_quality": 255}, {"min_base_quality": 1},
                                 FULL_FILTER, {"require_flags": 0x10}])
def test_general_path(ctx, seed, flt):
    recs = random_records(random.Random(seed), CONTIGS, 400)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    check(ctx, ref, ReadBatch.from_records(recs, ref), f"seed {seed}", flt)


# ---- 2. the record filter is a pre-filter ---------------------------------------------------------------------------
def _keep(recs, flt):
    return [r for r in recs if not tfo.filtered(to_py([r])[0], flt.get("require_flags", 0), flt.get("exclude_flags", 0),
                                               flt.get("min_mapq", 0))]


@pytest.mark.parametrize("flt", [RECORD_FILTER, {"require_flags": 0x10, "min_mapq": 1}])
def test_record_filter_equals_prefiltered_batch(ctx, flt):
    recs = random_records(random.Random(31), CONTIGS, 400)
    recs.insert(len(recs) // 3, Record(0x900, "chr1", 2900, "500M", b"A" * 500, bytes([30] * 500), 0))   # would fault
    recs.insert(len(recs) // 2, Record(0x904, "chr1", 1, "10M", CONTIGS[0][1][:10].encode(), bytes([30] * 10), 0))
    keep = _keep(recs, flt)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    ctx.upload_reference(ref)
    full, kept = ReadBatch.from_records(recs, ref), ReadBatch.from_records(keep, ref)
    for how, v in views(full):
        a = ctx.track(v, base_counts=True, indel_counts=True, **flt)
        b = ctx.track(kept, base_counts=True, indel_counts=True)
        for k in ("runs_plus", "runs_minus", "sites", "base_rows", "base_totals", "indel_rows"):
            assert np.array_equal(a[k], b[k]), (how, k)
        assert a["indel_totals"] == b["indel_totals"]
        ca, cb, fc = dict(a["counters"]), dict(b["counters"]), a["filter_counters"]
        assert ca.pop("num_reads_processed") == cb.pop("num_reads_processed") + fc["filtered_flags"] + fc["filtered_mapq"]
        assert ca == cb, how
    # without the filter the same batch faults
    with pytest.raises(abi.PsError):
        ctx.track(full)


def test_past_end_is_raised_for_a_filtered_record(ctx):
    seq = CONTIGS[0][1]
    recs = [Record(0, "chr1", 5, "10M", seq[4:14].encode(), bytes([30] * 10), 60),
            Record(0x100, "chr1", len(seq) + 3, "5S", b"ACGTA", bytes([30] * 5), 60),
            Record(0, "chr1", 20, "10M", seq[19:29].encode(), bytes([30] * 10), 60)]
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    ctx.upload_reference(ref)
    batch = ReadBatch.from_records(recs, ref)
    for how, v in views(batch):
        with pytest.raises(abi.PsError) as e:
            ctx.track(v, exclude_flags=0x100)
        assert e.value.status == abi.PS_ERR_UNSUPPORTED and e.value.fault == (po.PS_FAULT_PAST_END, 1), how


# ---- 3. errors and all-zero options ------------------------------------------------------------------------------
def _raw_call(ctx, batch, aux, fo):
    h = C.c_void_p()
    s = batch.as_struct()
    st = ctx.lib.ps_track_batch_ex3(ctx.h, C.byref(s), None, None, aux, fo, C.byref(h))
    return st, h


def test_option_errors(ctx):
    recs = random_records(random.Random(5), CONTIGS, 50)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    full = b.aux_struct()
    cases = [(None, abi.ps_track_filter_opts(10, 0, 0, 0)),
             (C.byref(abi.ps_read_aux(full.sam_flags, None)), abi.ps_track_filter_opts(10, 0, 0, 0)),
             (C.byref(abi.ps_read_aux(None, full.mapq)), abi.ps_track_filter_opts(0, 0, 0x100, 0)),
             (C.byref(abi.ps_read_aux(None, full.mapq)), abi.ps_track_filter_opts(0, 0x10, 0, 0)),
             (C.byref(full), abi.ps_track_filter_opts(0, 0, 0, 20, (C.c_uint32 * 4)(0, 0, 1, 0))),
             (C.byref(full), abi.ps_track_filter_opts(256, 0, 0, 0)),
             (C.byref(full), abi.ps_track_filter_opts(0, 0, 0, 256)),
             (C.byref(full), abi.ps_track_filter_opts(0, 0x10000, 0, 0))]
    for k, (aux, fo) in enumerate(cases):
        st, h = _raw_call(ctx, b, aux, C.byref(fo))
        assert st == abi.PS_ERR_INVALID_ARG and not h, k
    # the base filter alone needs no aux arrays
    st, h = _raw_call(ctx, b, None, C.byref(abi.ps_track_filter_opts(0, 0, 0, 20)))
    assert st == abi.PS_OK
    ctx.lib.ps_track_close(h)


def test_all_zero_options_equal_ex2(ctx):
    recs = random_records(random.Random(6), CONTIGS, 300)
    ref = PackedReference.from_contigs([(n, s.encode()) for n, s in CONTIGS])
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    want = ctx.track(b)
    st, h = _raw_call(ctx, b, None, C.byref(abi.ps_track_filter_opts()))
    assert st == abi.PS_OK
    try:
        ctr, fc = abi.ps_track_counters(), abi.ps_track_filter_counters()
        ctx.lib.ps_track_counters_get(h, C.byref(ctr))
        assert ctr.as_dict() == want["counters"]
        assert ctx.lib.ps_track_filter_counters_get(h, C.byref(fc)) == abi.PS_OK
        assert fc.as_dict() == {"filtered_flags": 0, "filtered_mapq": 0, "low_quality_bases": [0, 0]}
        for s_, k in ((0, "runs_plus"), (1, "runs_minus")):
            a = np.zeros(ctr.n_runs[s_], dtype=abi.TRACK_RUN_DTYPE)
            ctx.lib.ps_track_runs(h, s_, 0, a.ctypes.data, a.size)
            assert np.array_equal(a, want[k])
    finally:
        ctx.lib.ps_track_close(h)
    # a handle made without filter options has no filter counters
    h2 = C.c_void_p()
    s = b.as_struct()
    assert ctx.lib.ps_track_batch_ex2(ctx.h, C.byref(s), None, None, C.byref(h2)) == abi.PS_OK
    assert ctx.lib.ps_track_filter_counters_get(h2, C.byref(abi.ps_track_filter_counters())) == abi.PS_ERR_STATE
    ctx.lib.ps_track_close(h2)


# ---- 4. the file tool -------------------------------------------------------------------------------------------
FILES = ("plus.bedGraph", "minus.bedGraph", "t2c.tsv", "bases.tsv", "indels.tsv")


def _file_case(tmp_path, fmt):
    rng = random.Random(77)
    contigs = [("chrA", "".join(rng.choice("ACGT") for _ in range(70000))), ("chrB", CONTIGS[1][1])]
    recs = random_records(rng, contigs, 5000)
    # a filtered record spanning windows: a secondary 20M50000N20M near the start of chrA
    a = next(i for i, r in enumerate(recs) if r.rname == "chrA" and r.pos >= 30)
    p = recs[a].pos
    sq = contigs[0][1]
    recs.insert(a, Record(0x100, "chrA", p, "20M50000N20M", (sq[p - 1:p + 19] + sq[p + 50019:p + 50039]).encode(),
                          bytes([30] * 40), 60))
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / f"reads.{fmt}")
    write_fasta(fa, [(n, s.encode()) for n, s in contigs])
    (write_bam if fmt == "bam" else write_sam)(path, [(n, len(s)) for n, s in contigs], recs)
    return contigs, recs, fa, path


def _want(contigs, recs, flt):
    g = genome_of(contigs)
    py = to_py(recs)
    out = dict(tfo.track_bases(py, g, **flt)["files"])
    out["indels.tsv"] = tfo.track_indels(py, g, **flt)["files"]["indels.tsv"]
    return out, tfo.track(py, g, **flt)


@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_track_bam_files(tmp_path, monkeypatch, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs, fa, path = _file_case(tmp_path, fmt)
    if fmt == "sam":       # SAM writes "30" for records without a MAPQ
        recs = [Record(r.flag, r.rname, r.pos, r.cigar, r.seq, r.qual, 30 if r.mapq is None else r.mapq) for r in recs]
    want, wt = _want(contigs, recs, FULL_FILTER)
    for window in (257, 4096, 10 ** 9):
        monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
        c = Context(0)
        try:
            c.load_fasta(fa)
            ctr = c.track_bam(path, str(tmp_path / "out"), base_counts=True, indel_counts=True, **FULL_FILTER)
        finally:
            c.close()
        got = {k: open(f"{tmp_path}/out.{k}").read() for k in FILES}
        assert got == want, (fmt, window)
        assert ctr["filter_counters"] == wt["filter_counters"], (fmt, window)
        assert ctr["reads_counted"] == wt["counters"]["reads_counted"]
        assert ctr["aligned_bases"] == wt["counters"]["aligned_bases"]


def test_two_contexts(tmp_path, monkeypatch):
    import torch
    from parasuite_b200.runtime import MultiContext
    contigs, recs, fa, path = _file_case(tmp_path, "bam")
    want, wt = _want(contigs, recs, FULL_FILTER)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", "257")
    devs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() > 1 else [])
    for d in devs:
        m = MultiContext(d)
        try:
            m.load_fasta(fa)
            ctr = m.track_bam(path, str(tmp_path / "m"), base_counts=True, indel_counts=True, **FULL_FILTER)
        finally:
            m.close()
        assert {k: open(f"{tmp_path}/m.{k}").read() for k in FILES} == want, d
        assert ctr["filter_counters"] == wt["filter_counters"], d


# ---- 5. full size ---------------------------------------------------------------------------------------------
def test_config2_size(ctx):
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(0x5EED0001, [10_000_000])
    b = synth.synth_reads(ref, 10_000_000, 36, seed=0x5EED0002)
    rng = np.random.default_rng(0x5EED0003)
    n = b.n_reads
    rev = ((np.asarray(b.meta[:n]) >> np.uint32(24)) & abi.PS_RF_REVERSE) != 0
    extra = rng.choice(np.array([0, 0, 0, 0, 0x100, 0x200, 0x400, 0x800], dtype=np.uint16), size=n)
    b.sam_flags = (np.where(rev, 0x10, 0) | extra).astype(np.uint16)
    b.mapq = rng.choice(np.array([0, 3, 10, 30, 60, 255], dtype=np.uint8), size=n)
    b.qual = np.asarray(b.qual).copy()
    b.qual[:n * 36] = rng.integers(2, 41, size=n * 36, dtype=np.uint8)
    ctx.upload_reference(ref)
    exp = tfo.track_cpp(ref, b, **FULL_FILTER)
    got = ctx.track(DeviceBatch(b, "cuda:0"), **FULL_FILTER)
    _same(got, exp, "config 2")
    assert got["filter_counters"] == exp["filter_counters"]
    assert got["counters"]["fast_path_reads"] == got["counters"]["reads_counted"] > 0
