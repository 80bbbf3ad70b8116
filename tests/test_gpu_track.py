"""GPU: the per-position T>C conversion and coverage track against the C++ restatement (batches) and the Python one
(file texts), through every window size, BAM and SAM, header orders other than the FASTA's, the pileup's faults, and
against the pileup's own clusters on input without D/N."""
import random

import numpy as np
import pytest

import py_oracle as po
import track_oracle as to
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi, synth
from parasuite_b200.bamio import write_bam, write_fasta, write_sam
from test_contig_order_cpu import HEADER, header_sq, permuted_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


def _equal(got, exp, what):
    for k in ("runs_plus", "runs_minus", "sites"):
        assert got[k].dtype == exp[k].dtype and np.array_equal(got[k], exp[k]), (what, k, len(got[k]), len(exp[k]))
    for k in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events",
              "n_runs", "n_sites"):
        assert got["counters"][k] == exp["counters"][k], (what, k)


def _clean(recs, contigs):
    """drop the records the pileup would die on (one at a time, as the Python restatement finds them)"""
    g = po.Genome(dict(contigs))
    while True:
        try:
            to.track(to_py(recs), g)
            return recs
        except to.TrackFault as e:
            recs = recs[:e.ordinal] + recs[e.ordinal + 1:]


@pytest.mark.parametrize("seed", range(4))
def test_random_batches_all_cigar_kinds(ctx, seed):
    rng = random.Random(7300 + seed)
    contigs = random_genome(rng, n_contigs=3, length=4000, n_frac=0.01, lower_frac=0.1)
    recs = random_records(rng, contigs, 3000, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 150),
                          flags_special=0.03)
    recs = _clean([r for r in recs if r.pos > 0], contigs)
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    got = ctx.track(b)
    _equal(got, to.track_cpp(ref, b), f"seed {seed}")
    assert got["counters"]["fast_path_reads"] == 0


@pytest.mark.parametrize("L,ragged", [(36, False), (64, False), (17, False), (0, True)])
def test_fast_and_general_paths(ctx, L, ragged):
    rng = random.Random(7400 + L)
    contigs = random_genome(rng, n_contigs=2, length=20000, n_frac=0.005, lower_frac=0.1)
    lr = (18, 64) if ragged else (L, L)
    recs = _clean(random_records(rng, contigs, 20000, kinds=("M",), Lrange=lr, flags_special=0.02), contigs)
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    got = ctx.track(b)
    _equal(got, to.track_cpp(ref, b), f"L {L} ragged {ragged}")
    fast = got["counters"]["fast_path_reads"]
    if ragged:
        assert fast == 0
    else:
        assert fast > 0.9 * got["counters"]["reads_counted"]


def test_long_reads_past_index_51(ctx):
    rng = random.Random(7500)
    contigs = random_genome(rng, n_contigs=1, length=5000, n_frac=0.0, lower_frac=0.0)
    seq = contigs[0][1]
    recs = []
    for pos in range(1, 4000, 37):
        s = bytearray(seq[pos - 1:pos - 1 + 120].upper())
        for k in range(52, 120):
            if s[k] == ord("T"):
                s[k] = ord("C")
        recs.append(Record(0, contigs[0][0], pos, "120M", bytes(s), bytes([30] * 120)))
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    got = ctx.track(b)
    _equal(got, to.track_cpp(ref, b), "long reads")
    assert got["counters"]["t2c_events"][0] > 1000
    with pytest.raises(abi.ReferenceWouldThrow):          # the pileup refuses the same batch
        ctx.pileup(b)


def test_config2_million(ctx):
    ref = synth.synth_reference(0x5EED0001, [10_000_000])
    b = synth.synth_reads(ref, 1_000_000, 36, seed=0x5EED0002)
    ctx.upload_reference(ref)
    got = ctx.track(b)
    _equal(got, to.track_cpp(ref, b), "config2 1M")
    assert got["counters"]["fast_path_reads"] == got["counters"]["reads_counted"] > 0


# ---- file tool -------------------------------------------------------------------------------------------------------
def _texts(prefix):
    return {k: open(f"{prefix}.{k}").read() for k in ("plus.bedGraph", "minus.bedGraph", "t2c.tsv")}


@pytest.mark.parametrize("window", [10 ** 9, 700, 97, 1])
@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_track_bam_files(tmp_path, monkeypatch, window, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(63, n=1500, kinds=("M", "M", "clip", "indel", "splice"))
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / f"reads.{fmt}")
    write_fasta(fa, contigs)
    (write_bam if fmt == "bam" else write_sam)(path, header_sq(contigs), recs)
    want = to.track(to_py(recs), po.Genome(dict(contigs)), [contigs[c][0] for c in HEADER])
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
    c = Context(0)
    try:
        c.load_fasta(fa)
        ctr = c.track_bam(path, str(tmp_path / "out"))
    finally:
        c.close()
    assert _texts(tmp_path / "out") == want["files"]
    assert ctr["n_sites"] == want["counters"]["n_sites"] and ctr["n_runs"] == want["counters"]["n_runs"]
    assert ctr["reads_counted"] == want["counters"]["reads_counted"]


def test_config1_fixture_two_windows(tmp_path, monkeypatch):
    """the config-1 records (N-spliced reads included) give the same files at two window sizes"""
    import gzip
    import json
    import os
    from parasuite_b200.runtime import Context
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config1")
    raw, fa = str(tmp_path / "raw.fa"), str(tmp_path / "ref.fa")
    open(raw, "wb").write(gzip.open(os.path.join(d, "reference_chr1.fa.gz")).read())
    contigs = _fasta(raw)
    write_fasta(fa, contigs)
    recs = [Record(f, rn, p, c, s.encode(), bytes(q)) for f, rn, p, c, s, q in
            json.loads(gzip.open(os.path.join(d, "reads.json.gz"), "rb").read())]
    recs = _clean(recs, contigs)
    path = str(tmp_path / "reads.bam")
    write_bam(path, [(n, len(s)) for n, s in contigs], recs)
    want = to.track(to_py(recs), po.Genome(dict(contigs)))["files"]
    c = Context(0)
    try:
        c.load_fasta(fa)
        for w in (10 ** 9, 333):
            monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(w))
            c.track_bam(path, str(tmp_path / f"o{w}"))
            assert _texts(tmp_path / f"o{w}") == want, w
    finally:
        c.close()


def _fasta(path):
    name, seq, out = None, [], []
    for line in open(path, "rb"):
        line = line.strip()
        if line.startswith(b">"):
            if name:
                out.append((name, b"".join(seq)))
            name, seq = line[1:].split()[0].decode(), []
        elif line:
            seq.append(line)
    if name:
        out.append((name, b"".join(seq)))
    return out


def test_file_faults_and_unsorted(tmp_path, ctx, monkeypatch):
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(64, n=600)
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs)
    # a header contig the FASTA lacks: the pileup's fault, same ordinal
    sq = header_sq(contigs)
    k = len(recs) // 2
    bad = recs[:k] + [Record(0, "chrUn", 10, "20M", b"A" * 20, bytes([30] * 20))] + recs[k:]
    bad.sort(key=lambda r: ([s[0] for s in sq].index(r.rname), r.pos))
    path = str(tmp_path / "bad.bam")
    write_bam(path, sq, bad)
    c = Context(0)
    try:
        c.load_fasta(fa)
        with pytest.raises(abi.ReferenceWouldThrow) as e_p:
            c.pileup_bam(path)
        for w in (10 ** 9, 50):
            monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(w))
            with pytest.raises(abi.ReferenceWouldThrow) as e_t:
                c.track_bam(path, str(tmp_path / "bad"))
            assert e_t.value.fault == e_p.value.fault, w
        # a start going backwards within a contig, inside a window and across windows
        back = list(recs)
        j = next(i for i in range(200, len(back)) if back[i].rname == back[i - 1].rname and back[i].pos > back[i - 1].pos + 2)
        back[j - 1], back[j] = back[j], back[j - 1]
        path = str(tmp_path / "back.bam")
        write_bam(path, sq, back)
        for w in (10 ** 9, j):
            monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(w))
            with pytest.raises(abi.PsError) as e:
                c.track_bam(path, str(tmp_path / "back"))
            assert e.value.status == abi.PS_ERR_UNSORTED, w
    finally:
        c.close()


def test_cigar_ops_fault_like_the_pileup(ctx):
    rng = random.Random(7600)
    contigs = random_genome(rng, n_contigs=1, length=3000, n_frac=0.0, lower_frac=0.0)
    recs = _clean(random_records(rng, contigs, 300, kinds=("M",), Lrange=(30, 30)), contigs)
    cg = "1M1I" * 130 + "10M"
    recs[150] = Record(0, contigs[0][0], recs[150].pos, cg, b"A" * 270, bytes([30] * 270))
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    with pytest.raises(abi.PsError) as e_p:
        ctx.pileup(b)
    with pytest.raises(abi.PsError) as e_t:
        ctx.track(b)
    assert e_p.value.status == e_t.value.status == abi.PS_ERR_UNSUPPORTED
    assert e_t.value.fault == (abi.PS_FAULT_CIGAR_OPS, 150)


def test_cross_check_with_the_pileup(ctx):
    """No D/N: the pileup's checkPosition and the genomic walk coincide.  For every cluster whose span overlaps no
    neighbour's, its sites are the track's plus + minus at those positions."""
    rng = random.Random(7700)
    contigs = random_genome(rng, n_contigs=2, length=60000, n_frac=0.005, lower_frac=0.1)    # sparse: most clusters
    recs = _clean(random_records(rng, contigs, 2500, kinds=("M", "clip"), Lrange=(18, 45)), contigs)   # stand alone
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    tr = ctx.track(b)
    pl = ctx.pileup(b)
    cov = {}
    for s, name in ((0, "runs_plus"), (1, "runs_minus")):
        for x in tr[name]:
            for p in range(int(x["start0"]) + 1, int(x["end0"]) + 1):
                cov[(int(x["contig"]), p)] = cov.get((int(x["contig"]), p), 0) + int(x["cov"])
    t2c = {}
    for x in tr["sites"]:
        t2c[(int(x["contig"]), int(x["pos"]))] = t2c.get((int(x["contig"]), int(x["pos"])), 0) + int(x["t2c"])
    clusters = [(c, pl["sites"][int(c["site_begin"]):int(c["site_end"])]) for c in pl["clusters"]]
    if pl["open_cluster"] is not None:
        clusters.append((pl["open_cluster"], pl["open_sites"]))
    spans = [(int(c["contig"]), int(c["start"]), int(c["end"])) for c, _ in clusters]
    checked = 0
    for i, (c, sites) in enumerate(clusters):
        ci, lo, hi = spans[i]
        if any(j != i and s[0] == ci and s[1] <= hi and lo <= s[2] for j, s in enumerate(spans)):
            continue
        got = {int(s["pos"]) for s in sites}
        for s in sites:
            assert int(s["t2c"]) == t2c.get((ci, int(s["pos"])), 0)
            assert int(s["cov"]) == cov.get((ci, int(s["pos"])), 0)
        assert {p for (cc, p) in t2c if cc == ci and lo <= p <= hi} <= got
        checked += 1
    assert checked > 500


def test_two_devices_match_one(tmp_path, monkeypatch):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from parasuite_b200.runtime import Context, MultiContext
    contigs, recs = permuted_records(65, n=1500, kinds=("M", "clip", "splice"))
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / "reads.bam")
    write_fasta(fa, contigs)
    write_bam(path, header_sq(contigs), recs)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", "211")
    c = Context(0)
    try:
        c.load_fasta(fa)
        c.track_bam(path, str(tmp_path / "one"))
    finally:
        c.close()
    m = MultiContext([0, 1])
    try:
        m.load_fasta(fa)
        m.track_bam(path, str(tmp_path / "two"))
    finally:
        m.close()
    assert _texts(tmp_path / "one") == _texts(tmp_path / "two")
