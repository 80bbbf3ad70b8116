"""GPU: the track's per-position base counts (ps_track_opts.base_counts) against the restatements of
tests/track_bases_oracle.py, bit for bit: batches through the host, device and misaligned views (the last one takes
the per-base path), every length arm of the bit-parallel path, thresholds and masks, config 2 at 1 M reads, the file
tool at several window sizes on one and two contexts, and faults.  With the option off, or beside it, the track's own
outputs are unchanged."""
import ctypes as C
import random

import numpy as np
import pytest

import py_oracle as po
import track_bases_oracle as tb
import track_oracle as to
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi, synth
from parasuite_b200.bamio import write_bam, write_fasta, write_sam
from parasuite_b200.runtime import substitution_mask
from test_contig_order_cpu import HEADER, header_sq, permuted_records

pytestmark = pytest.mark.gpu

T2C = substitution_mask(["T>C"])
MASKS = {"all": 0, "T>C": T2C, "G>A": substitution_mask(["G>A"]), "A>G|T>C": substitution_mask(["A>G", "T>C"])}


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


def _clean(recs, contigs):
    g = po.Genome(dict(contigs))
    while True:
        try:
            to.track(to_py(recs), g)
            return recs
        except to.TrackFault as e:
            recs = recs[:e.ordinal] + recs[e.ordinal + 1:]


def _same_track(got, exp, what):
    for k in ("runs_plus", "runs_minus", "sites"):
        assert got[k].dtype == exp[k].dtype and np.array_equal(got[k], exp[k]), (what, k)
    for k in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events",
              "n_runs", "n_sites"):
        assert got["counters"][k] == exp["counters"][k], (what, k)


def check(ctx, ref, batch, what, fast=None, **kw):
    """every view against track_bases_cpp; fast: the batch is uniform and takes the bit-parallel path"""
    exp = tb.track_bases_cpp(ref, batch, **kw)
    ctx.upload_reference(ref)
    for how, v in views(batch):
        got = ctx.track(v, base_counts=True, min_coverage=kw.get("min_coverage", 1),
                        min_events=kw.get("min_events", 1), substitutions=_subs(kw.get("substitutions", 0)))
        _same_track(got, exp, (what, how))
        assert got["base_rows"].dtype == exp["base_rows"].dtype
        assert np.array_equal(got["base_rows"], exp["base_rows"]), (what, how, got["base_rows"].size, exp["base_rows"].size)
        assert np.array_equal(got["base_totals"], exp["base_totals"]), (what, how)
        c = got["counters"]
        if fast and how != "misaligned":
            assert c["fast_path_reads"] > 0.9 * c["reads_counted"], (what, how)
        if how == "misaligned":
            assert c["fast_path_reads"] == 0
    return exp


def _subs(mask):
    """the "X>Y" list of a mask (None: all)"""
    if not mask:
        return None
    return [f"{'ACGT'[b >> 2]}>{'ACGT'[b & 3]}" for b in range(16) if (mask >> b) & 1 and b >> 2 != b & 3]


def _random_ns(rng, recs, every=5):
    for r in recs[::every]:
        s = bytearray(r.seq)
        for _ in range(rng.randint(1, 3)):
            s[rng.randrange(len(s))] = ord("N")
        r.seq = bytes(s)
    return recs


def _scramble_listed_codes(batch, rng):
    """arbitrary 2-bit codes under the listed N calls of a uniform batch (the producer may store any)"""
    L = batch.uniform_len
    stride = (L + 3) // 4
    te = np.asarray(batch.tile_exc_off)
    exc = np.asarray(batch.exc)
    for t in range(te.size - 1):
        for e in exc[te[t]:te[t + 1]]:
            r, p = t * abi.PS_TILE_READS + (int(e) >> 16), int(e) & 0xFFFF
            i = r * stride + p // 4
            batch.bases2[i] = (int(batch.bases2[i]) & ~(3 << (2 * (p % 4)))) | (rng.randrange(4) << (2 * (p % 4)))
    return batch


# ---- 1. the option off ---------------------------------------------------------------------------------------------
def test_option_off_and_beside(ctx):
    rng = random.Random(8100)
    contigs = random_genome(rng, n_contigs=2, length=6000, n_frac=0.01, lower_frac=0.1)
    recs = _clean(_random_ns(rng, random_records(rng, contigs, 4000, kinds=("M", "clip", "indel", "splice"),
                                                 Lrange=(20, 80), flags_special=0.03)), contigs)
    ref = PackedReference.from_contigs(contigs)
    ctx.upload_reference(ref)
    b = ReadBatch.from_records(recs, ref)
    plain = ctx.track(b)
    on = ctx.track(b, base_counts=True)
    assert set(plain) == {"runs_plus", "runs_minus", "sites", "counters"}
    _same_track(on, plain, "beside")
    assert on["counters"] == plain["counters"]
    lib = ctx.lib
    s = b.as_struct()
    for opts in (None, abi.ps_track_opts(0, 5, 5, T2C)):          # _ex with the option off is the plain call
        h = C.c_void_p()
        assert lib.ps_track_batch_ex(ctx.h, C.byref(s), C.byref(opts) if opts else None, C.byref(h)) == abi.PS_OK
        ctr = abi.ps_track_counters()
        lib.ps_track_counters_get(h, C.byref(ctr))
        assert ctr.as_dict() == plain["counters"]
        assert lib.ps_track_base_rows(h, 0, None, 0) == abi.PS_ERR_STATE
        assert lib.ps_track_base_totals_get(h, C.byref(abi.ps_track_base_totals())) == abi.PS_ERR_STATE
        lib.ps_track_close(h)
    h = C.c_void_p()
    bad = abi.ps_track_opts(1, 1, 1, 1 << 16)
    assert lib.ps_track_batch_ex(ctx.h, C.byref(s), C.byref(bad), C.byref(h)) == abi.PS_ERR_INVALID_ARG
    assert not h.value


# ---- 2. batches against track_cpp with base counts -----------------------------------------------------------------
@pytest.mark.parametrize("seed", range(3))
def test_random_batches_all_cigar_kinds(ctx, seed):
    rng = random.Random(8200 + seed)
    contigs = random_genome(rng, n_contigs=3, length=4000, n_frac=0.02, lower_frac=0.1)
    recs = random_records(rng, contigs, 3000, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 150),
                          err=0.05, flags_special=0.03)
    recs = _clean(_random_ns(rng, [r for r in recs if r.pos > 0]), contigs)
    ref = PackedReference.from_contigs(contigs)
    check(ctx, ref, ReadBatch.from_records(recs, ref), f"random {seed}")


@pytest.mark.parametrize("L", [1, 15, 16, 17, 32, 33, 36, 48, 49, 63, 64, 65])
def test_uniform_lengths(ctx, L):
    rng = random.Random(8300 + L)
    contigs = random_genome(rng, n_contigs=2, length=8000, n_frac=0.01, lower_frac=0.1)
    recs = _clean(_random_ns(rng, random_records(rng, contigs, 8000, kinds=("M",), Lrange=(L, L), err=0.05,
                                                 flags_special=0.02), every=4), contigs)
    ref = PackedReference.from_contigs(contigs)
    b = _scramble_listed_codes(ReadBatch.from_records(recs, ref), rng)
    assert b.uniform_len == L and b.exc_count > 0
    check(ctx, ref, b, f"L {L}", fast=L <= 64)


def test_ragged(ctx):
    rng = random.Random(8400)
    contigs = random_genome(rng, n_contigs=2, length=8000, n_frac=0.01, lower_frac=0.1)
    recs = _clean(_random_ns(rng, random_records(rng, contigs, 6000, kinds=("M",), Lrange=(18, 64), err=0.05)), contigs)
    ref = PackedReference.from_contigs(contigs)
    check(ctx, ref, ReadBatch.from_records(recs, ref), "ragged")


def test_contig_ends_and_reference_n(ctx):
    """reads flush with both ends of every contig, and reads over runs of reference N"""
    rng = random.Random(8500)
    L = 36
    contigs = []
    for c in range(3):
        s = bytearray(rng.choice(b"ACGT") for _ in range(300 + 17 * c))
        s[100:130] = b"N" * 30
        s[200:210] = bytes(s[200:210]).lower()
        contigs.append((f"chr{c + 1}", bytes(s)))
    recs = []
    for name, seq in contigs:
        starts = sorted([1, len(seq) - L + 1] + [rng.randint(1, len(seq) - L + 1) for _ in range(200)] + [85, 95, 125])
        for p in starts:
            rd = bytearray(seq[p - 1:p - 1 + L].upper().replace(b"N", b"A"))
            for k in range(L):
                if rng.random() < 0.1:
                    rd[k] = rng.choice(b"ACGTN")
            if p == len(seq) - L + 1:            # an event on the contig's last base
                rd[-1] = b"CAAA"[b"ACGT".index(rd[-1])] if rd[-1] in b"ACGT" else ord("A")
            recs.append(Record(16 if rng.random() < 0.5 else 0, name, p, f"{L}M", bytes(rd), bytes([30] * L)))
    ref = PackedReference.from_contigs(contigs)
    b = _scramble_listed_codes(ReadBatch.from_records(recs, ref), rng)
    exp = check(ctx, ref, b, "ends and N", fast=True)
    last = exp["base_rows"][exp["base_rows"]["contig"] == 2]
    assert int(last["pos"].max()) == len(contigs[2][1])


def test_more_than_65536_events_at_one_position(ctx):
    """70 000 reads on each strand convert the same position (T>C on the read's strand) and carry a second substitution"""
    seq = bytearray(b"ACGTACGTAC" * 20)
    seq[59], seq[61] = ord("T"), ord("A")          # positions 60 (plus: T) and 62 (minus: ref A = T on the read)
    contigs = [("chr1", bytes(seq))]
    plus = bytearray(seq[50:70])
    plus[9], plus[3] = ord("C"), ord("G") if plus[3] != ord("G") else ord("T")
    minus = bytearray(seq[50:70])
    minus[11], minus[5] = ord("G"), ord("C") if minus[5] != ord("C") else ord("A")
    n = 70_000
    recs = [Record(0, "chr1", 51, "20M", bytes(plus), bytes([30] * 20)) for _ in range(n)]
    recs += [Record(16, "chr1", 51, "20M", bytes(minus), bytes([30] * 20)) for _ in range(n)]
    ref = PackedReference.from_contigs(contigs)
    exp = check(ctx, ref, ReadBatch.from_records(recs, ref), "65536", fast=True)
    rows = exp["base_rows"]
    hit = rows[(rows["pos"] == 60) & (rows["strand"] == 0)]
    assert hit.size == 1 and int(hit["n"][0][1]) == n
    hit = rows[(rows["pos"] == 62) & (rows["strand"] == 1)]
    assert hit.size == 1 and int(hit["ref"][0]) == 3 and int(hit["n"][0][1]) == n


# ---- 3. thresholds and masks ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("mask", sorted(MASKS))
def test_thresholds(ctx, mask):
    rng = random.Random(8600)
    contigs = random_genome(rng, n_contigs=2, length=3000, n_frac=0.01, lower_frac=0.1)
    recs = _clean(_random_ns(rng, random_records(rng, contigs, 6000, kinds=("M", "clip", "indel"), Lrange=(36, 36),
                                                 err=0.08)), contigs)
    ref = PackedReference.from_contigs(contigs)
    b = ReadBatch.from_records(recs, ref)
    sizes = []
    for mc, me in ((0, 0), (1, 1), (5, 1), (1, 2), (20, 3), (60, 5), (10 ** 6, 1)):
        exp = check(ctx, ref, b, (mask, mc, me), substitutions=MASKS[mask], min_coverage=mc, min_events=me)
        sizes.append(exp["base_rows"].size)
        if mask == "T>C" and me <= 1 and mc <= 1:
            assert np.array_equal(exp["base_rows"]["n"][:, 1], exp["sites"]["t2c"])
    assert sizes[0] == sizes[1] > 0 and sizes[1] >= sizes[2] and sizes[1] >= sizes[3] and sizes[-1] == 0


# ---- 4. config 2 at 1 M reads --------------------------------------------------------------------------------------
def test_config2_million(ctx):
    ref = synth.synth_reference(0x5EED0001, [10_000_000])
    b = synth.synth_reads(ref, 1_000_000, 36, seed=0x5EED0002)
    ctx.upload_reference(ref)
    from parasuite_b200.runtime import DeviceBatch
    exp = tb.track_bases_cpp(ref, b)
    got = ctx.track(DeviceBatch(b, "cuda:0"), base_counts=True)
    _same_track(got, exp, "config 2")
    assert np.array_equal(got["base_rows"], exp["base_rows"]) and np.array_equal(got["base_totals"], exp["base_totals"])
    c, tot, rows = got["counters"], got["base_totals"], got["base_rows"]
    assert c["fast_path_reads"] == c["reads_counted"] > 0
    assert [int(tot[s, 3, 1]) for s in (0, 1)] == c["t2c_events"]
    assert np.array_equal(rows["n"].sum(axis=1), rows["cov"])
    assert int(tot.sum()) <= sum(c["aligned_bases"]) and int(tot[:, :, 4].sum()) > 0
    sub = ctx.track(DeviceBatch(b, "cuda:0"), base_counts=True, substitutions=["T>C"])["base_rows"]
    assert np.array_equal(sub["pos"], got["sites"]["pos"]) and np.array_equal(sub["n"][:, 1], got["sites"]["t2c"])


# ---- 5. the file tool ----------------------------------------------------------------------------------------------
def _texts(prefix, bases=True):
    ks = ("plus.bedGraph", "minus.bedGraph", "t2c.tsv") + (("bases.tsv",) if bases else ())
    return {k: open(f"{prefix}.{k}").read() for k in ks}


def _file_case(tmp_path, fmt):
    contigs, recs = permuted_records(65, n=1500, kinds=("M", "M", "clip", "indel", "splice"))
    rng = random.Random(8700)
    recs = _random_ns(rng, recs, every=6)
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / f"reads.{fmt}")
    write_fasta(fa, contigs)
    (write_bam if fmt == "bam" else write_sam)(path, header_sq(contigs), recs)
    order = [contigs[c][0] for c in HEADER]
    return contigs, recs, fa, path, order


@pytest.mark.parametrize("window", [10 ** 9, 700, 97, 1])
@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_track_bam_files(tmp_path, monkeypatch, window, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs, fa, path, order = _file_case(tmp_path, fmt)
    g = po.Genome(dict(contigs))
    want = tb.track_bases(to_py(recs), g, order, min_events=2, substitutions=0)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
    c = Context(0)
    try:
        c.load_fasta(fa)
        plain = c.track_bam(path, str(tmp_path / "plain"))
        ctr = c.track_bam(path, str(tmp_path / "out"), base_counts=True, min_events=2)
    finally:
        c.close()
    assert _texts(tmp_path / "out") == want["files"]
    assert _texts(tmp_path / "plain", bases=False) == {k: v for k, v in want["files"].items() if k != "bases.tsv"}
    assert not (tmp_path / "plain.bases.tsv").exists()
    assert {k: v for k, v in ctr.items() if k not in ("base_totals", "n_base_rows")} == plain
    assert np.array_equal(ctr["base_totals"], want["base_totals"])
    assert ctr["n_base_rows"] == len(want["base_rows"]) > 0


def test_two_contexts(tmp_path, monkeypatch):
    import torch
    from parasuite_b200.runtime import MultiContext
    contigs, recs, fa, path, order = _file_case(tmp_path, "bam")
    want = tb.track_bases(to_py(recs), po.Genome(dict(contigs)), order, substitutions=MASKS["A>G|T>C"])
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", "211")
    devs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() > 1 else [])
    for d in devs:
        m = MultiContext(d)
        try:
            m.load_fasta(fa)
            ctr = m.track_bam(path, str(tmp_path / "m"), base_counts=True, substitutions=["A>G", "T>C"])
        finally:
            m.close()
        assert _texts(tmp_path / "m") == want["files"], d
        assert np.array_equal(ctr["base_totals"], want["base_totals"]), d


# ---- 6. faults ----------------------------------------------------------------------------------------------------
def _outcome(fn):
    try:
        return ("ok", fn())
    except abi.PsError as e:
        return (e.status, e.fault)


def test_faults_match_the_plain_track(ctx):
    rng = random.Random(8800)
    contigs = random_genome(rng, n_contigs=2, length=3000, n_frac=0.0, lower_frac=0.0)
    recs = _clean(random_records(rng, contigs, 400, kinds=("M",), Lrange=(30, 30)), contigs)
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
        "unsorted": recs[:50] + [recs[300]] + recs[50:],
    }
    for what, rs in cases.items():
        b = ReadBatch.from_records(rs, ref)
        for how, v in views(b):
            plain = _outcome(lambda: ctx.track(v))
            based = _outcome(lambda: ctx.track(v, base_counts=True))
            assert plain[0] != "ok" and plain == based, (what, how, plain, based)
        # the handle of a faulting call carries no base rows
        h = C.c_void_p()
        s = b.as_struct()
        opts = abi.ps_track_opts(1, 1, 1, 0)
        st = ctx.lib.ps_track_batch_ex(ctx.h, C.byref(s), C.byref(opts), C.byref(h))
        assert st != abi.PS_OK
        if h.value:
            assert ctx.lib.ps_track_base_rows(h, 0, None, 0) == 0
            tot = abi.ps_track_base_totals()
            assert ctx.lib.ps_track_base_totals_get(h, C.byref(tot)) == abi.PS_OK and tot.n_rows == 0
            ctx.lib.ps_track_close(h)
