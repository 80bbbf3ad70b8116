"""GPU: the fast profile kernel (profile_fast.cuh) at its edges, bit for bit against the C++ oracle.

* every length arm (compile-time L = 32, 36, 40, 50, 51 and the run-time instantiations nw = 1..4) against
  maxReadLength L - 1, L, 51, 256 (the last value the fast kernel takes) and 257 (the first on the warp-per-read kernel),
  with -q wherever maxReadLength <= 64;
* quality bytes over the whole byte range: Java sums them as signed bytes (ErrorProfiling.java:301), the -q histogram
  counts them by byte value;
* the T>C mask words handed to the pileup, word by word;
* batches split over several launches of the fast kernel (PARASUITE_B200_FAST_READS_PER_BLOCK shortens the split).

The debug word 1 (reads the fast kernels took) shows that each case ran the arm it names."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import assert_profile_equal
from parasuite_b200 import PackedReference, ReadBatch, abi
from test_gpu_fused import check_mask_words, mask_words
from test_gpu_pileup import assert_pileup_equal

pytestmark = pytest.mark.gpu

OP_M, OP_EQ, OP_X = 0, 7, 8
LENGTHS = [1, 7, 15, 16, 17, 31, 32, 33, 36, 40, 47, 48, 49, 50, 51, 62, 63, 64]
SHORTER_MAX_LEN = {7, 17, 36, 50, 64}          # lengths also run with maxReadLength = L - 1


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    c.lib.ps_debug_word.restype = C.c_ulonglong
    c.lib.ps_debug_word.argtypes = [C.c_void_p, C.c_int]
    yield c
    c.close()


# ---- inputs -------------------------------------------------------------------------------------------------------
_CODE = np.full(256, 255, dtype=np.uint8)
for _ch, _v in zip(b"ACGTacgt", (0, 1, 2, 3, 0, 1, 2, 3)):
    _CODE[_ch] = _v


def make_reference(seed, lengths):
    """Random contigs with N runs, stray IUPAC codes and lower-case stretches; returns (PackedReference, codes) where
    codes holds 255 at invalid positions."""
    rng = np.random.default_rng(seed)
    n = int(sum(lengths))
    raw = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].copy()
    for s in rng.integers(0, n - 40, size=max(1, n // 4000)):
        raw[s:s + int(rng.integers(1, 25))] = ord("N")
    raw[rng.integers(0, n, size=max(1, n // 3000))] = ord("R")
    for s in rng.integers(0, n - 200, size=max(1, n // 20000)):
        raw[s:s + 200] |= 0x20                        # lower case: same codes
    raw[raw == ord("n")] = ord("N")
    raw[raw == ord("r")] = ord("R")
    ref = PackedReference.from_ascii([f"chr{k + 1}" for k in range(len(lengths))], lengths, raw)
    return ref, _CODE[raw]


def uniform_batch(ref, codes, n, L, seed, op=OP_M, special=0.02, n_call=0.004, qual=(2, 41), chunk=1 << 16):
    """A coordinate-sorted uniform batch of n single-op `L op` reads in clusters (+ two reads flush with each end of
    every contig, one per strand): sequencing errors, T>C (plus) / A>G (minus, forward view) conversions, N calls, duplicates,
    unmapped and POS-0 records (they keep their start, as the synthetic generator's do).  Qualities drawn from
    qual[0]..qual[1]."""
    rng = np.random.default_rng(seed)
    T = abi.PS_TILE_READS
    lens = np.asarray(ref.lengths, dtype=np.int64)
    off = ref.contig_off.astype(np.int64)
    # clusters of about 20 reads, starts within a few bases of the cluster's (what the pileup sees in PAR-CLIP data)
    k = max(1, n // 20)
    ci = rng.choice(len(lens), size=k, p=lens / lens.sum())
    centre = (rng.random(k) * (lens[ci] - L + 1)).astype(np.int64)
    which = rng.integers(0, k, size=n)
    starts = off[ci[which]] + np.clip(centre[which] + rng.integers(-3, 4, size=n), 0, lens[ci[which]] - L)
    flush = np.concatenate([[off[k], off[k], off[k + 1] - L, off[k + 1] - L] for k in range(len(lens))])
    starts = np.sort(np.concatenate((starts, flush)), kind="stable")
    n = starts.size
    rev = rng.random(n) < 0.5
    rev[np.isin(starts, flush)] = np.resize([False, True], int(np.isin(starts, flush).sum()))
    flags = np.where(rev, abi.PS_RF_REVERSE, 0).astype(np.uint32)
    sp = rng.random(n) < special
    flags[sp] |= np.array([abi.PS_RF_DUPLICATE, abi.PS_RF_UNMAPPED, abi.PS_RF_POS_ZERO],
                          dtype=np.uint32)[rng.integers(0, 3, size=int(sp.sum()))]
    bpr = (L + 3) // 4
    bases = np.zeros(n * bpr + 64, dtype=np.uint8)
    quals = np.zeros(n * L + 64, dtype=np.uint8)
    exc_read, exc_pos = [], []
    for a in range(0, n, chunk):                   # bounded temporaries for batches of millions of reads
        b = min(n, a + chunk)
        m = b - a
        c = codes[starts[a:b, None] + np.arange(L)[None, :]].astype(np.int64)
        c = np.where(c == 255, rng.integers(0, 4, size=c.shape), c)
        u = rng.random(c.shape)
        r = rev[a:b, None]
        c = np.where(u < 0.02, rng.integers(0, 4, size=c.shape), c)
        c = np.where((u > 0.9) & ~r & (c == 3), 1, c)           # T>C on the plus strand
        c = np.where((u > 0.9) & r & (c == 0), 2, c)            # A>G in the forward view of a minus-strand read
        nc = rng.random(c.shape) < n_call
        c[nc] = 0
        rr, pp = np.nonzero(nc)                   # row-major: sorted by (read, position)
        exc_read.append(rr + a)
        exc_pos.append(pp)
        pad = np.zeros((m, bpr * 4), dtype=np.int64)
        pad[:, :L] = c
        p4 = pad.reshape(m, bpr, 4)
        bases[a * bpr:b * bpr] = (p4[:, :, 0] | (p4[:, :, 1] << 2) | (p4[:, :, 2] << 4) | (p4[:, :, 3] << 6)).reshape(-1)
        quals[a * L:b * L] = rng.integers(qual[0], qual[1] + 1, size=m * L)
    exc_read = np.concatenate(exc_read)
    exc_pos = np.concatenate(exc_pos)
    flags[np.unique(exc_read)] |= abi.PS_RF_HAS_INVALID
    meta = (np.uint32(L) | np.uint32(1 << 16) | (flags << np.uint32(24))).astype(np.uint32)
    nt = (n + T - 1) // T
    edges = np.minimum(np.arange(nt + 1, dtype=np.int64) * T, n)
    teo = np.searchsorted(exc_read, edges).astype(np.uint32)
    exc = (((exc_read % T) << 16) | exc_pos).astype(np.uint32)
    return ReadBatch(n, meta, starts.astype(np.uint32), bases, quals,
                     np.concatenate((np.full(n, (L << 4) | op, dtype=np.uint32), np.zeros(16, np.uint32))),
                     (edges * bpr).astype(np.uint64), (edges * L).astype(np.uint64), edges.astype(np.uint64), teo,
                     np.concatenate((exc, np.zeros(16, np.uint32))), uniform_len=L, uniform_ncigar=1,
                     bases_bytes=n * bpr, qual_bytes=n * L, cigar_count=n, exc_count=int(exc.size))


def pos_zero_unmapped(batch):
    """The same batch with POS-0 records marked unmapped: a mapped record at POS 0 kills the JVM in the pileup loop."""
    meta = batch.meta.copy()
    pz = ((meta >> np.uint32(24)) & abi.PS_RF_POS_ZERO) != 0
    meta[pz] |= np.uint32(abi.PS_RF_UNMAPPED << 24)
    return ReadBatch(batch.n_reads, meta, batch.ref_start, batch.bases2, batch.qual, batch.cigar, batch.tile_base_off,
                     batch.tile_qual_off, batch.tile_cigar_off, batch.tile_exc_off, batch.exc,
                     uniform_len=batch.uniform_len, uniform_ncigar=batch.uniform_ncigar, bases_bytes=batch.bases_bytes,
                     qual_bytes=batch.qual_bytes, cigar_count=batch.cigar_count, exc_count=batch.exc_count)


def fast_shaped(batch, max_len):
    """Reads the fast kernel can take: single M op, no flag but strand / N calls, L <= maxReadLength."""
    n = batch.n_reads
    flags = np.asarray(batch.meta[:n]) >> np.uint32(24)
    ok = (flags & ~np.uint32(abi.PS_RF_REVERSE | abi.PS_RF_HAS_INVALID)) == 0
    ok &= (np.asarray(batch.cigar[:n]) & 15) == OP_M
    return ok & ((np.asarray(batch.meta[:n]) & 0xFFFF) <= max_len)


def contig_boundaries(ref, batch, sel):
    contig = np.searchsorted(ref.contig_off, np.asarray(batch.ref_start[:batch.n_reads]), side="right") - 1
    return int(np.count_nonzero(np.diff(contig[sel]) != 0))


_REF = {}
_BATCHES = {}


def edge_reference():
    if "edges" not in _REF:
        _REF["edges"] = make_reference(5, [70_000, 50_000, 30_000])
    return _REF["edges"]


def edge_batch(L):
    """One batch per length, shared by every maxReadLength / -q / mask case of that length."""
    if L not in _BATCHES:
        ref, codes = edge_reference()
        _BATCHES[L] = uniform_batch(ref, codes, 24_000, L, seed=700 + L, special=0.02)
    return _BATCHES[L]


# ---- running and comparing ----------------------------------------------------------------------------------------
def gpu_profile(ctx, ref, batch, max_len, infer_q=False, device=True):
    """(result, fast reads) or (ReferenceWouldThrow, fast reads)."""
    ctx.upload_reference(ref)
    ctx.profile_begin(max_len, infer_q)
    if device:
        from parasuite_b200.runtime import DeviceBatch
        ctx.profile_batch_device(DeviceBatch(batch, "cuda:0"), torch.cuda.current_stream().cuda_stream)
    else:
        ctx.profile_batch(batch)
    fast = int(ctx.lib.ps_debug_word(ctx.h, 1))
    try:
        return ctx.profile_end(), fast
    except abi.ReferenceWouldThrow as e:
        return e, fast


def oracle_profile(oracle, ref, batch, max_len, infer_q=False):
    try:
        return oracle.profile(ref, batch, max_len, infer_q, threads=8)
    except oracle.OracleFault as e:
        return e


def assert_same(got, exp, oracle, what, infer_q=False):
    """Equal results, or the same (code, ordinal) where the JVM would die."""
    if isinstance(exp, oracle.OracleFault):
        assert isinstance(got, abi.ReferenceWouldThrow), (what, "oracle faults", exp.code, exp.ordinal)
        assert got.fault == (exp.code, exp.ordinal), (what, got.fault, (exp.code, exp.ordinal))
        return
    assert not isinstance(got, Exception), (what, got)
    assert_profile_equal(got, exp, what)
    assert np.array_equal(got["wide"], exp["wide"]), what
    if infer_q:
        assert np.array_equal(got["quality_hist"], exp["quality_hist"]), what


def max_lens(L):
    out = sorted({L, max(L, 51), 256, 257})
    return out + [L - 1] if L in SHORTER_MAX_LEN else out


MATRIX = [(L, m, q) for L in LENGTHS for m in max_lens(L) for q in ((False, True) if m <= 64 else (False,))]


@pytest.mark.parametrize("L,max_len,infer_q", MATRIX)
def test_length_and_max_read_length(ctx, oracle, L, max_len, infer_q):
    ref, _ = edge_reference()
    batch = edge_batch(L)
    exp = oracle_profile(oracle, ref, batch, max_len, infer_q)
    got, fast = gpu_profile(ctx, ref, batch, max_len, infer_q)
    what = f"L {L} maxReadLength {max_len} -q {infer_q}"
    assert_same(got, exp, oracle, what, infer_q)
    shaped = fast_shaped(batch, max_len)
    if max_len < L:
        # every read fails the kernel's length test and goes to the deferred kernel, which reports the JVM's fault
        assert fast == 0 and isinstance(exp, oracle.OracleFault), what
    elif max_len > 256:
        assert fast == 0, (what, "the warp-per-read kernel takes maxReadLength > 256")
    else:
        assert fast <= shaped.sum() and fast >= shaped.sum() - 64 * contig_boundaries(ref, batch, shaped), (what, fast)
        assert not isinstance(exp, oracle.OracleFault), what


# ---- full-range qualities -----------------------------------------------------------------------------------------
FULL = (0, 254)                                   # 0xFF as the first byte would mean "no qualities"


@pytest.mark.parametrize("infer_q", [False, True])
@pytest.mark.parametrize("L", [36, 47])
def test_full_range_qualities_uniform(ctx, oracle, L, infer_q):
    """Compile-time (36) and run-time (47) length: dp4a.s32 sums, signed mismatch / invalid-position corrections, the
    -q histogram by byte value.  The same batch through the compact host form, which cannot pack such qualities."""
    from parasuite_b200.runtime import PinnedBatch
    ref, codes = edge_reference()
    batch = uniform_batch(ref, codes, 30_000, L, seed=900 + L, qual=FULL)
    exp = oracle_profile(oracle, ref, batch, 51, infer_q)
    got, fast = gpu_profile(ctx, ref, batch, 51, infer_q)
    assert_same(got, exp, oracle, f"full-range qualities L {L} -q {infer_q}", infer_q)
    assert fast > 0.9 * batch.n_reads
    pinned = PinnedBatch(batch, compact=True)
    assert pinned.compact and not pinned.packed_qual
    got_c, fast_c = gpu_profile(ctx, ref, pinned, 51, infer_q, device=False)
    assert_same(got_c, exp, oracle, f"compact host form L {L} -q {infer_q}", infer_q)
    assert fast_c == fast


@pytest.mark.parametrize("infer_q", [False, True])
@pytest.mark.parametrize("S", [16, 32, 48, 64])
def test_full_range_qualities_ragged(ctx, oracle, S, infer_q):
    """Trimmed reads re-laid into rows of S positions (the RG instantiations)."""
    from parasuite_b200 import synth
    ref, codes = edge_reference()
    batch = synth.trim_uniform(uniform_batch(ref, codes, 30_000, S, seed=950 + S, qual=FULL), max(1, S - 20), seed=S)
    assert batch.uniform_len == 0 and batch.max_len == S
    exp = oracle_profile(oracle, ref, batch, S, infer_q)
    got, fast = gpu_profile(ctx, ref, batch, S, infer_q, device=False)
    assert_same(got, exp, oracle, f"full-range qualities ragged S {S} -q {infer_q}", infer_q)
    assert fast > 0.9 * batch.n_reads


@pytest.mark.parametrize("infer_q", [False, True])
def test_full_range_qualities_warp_per_read(ctx, oracle, infer_q):
    """150-nt reads with clips, indels and =/X blocks: the warp-per-read kernel's (signed char) sums and its -q."""
    import random
    from helpers import random_genome, random_records
    from parasuite_b200 import Record
    rng = random.Random(150)
    contigs = random_genome(rng, n_contigs=2, length=20_000, n_frac=0.002, lower_frac=0.05)
    recs = random_records(rng, contigs, 1500, kinds=("M", "clip", "indel", "wild"), Lrange=(120, 150), flags_special=0.02)
    recs = [Record(r.flag, r.rname, r.pos, r.cigar, r.seq, bytes(rng.randint(*FULL) for _ in r.seq)) for r in recs]
    ref = PackedReference.from_contigs(contigs)
    ok = []
    for r in recs:                       # keep what the JVM survives (C++ oracle, one record at a time)
        try:
            oracle.profile(ref, ReadBatch.from_records([r], ref), 176, infer_q)
            ok.append(r)
        except oracle.OracleFault:
            pass
    assert len(ok) > 500
    batch = ReadBatch.from_records(ok, ref)
    exp = oracle_profile(oracle, ref, batch, 176, infer_q)
    got, fast = gpu_profile(ctx, ref, batch, 176, infer_q, device=False)
    assert_same(got, exp, oracle, f"full-range qualities 150 nt -q {infer_q}", infer_q)
    assert fast == 0


@pytest.mark.parametrize("infer_q", [False, True])
def test_full_range_qualities_deferred(ctx, oracle, infer_q):
    """A uniform batch of `36=` reads: the fast kernel defers every read (its shape is L x M), the deferred kernel
    counts them with its own (signed char) sums."""
    ref, codes = edge_reference()
    batch = uniform_batch(ref, codes, 20_000, 36, seed=960, op=OP_EQ, qual=FULL)
    exp = oracle_profile(oracle, ref, batch, 51, infer_q)
    got, fast = gpu_profile(ctx, ref, batch, 51, infer_q)
    assert_same(got, exp, oracle, f"full-range qualities deferred -q {infer_q}", infer_q)
    assert fast == 0 and int(got["counters"][0]) > 0.9 * batch.n_reads


# ---- T>C mask words -----------------------------------------------------------------------------------------------
def fused(ctx, ref, batch, max_len):
    """Profile with mask words, then the pileup fed by them.  (profile result, host words or None, pileup or fault)."""
    from parasuite_b200.runtime import DeviceBatch
    ctx.upload_reference(ref)
    d = DeviceBatch(batch, "cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    ctx.profile_begin(max_len, emit_t2c_masks=True)
    ctx.profile_batch_device(d, st)
    masks = ctx.profile_masks()
    words = mask_words(masks) if masks is not None else None
    try:
        with ctx.pileup_run(d, stream=st, masks=masks) as h:
            pile = h.fetch()
    except abi.ReferenceWouldThrow as e:
        pile = e
    return ctx.profile_end(), words, pile


def assert_pileup_same(got, ref, batch, oracle, what):
    try:
        exp = oracle.pileup(ref, batch)
    except oracle.OracleFault as e:
        assert isinstance(got, abi.ReferenceWouldThrow), (what, "oracle faults", e.code, e.ordinal)
        assert got.fault == (e.code, e.ordinal), what
        return
    assert not isinstance(got, Exception), (what, got)
    assert_pileup_equal(got, exp, what)


@pytest.mark.parametrize("L", [L for L in LENGTHS if L <= 62] + [63, 64])
def test_mask_words_every_length(ctx, oracle, L):
    ref, _ = edge_reference()
    batch = pos_zero_unmapped(edge_batch(L))
    max_len = max(L, 51)
    prof, words, pile = fused(ctx, ref, batch, max_len)
    assert_profile_equal(prof, oracle.profile(ref, batch, max_len, threads=8), f"profile with masks L {L}")
    if L > 62:          # bits 62 and 63 are flags: no words for longer reads, the pileup decodes them
        assert words is None
    else:
        check_mask_words(words, ref, batch, oracle, f"L {L}")
    assert_pileup_same(pile, ref, batch, oracle, f"mask-fed pileup L {L}")


@pytest.mark.parametrize("op", [OP_EQ, OP_X])
def test_mask_words_of_eq_and_x_reads(ctx, oracle, op):
    """`36=` / `36X` reads: the profile defers them (no valid word), the pileup counts them as alignment blocks all the
    same and must decode them itself."""
    ref, codes = edge_reference()
    batch = pos_zero_unmapped(uniform_batch(ref, codes, 20_000, 36, seed=970 + op, op=op))
    prof, words, pile = fused(ctx, ref, batch, 51)
    assert_profile_equal(prof, oracle.profile(ref, batch, 51, threads=8), f"profile op {op}")
    assert words is not None and (words == 0).all()
    assert_pileup_same(pile, ref, batch, oracle, f"mask-fed pileup op {op}")
    assert int(oracle.read_t2c_masks(ref, batch).astype(bool).sum()) > 1000     # the reads do carry T>C


# ---- one batch, several launches of the fast kernel ---------------------------------------------------------------
SPLIT_READS = 1_000_000


@pytest.fixture(scope="module")
def split_ref():
    # 24 contigs: warp-tiles that straddle two contigs, and reads flush with contig ends, in every launch
    return make_reference(17, [300_000 + 7_000 * k for k in range(24)])


def split_and_whole(monkeypatch, fn):
    """fn() -> (out, kernels the profile call launched), once with the batch in one launch of the fast kernel and once
    split at 256 reads per block: (whole out, split out, extra launches)."""
    monkeypatch.delenv("PARASUITE_B200_FAST_READS_PER_BLOCK", raising=False)
    whole, n_whole = fn()
    monkeypatch.setenv("PARASUITE_B200_FAST_READS_PER_BLOCK", str(abi.PS_TILE_READS))
    split, n_split = fn()
    monkeypatch.delenv("PARASUITE_B200_FAST_READS_PER_BLOCK")
    return whole, split, n_split - n_whole


def counting_launches(ctx, fn):
    n0 = ctx.kernel_launches()
    out = fn()
    return out, ctx.kernel_launches() - n0


@pytest.mark.parametrize("L", [36, 17])
def test_split_launches_uniform(ctx, oracle, monkeypatch, split_ref, L):
    """1 M reads with mask words and -q (L = 17: quality rows at every byte offset): per launch, the kernel's views of
    meta, starts, cigars, bases, qualities, the exception tiles, the mask words, the ok-map and the deferred indices."""
    ref, codes = split_ref
    batch = pos_zero_unmapped(uniform_batch(ref, codes, SPLIT_READS, L, seed=1000 + L, special=0.01))
    max_len = 51

    def run():
        from parasuite_b200.runtime import DeviceBatch
        ctx.upload_reference(ref)
        d = DeviceBatch(batch, "cuda:0")
        st = torch.cuda.current_stream().cuda_stream
        ctx.profile_begin(max_len, infer_qualities=True, emit_t2c_masks=True)
        _, launches = counting_launches(ctx, lambda: ctx.profile_batch_device(d, st))
        masks = ctx.profile_masks()
        with ctx.pileup_run(d, stream=st, masks=masks) as h:
            pile = h.fetch()
        fast = int(ctx.lib.ps_debug_word(ctx.h, 1))
        return (ctx.profile_end(), mask_words(masks), pile, fast), launches

    whole, split, extra = split_and_whole(monkeypatch, run)
    assert extra >= 4, extra
    exp = oracle.profile(ref, batch, max_len, True, threads=8)
    exp_pile = oracle.pileup(ref, batch)
    for (prof, words, pile, fast), how in ((whole, "one launch"), (split, "split")):
        what = f"L {L} {how}"
        assert_same(prof, exp, oracle, what, infer_q=True)
        check_mask_words(words, ref, batch, oracle, what)
        assert_pileup_equal(pile, exp_pile, what)
        shaped = fast_shaped(batch, max_len)
        assert shaped.sum() - 64 * contig_boundaries(ref, batch, shaped) <= fast <= shaped.sum(), (what, fast)
    assert np.array_equal(whole[1], split[1]) and whole[3] == split[3]


def test_split_launches_ragged(ctx, oracle, monkeypatch, split_ref):
    """Trimmed reads in chunks of 2^18 reads (PARASUITE_B200_RAGGED_CHUNK), every chunk split again, with -q."""
    from parasuite_b200 import synth
    ref, codes = split_ref
    batch = synth.trim_uniform(uniform_batch(ref, codes, SPLIT_READS, 40, seed=1100, special=0.01), 18, seed=3)
    monkeypatch.setenv("PARASUITE_B200_RAGGED_CHUNK", str(1 << 18))

    whole, split, extra = split_and_whole(
        monkeypatch, lambda: counting_launches(ctx, lambda: gpu_profile(ctx, ref, batch, 51, True, device=False)))
    assert extra >= 4, extra
    exp = oracle.profile(ref, batch, 51, True, threads=8)
    for (got, fast), how in ((whole, "one launch per chunk"), (split, "split")):
        assert_same(got, exp, oracle, f"ragged {how}", infer_q=True)
        assert fast > 0.95 * batch.n_reads
    assert whole[1] == split[1]


def test_split_launches_fault_in_a_late_launch(ctx, oracle, monkeypatch, split_ref):
    """A record the JVM dies on (its reference name is not in the FASTA) near the end of the batch: the deferred read
    comes from the last launches, its ordinal must be the oracle's."""
    ref, codes = split_ref
    batch = uniform_batch(ref, codes, SPLIT_READS, 36, seed=1200, special=0.01)
    flags = np.asarray(batch.meta[:batch.n_reads]) >> np.uint32(24)
    late = int(np.nonzero(flags[int(0.93 * batch.n_reads):] == 0)[0][0]) + int(0.93 * batch.n_reads)
    batch.meta[late] |= np.uint32(abi.PS_RF_REF_RANGE << 24)
    with pytest.raises(oracle.OracleFault) as eo:
        oracle.profile(ref, batch, 51, threads=8)
    assert (eo.value.code, eo.value.ordinal) == (abi.PS_THROW_REF_RANGE, late)
    whole, split, extra = split_and_whole(
        monkeypatch, lambda: counting_launches(ctx, lambda: gpu_profile(ctx, ref, batch, 51, device=False)[0]))
    assert extra >= 4, extra
    for got in (whole, split):
        assert isinstance(got, abi.ReferenceWouldThrow) and got.fault == (eo.value.code, eo.value.ordinal), got
