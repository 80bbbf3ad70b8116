"""GPU: the bit-parallel T>C word (t2c_word) in the pileup (pl_decode<NW, false> -> t2c_mask_fast) and in the track
(tr_accum_kernel<NW>) at its edges, bit for bit against the C++ restatements.

* every length arm: L = 1 .. 64 across the word edges 16 / 32 / 48, and 65, the first length on the generic paths;
  reads flush with both ends of every contig (the last one ends the genome), both strands, N calls, duplicates,
  unmapped and POS-0 records; `=` / `X` single-op reads in the track;
* fast against generic on the same reads, with no switch: a view of the batch whose `bases2` is not 4-byte aligned
  sends both tools to their generic decoders, which read bases bytewise;
* the 2-bit code stored under a listed N call (`exc`) and under a reference N is arbitrary: no tool may read it;
* reads that run over the end of a contig fault at the oracle's ordinal.

The mask-fed pileup at every length is test_gpu_fast_edges.py::test_mask_words_every_length."""
import numpy as np
import pytest
import torch

import track_oracle as to
from helpers import assert_profile_equal
from parasuite_b200 import PackedReference, ReadBatch, abi
from test_gpu_fast_edges import (LENGTHS, OP_EQ, OP_X, edge_batch, edge_reference, fused, pos_zero_unmapped,
                                 uniform_batch)
from test_gpu_pileup import assert_pileup_equal
from test_gpu_track import _equal

pytestmark = pytest.mark.gpu

T = abi.PS_TILE_READS
EVERY_LENGTH = LENGTHS + [65]


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


# ---- inputs -------------------------------------------------------------------------------------------------------
def _with(batch, **kw):
    """The batch with some of its arrays (ReadBatch.FIELDS) or sizes replaced."""
    arrays = {f: kw.pop(f, getattr(batch, f)) for f in ReadBatch.FIELDS}
    sizes = dict(uniform_len=batch.uniform_len, uniform_ncigar=batch.uniform_ncigar, bases_bytes=batch.bases_bytes,
                 qual_bytes=batch.qual_bytes, cigar_count=batch.cigar_count, exc_count=batch.exc_count)
    sizes.update(kw)
    return ReadBatch(batch.n_reads, *(arrays[f] for f in ReadBatch.FIELDS), **sizes)


def exc_entries(batch):
    """(read, position) of every `exc` entry, in list order: the read is tile * 256 + (entry >> 16)."""
    teo = np.asarray(batch.tile_exc_off).astype(np.int64)
    tile = np.repeat(np.arange(teo.size - 1), np.diff(teo))
    e = np.asarray(batch.exc[:batch.exc_count]).astype(np.int64)
    return tile * T + (e >> 16), e & 0xFFFF


def _set_codes(bases2, read, pos, code, bpr):
    out = bases2.copy()
    byte, shift = read * bpr + pos // 4, 2 * (pos % 4)
    for s in (0, 2, 4, 6):                  # the positions of one byte are written in separate passes
        k = shift == s
        out[byte[k]] = (out[byte[k]] & np.uint8(~(3 << s) & 0xFF)) | (np.asarray(code)[k] << s).astype(np.uint8)
    return out


def _flags(batch, reads):
    return np.asarray(batch.meta)[reads] >> np.uint32(24)


def with_tile_edge_calls(batch, ref_codes):
    """The uniform batch with one more N call (code 0, as the producers store it) on the first and the last read of
    every tile: the ends of a tile's exception list.  It sits on the first reference T (plus) / A (minus) under the
    read where there is one, so a decoder that read the code under it could count an event there."""
    n, L = batch.n_reads, batch.uniform_len
    read, pos = exc_entries(batch)
    edge = np.unique(np.concatenate((np.arange(0, n, T), np.minimum(np.arange(T - 1, n + T - 1, T), n - 1))))
    rev = (_flags(batch, edge) & abi.PS_RF_REVERSE) != 0
    under = ref_codes[np.asarray(batch.ref_start)[edge].astype(np.int64)[:, None] + np.arange(L)]
    on_target = under == np.where(rev, 0, 3)[:, None]
    edge_pos = np.where(on_target.any(axis=1), on_target.argmax(axis=1), 0)
    key = np.unique(np.concatenate((read * 65536 + pos, edge * 65536 + edge_pos)))
    read, pos = key >> 16, key & 0xFFFF
    meta = batch.meta.copy()
    meta[edge] |= np.uint32(abi.PS_RF_HAS_INVALID << 24)
    teo = np.searchsorted(read, np.arange((n + T - 1) // T + 1) * T).astype(np.uint32)
    exc = (((read % T) << 16) | pos).astype(np.uint32)
    return _with(batch, meta=meta, bases2=_set_codes(batch.bases2, edge, edge_pos, np.zeros(edge.size, np.int64),
                                                         (L + 3) // 4),
                 tile_exc_off=teo, exc=np.concatenate((exc, np.zeros(16, np.uint32))), exc_count=int(exc.size))


def poison_reads(batch, ref_codes, mode, seed=0):
    """A copy of the uniform batch with the code under every `exc` entry rewritten -- mode "hit": C (1) on plus reads
    and G (2) on minus reads; "random": uniform 0..3 -- and the number of rewritten positions where that code would
    make a T>C event (plus: reference T and read C; minus: reference A and read G) in a live read."""
    read, pos = exc_entries(batch)
    flags = _flags(batch, read)
    rev = (flags & abi.PS_RF_REVERSE) != 0
    code = np.where(rev, 2, 1) if mode == "hit" else np.random.default_rng(seed).integers(0, 4, size=read.size)
    live = (flags & (abi.PS_RF_UNMAPPED | abi.PS_RF_POS_ZERO)) == 0
    under = ref_codes[np.asarray(batch.ref_start)[read].astype(np.int64) + pos]
    hits = live & np.where(rev, (under == 0) & (code == 2), (under == 3) & (code == 1))
    return _with(batch, bases2=_set_codes(batch.bases2, read, pos, code, (batch.uniform_len + 3) // 4)), int(hits.sum())


def reference_codes(ref):
    """(2-bit code, invalid bit) of every base of the packed reference."""
    n = ref.n_bases
    codes = ((ref.seq2[:, None] >> (2 * np.arange(16, dtype=np.uint32))) & 3).reshape(-1)[:n]
    inv = np.unpackbits(ref.inv.view(np.uint8), bitorder="little")[:n].astype(bool)
    return codes, inv


def poison_reference(ref, code, seed=0):
    """A copy of the packed reference with `code` (0..3 or "random") as the 2-bit code under every invalid bit.  The
    packer stores 0 (A) there, which only a minus-strand read can meet."""
    codes, inv = reference_codes(ref)
    k = np.nonzero(inv)[0]
    codes = codes.copy()
    codes[k] = np.random.default_rng(seed).integers(0, 4, size=k.size) if code == "random" else code
    w2 = ref.seq2.size
    padded = np.zeros(w2 * 16, dtype=np.uint32)
    padded[:codes.size] = codes
    seq2 = np.bitwise_or.reduce(padded.reshape(w2, 16) << (2 * np.arange(16, dtype=np.uint32)), axis=1)
    return PackedReference(ref.names, ref.lengths, seq2.astype(np.uint32), ref.inv.copy())


def read_codes(batch):
    """[n, L] 2-bit codes of a uniform batch."""
    n, L = batch.n_reads, batch.uniform_len
    bpr = (L + 3) // 4
    b = np.asarray(batch.bases2[:n * bpr]).reshape(n, bpr)
    return ((b[:, :, None] >> (2 * np.arange(4, dtype=np.uint8))) & 3).reshape(n, 4 * bpr)[:, :L]


def _under(batch, ref_codes):
    """[n, L] reference codes under the reads of a uniform batch, and the strand of every read."""
    n, L = batch.n_reads, batch.uniform_len
    g = np.asarray(batch.ref_start[:n]).astype(np.int64)[:, None] + np.arange(L)
    return ref_codes[g], ((_flags(batch, np.arange(n)) & abi.PS_RF_REVERSE) != 0)[:, None]


def mask51_late(batch, ref_codes, first):
    """The uniform batch without T>C events at a strand-oriented index >= 51 in the reads before `first` (the read
    base set to the reference's): the pileup's MASK51 fault comes from a read at `first` or later, and a decoder that
    saw a false event beyond index 50 in an earlier read would name that read instead."""
    L = batch.uniform_len
    under, rev = _under(batch, ref_codes)
    rd = read_codes(batch)
    ev = np.where(rev, (under == 0) & (rd == 2), (under == 3) & (rd == 1))
    ev &= np.where(rev, L - 1 - np.arange(L), np.arange(L)) >= 51
    ev[first:] = False
    r, p = np.nonzero(ev)
    return _with(batch, bases2=_set_codes(batch.bases2, r, p, under[r, p], (L + 3) // 4))


def late_fault(batch, ref_codes):
    """L > 51: mask51_late from the middle of the batch on (the MASK51 fault otherwise comes from one of the first
    reads)."""
    return mask51_late(batch, ref_codes, batch.n_reads // 2) if batch.uniform_len > 51 else batch


def assert_late_mask51(exp, batch, oracle):
    assert isinstance(exp, oracle.OracleFault) and exp.code == abi.PS_THROW_MASK51, batch.uniform_len
    assert exp.ordinal >= batch.n_reads // 2, exp.ordinal


def events_over_reference_n(batch, ref):
    """Aligned positions of live reads where `ref` holds an invalid base whose stored code, read as a base, would make a
    T>C event with the read's (not listed) base."""
    n, L = batch.n_reads, batch.uniform_len
    listed = np.zeros((n, L), dtype=bool)
    read, pos = exc_entries(batch)
    listed[read, pos] = True
    codes, inv = reference_codes(ref)
    under, rev = _under(batch, codes)
    rd = read_codes(batch)
    flags = _flags(batch, np.arange(n))
    live = ((flags & (abi.PS_RF_UNMAPPED | abi.PS_RF_POS_ZERO)) == 0)[:, None]
    hit = np.where(rev, (under == 0) & (rd == 2), (under == 3) & (rd == 1))
    g = np.asarray(batch.ref_start[:n]).astype(np.int64)[:, None] + np.arange(L)
    return int((hit & inv[g] & ~listed & live).sum())


def misaligned(batch):
    """A DeviceBatch of the batch whose `bases2` starts one byte into a fresh allocation, padding kept.  For ctx.track
    and ctx.pileup without mask words only: both check the alignment before they take the bit-parallel path and read
    bases bytewise otherwise."""
    from parasuite_b200.runtime import DeviceBatch
    d = DeviceBatch(batch, "cuda:0")
    src = d._t["bases2"]
    buf = torch.zeros(src.numel() + 4, dtype=torch.uint8, device=src.device)
    buf[1:1 + src.numel()] = src
    torch.cuda.synchronize()                   # the library's stream is not ordered behind torch's
    d._t["bases2"] = buf                       # keeps the allocation alive with the view
    d.struct.bases2 = buf.data_ptr() + 1
    assert d.struct.bases2 % 4 == 1
    return d


def views(batch):
    """The host batch (staged by the call), the same batch resident in HBM, and the misaligned view."""
    from parasuite_b200.runtime import DeviceBatch
    return [("host", batch), ("device", DeviceBatch(batch, "cuda:0")), ("misaligned", misaligned(batch))]


# ---- running and comparing ----------------------------------------------------------------------------------------
def outcome(fn, *faults):
    try:
        return fn()
    except faults as e:
        return e


def oracle_track(ref, batch):
    return outcome(lambda: to.track_cpp(ref, batch), to.TrackFault)


def oracle_pileup(oracle, ref, batch):
    return outcome(lambda: oracle.pileup(ref, batch), oracle.OracleFault)


def assert_like(got, exp, equal, what):
    """Equal results, or the same (code, ordinal) where the oracle faults."""
    if isinstance(exp, Exception):
        assert isinstance(got, abi.ReferenceWouldThrow), (what, "the oracle faults", exp.code, exp.ordinal, got)
        assert got.fault == (exp.code, exp.ordinal), (what, got.fault, (exp.code, exp.ordinal))
        return
    assert not isinstance(got, Exception), (what, got)
    equal(got, exp, what)


def check_track(ctx, batch, exp, what):
    """Every view against the restatement; the uniform single-op views of L <= 64 take the bit-parallel path with every
    counted read, the misaligned view and longer reads none."""
    fast_arm = 1 <= batch.uniform_len <= 64 and batch.uniform_ncigar == 1
    for how, b in views(batch):
        got = outcome(lambda: ctx.track(b), abi.ReferenceWouldThrow)
        assert_like(got, exp, _equal, f"{what} {how}")
        if not isinstance(got, Exception):
            c = got["counters"]
            assert c["fast_path_reads"] == (c["reads_counted"] if fast_arm and how != "misaligned" else 0), (what, how)


def check_pileup(ctx, batch, exp, what):
    for how, b in views(batch):
        assert_like(outcome(lambda: ctx.pileup(b), abi.ReferenceWouldThrow), exp, assert_pileup_equal, f"{what} {how}")


# ---- every length -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", EVERY_LENGTH)
def test_track_every_length(ctx, L):
    ref, _ = edge_reference()
    ctx.upload_reference(ref)
    raw = edge_batch(L)
    exp = oracle_track(ref, raw)              # a mapped record at POS 0: the pileup's fault
    assert isinstance(exp, to.TrackFault) and exp.code == abi.PS_THROW_REF_RANGE
    check_track(ctx, raw, exp, f"L {L} POS-0 mapped")
    batch = pos_zero_unmapped(raw)
    exp = oracle_track(ref, batch)
    assert exp["counters"]["t2c_events"][0] > 0 and exp["counters"]["t2c_events"][1] > 0
    check_track(ctx, batch, exp, f"L {L}")


@pytest.mark.parametrize("op", [OP_EQ, OP_X])
@pytest.mark.parametrize("L", [16, 36, 64])
def test_track_eq_and_x_reads(ctx, L, op):
    ref, codes = edge_reference()
    ctx.upload_reference(ref)
    raw = uniform_batch(ref, codes, 24_000, L, seed=1300 + 10 * L + op, op=op)
    check_track(ctx, raw, oracle_track(ref, raw), f"L {L} op {op} POS-0 mapped")
    batch = pos_zero_unmapped(raw)
    exp = oracle_track(ref, batch)
    assert exp["counters"]["t2c_events"][0] > 0 and exp["counters"]["t2c_events"][1] > 0
    check_track(ctx, batch, exp, f"L {L} op {op}")


@pytest.mark.parametrize("L", EVERY_LENGTH)
def test_pileup_every_length(ctx, oracle, L):
    ref, codes = edge_reference()
    ctx.upload_reference(ref)
    batch = late_fault(pos_zero_unmapped(edge_batch(L)), codes)
    exp = oracle_pileup(oracle, ref, batch)
    if L > 51:      # a T>C index beyond 50 kills the JVM (boolean[51]): every flavour names the oracle's record
        assert_late_mask51(exp, batch, oracle)
    else:
        assert len(exp["sites"]) > 0
    check_pileup(ctx, batch, exp, f"L {L}")


# ---- codes no tool may read ---------------------------------------------------------------------------------------
N_CALL_LENGTHS = [7, 16, 17, 36, 48, 50, 64]


@pytest.mark.parametrize("mode", ["hit", "random"])
@pytest.mark.parametrize("L", N_CALL_LENGTHS)
def test_codes_under_n_calls(ctx, oracle, L, mode):
    """A producer may store any code under a listed N call: the results equal those of the batch that stores A there,
    and the oracles'.  N calls at 2 % of the bases, plus one on the first and the last read of every tile."""
    ref, codes = edge_reference()
    clean = late_fault(pos_zero_unmapped(with_tile_edge_calls(
        uniform_batch(ref, codes, 24_000, L, seed=1400 + L, n_call=0.02), codes)), codes)
    poisoned, hits = poison_reads(clean, codes, mode, seed=L)
    assert hits >= 100, hits
    exp_t = oracle_track(ref, clean)
    _equal(oracle_track(ref, poisoned), exp_t, "the restatement reads listed positions as N")
    exp_p = oracle_pileup(oracle, ref, clean)
    if L > 51:      # the fault must not move to an earlier record
        assert_late_mask51(exp_p, clean, oracle)
    max_len = max(L, 51)
    exp_prof = oracle.profile(ref, clean, max_len, threads=8)
    ctx.upload_reference(ref)
    for name, b in (("clean", clean), ("poisoned", poisoned)):
        what = f"L {L} {mode} {name}"
        check_track(ctx, b, exp_t, what)
        check_pileup(ctx, b, exp_p, what)
        prof, _, pile = fused(ctx, ref, b, max_len)
        assert_profile_equal(prof, exp_prof, f"{what} profile")
        assert_like(pile, exp_p, assert_pileup_equal, f"{what} mask-fed pileup")


@pytest.mark.parametrize("code", [3, "random"])
@pytest.mark.parametrize("L", [16, 36, 64])
def test_codes_under_reference_n(ctx, oracle, L, code):
    """The packed reference may hold any code under an invalid bit: the results equal those on the packer's."""
    ref, codes = edge_reference()
    poisoned = poison_reference(ref, code, seed=L)
    batch = late_fault(pos_zero_unmapped(edge_batch(L)), codes)
    assert events_over_reference_n(batch, poisoned) >= 50
    max_len = max(L, 51)
    exp_t = oracle_track(ref, batch)
    exp_p = oracle_pileup(oracle, ref, batch)
    if L > 51:
        assert_late_mask51(exp_p, batch, oracle)
    exp_prof = oracle.profile(ref, batch, max_len, threads=8)
    what = f"L {L} reference N as {code}"
    ctx.upload_reference(poisoned)
    check_track(ctx, batch, exp_t, what)
    check_pileup(ctx, batch, exp_p, what)
    prof, _, pile = fused(ctx, poisoned, batch, max_len)
    assert_profile_equal(prof, exp_prof, f"{what} profile")
    assert_like(pile, exp_p, assert_pileup_equal, f"{what} mask-fed pileup")


# ---- reads over a contig end ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("last", [False, True])
@pytest.mark.parametrize("back", ["1", "L-1"])
@pytest.mark.parametrize("L", [16, 32, 48, 50])
def test_reads_over_a_contig_end(ctx, oracle, L, back, last):
    """The last read of a middle contig (or of the genome) moved to start 1 or L - 1 bases before the contig's end: it
    reaches L - 1 or 1 bases past it.  The batch stays sorted and the bit-parallel shape holds for that read."""
    from parasuite_b200.runtime import DeviceBatch
    ref, _ = edge_reference()
    batch = pos_zero_unmapped(edge_batch(L))
    k = len(ref.lengths) - 1 if last else 1
    end = int(ref.contig_off[k + 1])
    starts = np.asarray(batch.ref_start[:batch.n_reads])
    r = int(np.searchsorted(starts, end, side="left")) - 1
    assert int(starts[r]) == end - L
    ref_start = batch.ref_start.copy()
    ref_start[r] = end - (1 if back == "1" else L - 1)
    meta = batch.meta.copy()
    meta[r] &= ~np.uint32((abi.PS_RF_UNMAPPED | abi.PS_RF_DUPLICATE | abi.PS_RF_POS_ZERO) << 24)
    bad = _with(batch, ref_start=ref_start, meta=meta)
    exp_t, exp_p = oracle_track(ref, bad), oracle_pileup(oracle, ref, bad)
    assert (exp_t.code, exp_t.ordinal) == (exp_p.code, exp_p.ordinal) == (abi.PS_THROW_REF_RANGE, r)
    ctx.upload_reference(ref)
    d = DeviceBatch(bad, "cuda:0")
    for how, b in (("host", bad), ("device", d)):
        what = f"L {L} starting {back} before the end of contig {k} {how}"
        assert_like(outcome(lambda: ctx.track(b), abi.ReferenceWouldThrow), exp_t, _equal, f"{what} track")
        assert_like(outcome(lambda: ctx.pileup(b), abi.ReferenceWouldThrow), exp_p, assert_pileup_equal, f"{what} pileup")
