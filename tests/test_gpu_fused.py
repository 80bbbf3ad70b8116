"""GPU: the profile kernel's T>C mask words (ps_profile_opts.emit_t2c_masks, ps_profile_masks_device) fed to the pileup
of the same device-resident batch (ps_pileup_opts.t2c_masks_device) give exactly the records the pileup produces when it
decodes the reads itself -- and both equal the oracle (PileupClusters.java:585-673, mutationMapInRead :651-661)."""
import numpy as np
import pytest
import torch

from parasuite_b200 import abi
from test_gpu_pileup import assert_pileup_equal
from helpers import assert_profile_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


def fused(ctx, dbatch, max_len, defer=False):
    st = torch.cuda.current_stream().cuda_stream
    ctx.profile_begin(max_len, emit_t2c_masks=True)
    ctx.profile_batch_device(dbatch, st)
    masks = ctx.profile_masks()
    with ctx.pileup_run(dbatch, stream=st, masks=masks, defer=defer) as h:
        prof = ctx.profile_end()
        pile = h.fetch()
    return prof, pile, masks


@pytest.mark.parametrize("L,n,ppm,max_len", [(36, 400_000, 0, 51), (36, 300_001, 3000, 51), (50, 300_000, 2000, 51),
                                             (21, 100_003, 500, 30), (62, 60_000, 0, 70), (7, 50_000, 0, 51)])
def test_masks_equal_decode_and_oracle(ctx, oracle, L, n, ppm, max_len):
    from parasuite_b200 import synth
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(77 + L, [4_000_000, 3_000_000], n_run=3000)
    batch = synth.synth_reads(ref, n, L, seed=300 + L, special_ppm=ppm)
    if ppm:   # POS==0 on a mapped record kills the JVM in the pileup loop: drop those for the parity run
        keep = ((batch.meta >> 24) & abi.PS_RF_POS_ZERO) == 0
        batch.meta[~keep] |= np.uint32(abi.PS_RF_UNMAPPED << 24)
    ctx.upload_reference(ref)
    d = DeviceBatch(batch, "cuda:0")
    if L > 51:
        # a T>C index beyond 50 kills the JVM (boolean[51], PileupClusters.java:654): both paths must name the same record
        try:
            ctx.pileup(d)
        except abi.ReferenceWouldThrow as e:
            with pytest.raises(abi.ReferenceWouldThrow) as eg:
                fused(ctx, d, max_len)
            assert eg.value.fault == e.fault
            with pytest.raises(oracle.OracleFault) as eo:
                oracle.pileup(ref, batch)
            assert e.fault == (eo.value.code, eo.value.ordinal)
            return
    exp = oracle.pileup(ref, batch)
    prof, pile, masks = fused(ctx, d, max_len)
    assert masks is not None and masks[1] == batch.n_reads
    assert_pileup_equal(pile, exp, f"masks L {L}")
    assert_pileup_equal(ctx.pileup(d), exp, f"decode L {L}")
    assert_profile_equal(prof, oracle.profile(ref, batch, max_len, threads=8), f"profile with masks L {L}")
    # deferred (submit / wait) flavour, as bench.py runs it
    prof2, pile2, _ = fused(ctx, d, max_len, defer=True)
    assert_pileup_equal(pile2, exp, f"masks deferred L {L}")
    assert np.array_equal(prof2["wide"], prof["wide"])


def mask_words(masks):
    """Copy the device-resident mask words (ctx.profile_masks()) to a host uint64 array."""
    ptr, n = masks

    class _Alias:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 3}

    return torch.as_tensor(_Alias(), device="cuda:0").cpu().numpy().view(np.uint64)


def check_mask_words(words, ref, batch, oracle, what=""):
    """Every valid word belongs to a read of the fast shape and holds the oracle's per-read T>C mask in bits 0..61 and the
    strand in bit 62; invalid words are 0.  Reads of the shape are valid except where a warp-tile of 64 reads straddles
    two contigs: the reads of the second contig in it are deferred."""
    n = batch.n_reads
    meta = np.asarray(batch.meta[:n])
    flags = (meta >> np.uint32(24)).astype(np.uint32)
    shaped = (flags & ~np.uint32(abi.PS_RF_REVERSE | abi.PS_RF_HAS_INVALID)) == 0
    if batch.uniform_len:
        shaped &= (np.asarray(batch.cigar[:n]) & 15) == 0
    valid = (words >> np.uint64(63)) == 1
    assert not (valid & ~shaped).any(), what
    assert (words[~valid] == 0).all(), what
    rev = ((words >> np.uint64(62)) & np.uint64(1)).astype(bool)
    assert np.array_equal(rev[valid], (flags[valid] & abi.PS_RF_REVERSE) != 0), what
    exp = oracle.read_t2c_masks(ref, batch)
    got = words & np.uint64((1 << 62) - 1)
    bad = np.nonzero(valid & (got != exp))[0]
    assert bad.size == 0, (what, "read", bad[:5].tolist(), hex(int(got[bad[0]])) if bad.size else None,
                           hex(int(exp[bad[0]])) if bad.size else None)
    contig = np.searchsorted(ref.contig_off, np.asarray(batch.ref_start[:n]), side="right") - 1
    boundaries = int(np.count_nonzero(np.diff(contig[shaped]) != 0))
    assert valid.sum() >= shaped.sum() - 64 * boundaries, (what, int(valid.sum()), int(shaped.sum()), boundaries)
    return valid


def test_mask_words(ctx, oracle):
    """The words themselves: valid bit, strand bit, and the T>C indices of the oracle's per-read masks."""
    from parasuite_b200 import synth
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(9, [1_000_000], n_run=500)
    batch = synth.synth_reads(ref, 50_000, 36, seed=31, special_ppm=20000)
    ctx.upload_reference(ref)
    d = DeviceBatch(batch, "cuda:0")
    ctx.profile_begin(51, emit_t2c_masks=True)
    ctx.profile_batch_device(d, torch.cuda.current_stream().cuda_stream)
    words = mask_words(ctx.profile_masks())
    ctx.profile_end()
    valid = check_mask_words(words, ref, batch, oracle, "synthetic L 36")
    # the T>C conversions of the bound clusters reach the words
    assert (words[valid] & np.uint64((1 << 62) - 1) != 0).sum() > 1000


def test_no_masks_for_other_shapes(ctx):
    from parasuite_b200 import synth
    from parasuite_b200.runtime import DeviceBatch
    ref = synth.synth_reference(5, [1_000_000], n_run=500)
    batch = synth.synth_reads(ref, 20_000, 150, seed=3, mode=1)      # ragged cigars: generic kernel, no mask words
    ctx.upload_reference(ref)
    d = DeviceBatch(batch, "cuda:0")
    ctx.profile_begin(176, emit_t2c_masks=True)
    ctx.profile_batch_device(d, torch.cuda.current_stream().cuda_stream)
    assert ctx.profile_masks() is None
    ctx.profile_end()
