"""The resident step (profile kernels with mask words, then the pileup kernels on the same stream) with chained launches
(programmatic dependent launch, the default) against the same step with plain launches (PARASUITE_B200_PDL=0 at
ps_create) and against the oracle: timers on and off, deferred reads, split fast-kernel launches, capacity re-runs, a
failed speculative flag pass, two steps in a row on one context's scratch, and the stamped stage and section times; and
two contexts on one device whose kernels need different amounts of dynamic shared memory."""
import os

import numpy as np
import pytest
import torch

from helpers import assert_profile_equal
from test_gpu_fast_edges import make_reference, pos_zero_unmapped, uniform_batch
from test_gpu_pileup import assert_pileup_equal

pytestmark = pytest.mark.gpu


def new_ctx(pdl):
    from parasuite_b200.runtime import Context
    old = os.environ.get("PARASUITE_B200_PDL")
    os.environ["PARASUITE_B200_PDL"] = "1" if pdl else "0"
    try:
        return Context(0)
    finally:
        if old is None:
            del os.environ["PARASUITE_B200_PDL"]
        else:
            os.environ["PARASUITE_B200_PDL"] = old


@pytest.fixture(scope="module")
def ctxs():
    c = {True: new_ctx(True), False: new_ctx(False)}
    yield c
    for x in c.values():
        x.close()


@pytest.fixture(scope="module")
def data():
    ref, codes = make_reference(11, [90_000, 60_000, 40_000])
    # flags, contig edges, N calls: the fast kernel defers a few percent of the reads
    batch = pos_zero_unmapped(uniform_batch(ref, codes, 60_000, 36, seed=1201, special=0.05))
    return ref, batch


def step(ctx, ref, batch, max_len=51, timers=True):
    """bench.step_resident at one GPU: (profile result, pileup records)."""
    from parasuite_b200.runtime import DeviceBatch
    ctx.upload_reference(ref)
    d = DeviceBatch(batch, "cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    ctx.kernel_times_reset(timers)
    ctx.profile_begin(max_len, emit_t2c_masks=True)
    ctx.profile_batch_device(d, st)
    masks = ctx.profile_masks()
    h = ctx.pileup_run(d, first_running_id=1, stream=st, defer=True, masks=masks)
    try:
        prof = ctx.profile_end()
        h.counters
        pile = h.fetch(boundary=True)
    finally:
        h.close()
    return prof, pile


def same_pileup(a, b, what):
    assert a["counters"] == b["counters"], what
    for t in ("clusters", "sites"):
        assert np.array_equal(a[t], b[t]), (what, t)


def check(ctxs, oracle, ref, batch, what, **kw):
    exp_p = oracle.profile(ref, batch, kw.get("max_len", 51), threads=8)
    exp_l = oracle.pileup(ref, batch)
    got = {}
    for pdl, ctx in ctxs.items():
        prof, pile = step(ctx, ref, batch, **kw)
        assert_profile_equal(prof, exp_p, f"{what} profile pdl={pdl}")
        assert_pileup_equal(pile, exp_l, f"{what} pileup pdl={pdl}")
        got[pdl] = (prof, pile)
    assert np.array_equal(got[True][0]["wide"], got[False][0]["wide"]), what
    same_pileup(got[True][1], got[False][1], what)


@pytest.mark.parametrize("timers", [True, False])
def test_resident_step_with_deferred_reads(ctxs, oracle, data, timers):
    ref, batch = data
    check(ctxs, oracle, ref, batch, f"resident step timers={timers}", timers=timers)


def test_two_steps_in_a_row(ctxs, oracle, data):
    """The second step reuses the scratch, the descriptors and the learnt capacities the first one left."""
    ref, batch = data
    for k in range(2):
        check(ctxs, oracle, ref, batch, f"step {k}")


@pytest.fixture(scope="module")
def big():
    """Enough reads (> 152 k at 36 nt) that a block limit of one tile splits the fast kernel into several launches."""
    ref, codes = make_reference(13, [600_000, 400_000])
    return ref, pos_zero_unmapped(uniform_batch(ref, codes, 240_000, 36, seed=1203, special=0.05))


def test_split_fast_launches(ctxs, oracle, big, monkeypatch):
    from parasuite_b200 import abi
    ref, batch = big
    ctx = ctxs[True]
    step(ctx, ref, batch)          # the first call of a batch this size may re-run the pileup for its capacities
    n0 = ctx.kernel_launches()
    step(ctx, ref, batch)
    whole = ctx.kernel_launches() - n0
    monkeypatch.setenv("PARASUITE_B200_FAST_READS_PER_BLOCK", str(abi.PS_TILE_READS))
    n0 = ctx.kernel_launches()
    check(ctxs, oracle, ref, batch, "split launches")
    assert ctx.kernel_launches() - n0 > whole, "the fast kernel was not split"


def test_speculative_flags_fail_and_rerun_exact(oracle):
    """A record whose reference span reaches over the flag pass's halo: the speculative pass fails, the call runs again
    with the exact look-back kernel, chained and plain alike (fresh contexts: the exact mode is kept per context)."""
    from parasuite_b200 import synth
    ref = synth.synth_reference(93, [2_000_000], n_run=0)
    batch = synth.synth_reads(ref, 200_000, 36, seed=15)
    k = 2048 * 3 - 200
    batch.cigar[k] = (6_000 << 4) | 3                     # a lone N op: alignment end 6 kb downstream
    ctxs = {True: new_ctx(True), False: new_ctx(False)}
    try:
        for c in ctxs.values():
            c.upload_reference(ref)
            assert c.lib.ps_pileup_flag_mode(c.h) == 0
        check(ctxs, oracle, ref, batch, "speculative flags fail")
        for c in ctxs.values():
            assert c.lib.ps_pileup_flag_mode(c.h) == 1
    finally:
        for c in ctxs.values():
            c.close()


def test_two_contexts_on_one_device_interleaved(oracle, data):
    """The dynamic shared memory a kernel may use belongs to the device, not to a context: a context that needs less
    (max_read_length 51) running between two runs of one that needs more (-q at 60: the histogram kernel; 151: the
    fast kernel's rows) must not leave the attribute too low for the latter."""
    from parasuite_b200.runtime import DeviceBatch
    ref, batch = data
    d = DeviceBatch(batch, "cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    big, small = new_ctx(True), new_ctx(True)
    try:
        for c in (big, small):
            c.upload_reference(ref)

        def run(c, max_len, q):
            c.profile_begin(max_len, q)
            c.profile_batch_device(d, st)
            got = c.profile_end()
            exp = oracle.profile(ref, batch, max_len, q, threads=8)
            assert_profile_equal(got, exp, f"max_len {max_len} -q {q}")
            if q:
                assert np.array_equal(got["quality_hist"], exp["quality_hist"])

        for max_len, q in ((60, True), (151, False)):
            run(big, max_len, q)
            run(small, 51, False)
            run(big, max_len, q)
    finally:
        big.close()
        small.close()


def test_capacity_rerun_on_a_fresh_context(oracle):
    """One read per cluster: the first call of a context overflows the cluster slots it assumes and runs again."""
    ref, codes = make_reference(12, [400_000])
    batch = uniform_batch(ref, codes, 3_000, 36, seed=1202, special=0.0)
    spaced = np.arange(batch.n_reads, dtype=np.uint32) * 120 + 100          # no two reads overlap
    batch.ref_start[:batch.n_reads] = spaced
    ctxs = {True: new_ctx(True), False: new_ctx(False)}
    try:
        check(ctxs, oracle, ref, batch, "capacity re-run")
    finally:
        for c in ctxs.values():
            c.close()


def test_stamped_times(ctxs, data):
    """Chain on, timers on: the stage and section times are stamps; finite, positive, and the pileup's stages fit in its
    section."""
    ref, batch = data
    ctx = ctxs[True]
    step(ctx, ref, batch)
    stages = ctx.pileup_stage_ms()
    sections = ctx.kernel_times_ms()
    assert sections.size == 2 and np.all(np.isfinite(sections)) and np.all(sections > 0), sections
    assert np.all(np.isfinite(stages)) and np.all(stages > 0), stages
    assert float(stages.sum()) <= float(sections[1]) * 1.05 + 1e-3, (stages, sections)
