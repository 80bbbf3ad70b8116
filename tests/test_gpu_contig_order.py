"""GPU: input whose contigs come in another order than the FASTA index (a BAM / SAM header that lists them differently).
The Java tools follow any order: they fetch bases by contig name and close a cluster whenever the contig changes
(PileupClusters.java:175-176).  The pileup's running maximum of (contig, end) takes the contig's position in the order the
records follow (ps_reference_set_contig_order); the file tools take the header's order themselves.  Everything is
compared with the oracles on the same records in file order."""
import ctypes as C
import gzip

import numpy as np
import pytest

import py_oracle as po
from helpers import assert_profile_equal, to_py
from parasuite_b200 import PackedReference, ReadBatch, abi
from parasuite_b200.bamio import write_bam, write_fasta, write_sam
from test_clust_writer_cpu import FILES
from test_contig_order_cpu import HEADER, header_sq, permuted_records, transitions
from test_gpu_pileup import _reorder, assert_pileup_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from parasuite_b200.runtime import Context
    c = Context(0)
    yield c
    c.close()


def _files(tmp_path, contigs, recs, fmt="bam"):
    fa, path = str(tmp_path / "ref.fa"), str(tmp_path / f"reads.{fmt}")
    write_fasta(fa, contigs)
    (write_bam if fmt == "bam" else write_sam)(path, header_sq(contigs), recs)
    return fa, path


# ---- file tools ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_profile_and_error_tool(tmp_path, oracle, fmt):
    from parasuite_b200.profile_files import profile_file_texts
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(61)
    fa, path = _files(tmp_path, contigs, recs, fmt)
    ref = PackedReference.from_contigs(contigs)
    exp = oracle.profile(ref, ReadBatch.from_records(recs, ref), 64)
    want = profile_file_texts(exp, False)
    c = Context(0)
    try:
        c.load_fasta(fa)
        assert_profile_equal(c.profile_bam(path, 64), exp, f"profile_bam {fmt}")
        ctr = c.error_bam(path, 64)
    finally:
        c.close()
    assert list(ctr) == [int(x) for x in exp["counters"]]
    for k in ("errorprofile", "errorprofile.vcf", "qualityPerMismatch", "indels", "indelprofile", "qualities"):
        assert open(f"{path}.{k}").read() == want[k], k


@pytest.mark.parametrize("window,fmt", [(257, "bam"), (1000, "sam"), (10 ** 9, "bam")])
def test_windowed_pileup_bam(tmp_path, oracle, monkeypatch, window, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(62)
    fa, path = _files(tmp_path, contigs, recs, fmt)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
    ref = PackedReference.from_contigs(contigs)
    exp = oracle.pileup(ref, ReadBatch.from_records(recs, ref))
    c = Context(0)
    try:
        c.load_fasta(fa)
        with c.pileup_bam(path) as res:
            got = res.fetch(boundary=True)
    finally:
        c.close()
    assert_pileup_equal(got, exp, f"window {window} {fmt}")
    # the clusters at every contig change: the read at position 1 opens one on the next contig
    starts = {(int(x["contig"]), int(x["start"])) for x in got["clusters"]}
    assert all((c_, 1) in starts for c_ in HEADER[1:]) and got["open_cluster"] is not None


@pytest.mark.parametrize("window,min_cov,fmt", [(10 ** 9, 1, "bam"), (400, 2, "sam")])
def test_clust_tool_files(tmp_path, monkeypatch, window, min_cov, fmt):
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(63, kinds=("M", "M", "clip", "indel", "splice"))
    g = po.Genome(dict(contigs))
    st = po.pileup(to_py(recs), g, po.SnpDb([]), min_cov)
    snps = sorted({(c.chrom[3:], pos, "T", "C") for c in st.clusters[::4] for pos, _, _ in c.sites[:1]})
    vcf = str(tmp_path / "snp.vcf.gz")
    with gzip.open(vcf, "wt") as f:
        f.write("##fileformat=VCFv4.1\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
        for ch, pos, r, a in snps:
            f.write(f"{ch}\t{pos}\t.\t{r}\t{a}\t.\t.\t.\n")
    exp = po.clust_files(to_py(recs), g, po.SnpDb(snps), min_cov)
    fa, path = _files(tmp_path, contigs, recs, fmt)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", str(window))
    out = str(tmp_path / "clusters.tsv")
    c = Context(0)
    try:
        c.load_fasta(fa)
        ctr = c.clust_bam(path, out, vcf, min_cov)
    finally:
        c.close()
    assert ctr["num_reads_processed"] == len(recs)
    for k, p in FILES.items():
        got = open(p.format(out=out, bam=path)).read()
        assert got == exp[k], (k, got[:300], exp[k][:300])
    assert exp["pileup"].count("\n") > 20 and "T-C mutations identified as SNPs: 0" not in exp["report"]


def test_two_contexts(tmp_path, oracle, monkeypatch):
    from parasuite_b200.runtime import MultiContext
    contigs, recs = permuted_records(64, n=5000)
    fa, path = _files(tmp_path, contigs, recs)
    monkeypatch.setenv("PARASUITE_B200_WINDOW_READS", "700")
    monkeypatch.setenv("PARASUITE_B200_BATCH_READS", "500")
    ref = PackedReference.from_contigs(contigs)
    batch = ReadBatch.from_records(recs, ref)
    m = MultiContext([0, 0])
    try:
        m.load_fasta(fa)
        prof = m.profile_bam(path, 64)
        with m.pileup_bam(path) as res:
            pile = res.fetch(boundary=True)
    finally:
        m.close()
    assert_profile_equal(prof, oracle.profile(ref, batch, 64), "two contexts, profile")
    assert_pileup_equal(pile, oracle.pileup(ref, batch), "two contexts, pileup")


def test_records_going_backwards_against_the_header(tmp_path, oracle):
    """A record on a contig that comes earlier in the header than the one before it: still PS_ERR_UNSORTED."""
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(65, n=1500)
    t = transitions(recs, contigs)
    back = recs[:t[1]] + recs[t[2]:t[3]] + recs[t[1]:t[2]] + recs[t[3]:]     # contig 1 before contig 5
    fa, path = _files(tmp_path, contigs, back)
    c = Context(0)
    try:
        c.load_fasta(fa)
        for call in (lambda: c.pileup_bam(path), lambda: c.clust_bam(path, str(tmp_path / "out.tsv"))):
            with pytest.raises(abi.PsError) as e:
                call()
            assert e.value.status == abi.PS_ERR_UNSORTED
    finally:
        c.close()


def test_file_tools_leave_the_callers_order(tmp_path, oracle):
    """After a file tool on a permuted file -- one that succeeds and one that fails -- the context keys batches in the
    order the caller set: FASTA order by default, else the caller's own."""
    from parasuite_b200.runtime import Context
    contigs, recs = permuted_records(66, n=2000)
    fa, path = _files(tmp_path, contigs, recs)
    t = transitions(recs, contigs)
    (tmp_path / "bad").mkdir()
    _, bad = _files(tmp_path / "bad", contigs, recs[:t[1]] + recs[t[2]:t[3]] + recs[t[1]:t[2]] + recs[t[3]:])
    ref = PackedReference.from_contigs(contigs)
    index = {n: i for i, (n, _) in enumerate(contigs)}
    fasta_sorted = sorted(recs, key=lambda r: (index[r.rname], r.pos))
    plain, perm = ReadBatch.from_records(fasta_sorted, ref), ReadBatch.from_records(recs, ref)
    c = Context(0)
    try:
        c.load_fasta(fa)
        with c.pileup_bam(path) as res:
            res.fetch()
        with pytest.raises(abi.PsError):
            c.pileup_bam(bad)
        assert_pileup_equal(c.pileup(plain), oracle.pileup(ref, plain), "FASTA order after the file tools")
        c.set_contig_order(HEADER)
        c.clust_bam(path, str(tmp_path / "out.tsv"))
        with pytest.raises(abi.PsError):
            c.clust_bam(bad, str(tmp_path / "out2.tsv"))
        assert_pileup_equal(c.pileup(perm), oracle.pileup(ref, perm), "the caller's order after the file tools")
        with pytest.raises(abi.PsError) as e:
            c.pileup(plain)
        assert e.value.status == abi.PS_ERR_UNSORTED
    finally:
        c.close()


# ---- batch level ----------------------------------------------------------------------------------------------------
ORDER = HEADER                      # FASTA contig 2 is not listed: its reads come last


def _synth_permuted(seed, n=240_000):
    """A config-2 style batch (36 nt, one M op) on six contigs, the reads re-sorted into the contig order
    3, 0, 5, 1, 4, 2; (reference, FASTA-sorted batch, permuted batch, first read of every contig in the permuted batch)."""
    from parasuite_b200 import synth
    ref = synth.synth_reference(seed, [300_000] * 6, n_run=200)
    batch = synth.synth_reads(ref, n, 36, seed=seed + 1, n_ppm=0)
    off = ref.contig_off.astype(np.int64)
    contig = np.searchsorted(off, batch.ref_start.astype(np.int64), side="right") - 1
    full = ORDER + [2]
    idx = np.concatenate([np.nonzero(contig == c)[0] for c in full])
    firsts = np.cumsum([0] + [int(np.sum(contig == c)) for c in full])[:-1]
    return ref, batch, _reorder(batch, idx), [int(x) for x in firsts]


def test_batch_needs_the_order(oracle):
    from parasuite_b200.runtime import Context, DeviceBatch
    ref, plain, perm, _ = _synth_permuted(71)
    exp = oracle.pileup(ref, perm)
    c = Context(0)
    try:
        c.upload_reference(ref)
        c.set_contig_order(ORDER)
        assert_pileup_equal(c.pileup(perm), exp, "host batch")
        assert_pileup_equal(c.pileup(DeviceBatch(perm, "cuda:0")), exp, "device batch")
        assert c.lib.ps_pileup_flag_mode(c.h) == 0                 # the speculative flag pass held
        c.set_contig_order(None)
        with pytest.raises(abi.PsError) as e:                      # FASTA order: the batch goes backwards
            c.pileup(perm)
        assert e.value.status == abi.PS_ERR_UNSORTED
        assert_pileup_equal(c.pileup(plain), oracle.pileup(ref, plain), "FASTA order again")
    finally:
        c.close()


def test_exact_look_back_path(oracle):
    """A record reaching over the halo makes the call repeat with the exact look-back flag kernel; under the order."""
    from parasuite_b200.runtime import Context
    ref, _, perm, firsts = _synth_permuted(72)
    k = (firsts[2] // 2048 - 1) * 2048 - 200           # in contig 0, 200 reads in front of a tile boundary
    assert firsts[1] < k and firsts[2] - k > 2048
    perm.cigar[k] = (6_000 << 4) | 3
    c = Context(0)
    try:
        c.upload_reference(ref)
        c.set_contig_order(ORDER)
        exp = oracle.pileup(ref, perm)
        assert_pileup_equal(c.pileup(perm), exp, "exact flags")
        assert c.lib.ps_pileup_flag_mode(c.h) == 1
        assert_pileup_equal(c.pileup(perm), exp, "exact mode, second call")
    finally:
        c.close()


def test_host_and_device_carry_over_shards(ctx, oracle):
    """Shards cut where the contig before the cut has a higher FASTA index than the one after (3 -> 0, 5 -> 1) and next
    to such places: the host carry (FASTA indices) and the device keys (positions in the order) both give the whole
    stream; pileup_max_key names the FASTA index of the contig last in the order."""
    import torch
    from parasuite_b200.distributed import exclusive_prefix_max
    from parasuite_b200.runtime import DeviceBatch
    from parasuite_b200.sharding import merge_pileup_shards, slice_batch
    ref, _, perm, firsts = _synth_permuted(73)
    ctx.upload_reference(ref)
    ctx.set_contig_order(ORDER)
    whole = oracle.pileup(ref, perm)
    n = perm.n_reads
    for cuts in ([0, firsts[1], n], [0, firsts[1] + 3, firsts[3], firsts[3] + 1, n], [0, firsts[3] - 1, firsts[5], n]):
        shards = [DeviceBatch(slice_batch(perm, lo, hi), "cuda:0") for lo, hi in zip(cuts[:-1], cuts[1:])]
        host_keys = [ctx.pileup_max_key(s) for s in shards]
        keys = torch.cat([ctx.pileup_max_key_tensor(s).clone() for s in shards])
        torch.cuda.synchronize()
        full = ORDER + [2]
        for k, hk in zip(keys.tolist(), host_keys):
            assert (None if k == 0 else (full[(k >> 32) - 1], k & 0xFFFFFFFF)) == hk
        carries = exclusive_prefix_max(host_keys, ORDER)
        by_host = [ctx.pileup(s, carry=cy) for s, cy in zip(shards, carries)]
        assert_pileup_equal(merge_pileup_shards(by_host, cuts[:-1]), whole, f"host carry {cuts}")
        by_dev = []
        for r, s in enumerate(shards):
            with ctx.pileup_run(s, carry_keys=(keys.data_ptr(), r)) as h:
                by_dev.append(h.fetch())
        assert_pileup_equal(merge_pileup_shards(by_dev, cuts[:-1]), whole, f"device carry {cuts}")
    assert ctx.pileup_max_key(DeviceBatch(perm, "cuda:0"))[0] == 2           # FASTA contig 2 comes last
    assert ctx.pileup_max_key(DeviceBatch(slice_batch(perm, 0, firsts[2]), "cuda:0"))[0] == 0
    ctx.set_contig_order(None)
    assert ctx.pileup_max_key(DeviceBatch(perm, "cuda:0"))[0] == 5


def test_backwards_against_the_order(ctx, oracle):
    ref, _, perm, firsts = _synth_permuted(74, n=60_000)
    ctx.upload_reference(ref)
    ctx.set_contig_order([0, 3, 5, 1, 4])                   # contigs 3 and 0 swapped: the batch goes backwards
    with pytest.raises(abi.PsError) as e:
        ctx.pileup(perm)
    assert e.value.status == abi.PS_ERR_UNSORTED
    ctx.set_contig_order(ORDER)
    assert_pileup_equal(ctx.pileup(perm), oracle.pileup(ref, perm), "after the refusal")


def test_invalid_orders(oracle):
    from parasuite_b200.runtime import Context, DeviceBatch
    c = Context(0)
    try:
        def call(order, n=None):
            a = (C.c_uint32 * max(len(order), 1))(*order)
            return c.lib.ps_reference_set_contig_order(c.h, a, len(order) if n is None else n)
        assert call([0]) == abi.PS_ERR_STATE                 # no reference yet
        ref, _, perm, _ = _synth_permuted(75, n=20_000)
        c.upload_reference(ref)
        assert call([0, 1, 0]) == abi.PS_ERR_INVALID_ARG     # an index twice
        assert call([0, 6]) == abi.PS_ERR_INVALID_ARG        # an index >= n_contigs
        assert call([0, 1, 2, 3, 4, 5, 0], 7) == abi.PS_ERR_INVALID_ARG     # n > n_contigs
        assert c.lib.ps_reference_set_contig_order(c.h, None, 0) == abi.PS_OK
        assert call(ORDER) == abi.PS_OK
        h = c.pileup_run(DeviceBatch(perm, "cuda:0"), defer=True)
        assert call(ORDER) == abi.PS_ERR_STATE               # a submitted call has not been waited for
        got = h.wait().fetch()
        h.close()
        assert_pileup_equal(got, oracle.pileup(ref, perm), "submitted under the order")
        c.upload_reference(ref)                              # a reference upload brings back FASTA order
        with pytest.raises(abi.PsError) as e:
            c.pileup(perm)
        assert e.value.status == abi.PS_ERR_UNSORTED
    finally:
        c.close()
