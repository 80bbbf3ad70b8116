"""CPU: BAM and SAM input whose @SQ order differs from the FASTA index.  The Java tools fetch bases by contig name and only
ask whether the contig changed (PileupClusters.java:175-176), so a coordinate-sorted file with any header order is valid
input: the host batcher takes it, reports the header's order, and packs the records exactly as under a FASTA-order
header.  The region-sharded pileup carry compares contigs in that order (parasuite_b200.distributed).

The genome and records here are shared with tests/test_gpu_contig_order.py."""
import os
import random
import socket

import numpy as np
import pytest

import py_oracle as po
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi
from parasuite_b200.bamio import BamBatcher, PackedFasta, write_bam, write_fasta, write_sam

pytestmark = pytest.mark.skipif(not os.path.exists(abi.lib_path()), reason="library not built")

HEADER = [3, 0, 5, 1, 4]          # FASTA indices in @SQ order; FASTA contig 2 is not in the header
UNKNOWN = ("chrUn", 3000)         # an @SQ contig the FASTA lacks (no reads on it), listed third
LENGTH = 3000


def genome(seed):
    rng = random.Random(seed)
    return rng, random_genome(rng, n_contigs=6, length=LENGTH, n_frac=0.004, lower_frac=0.1)


def header_sq(contigs):
    sq = [(contigs[c][0], len(contigs[c][1])) for c in HEADER]
    sq.insert(2, UNKNOWN)
    return sq


def _edge_read(contig, pos, L, rev):
    """A read copied from the reference at `pos` with one T>C (A>G on the minus strand) conversion."""
    name, seq = contig
    s = bytearray(b if b in b"ACGT" else ord("A") for b in seq[pos - 1:pos - 1 + L].upper())
    src, dst = (ord("A"), ord("G")) if rev else (ord("T"), ord("C"))
    k = s.find(bytes([src]))
    if k >= 0:
        s[k] = dst
    return Record(16 if rev else 0, name, pos, f"{L}M", bytes(s), bytes([30] * L))


def permuted_records(seed, n=3000, kinds=("M", "M", "clip", "indel")):
    """(FASTA contigs, records sorted by (header position, pos)) the JVM survives in both tools.  Every header contig
    with reads starts with a read at position 1 and ends with a read that reaches the contig end: consecutive clusters
    across a contig change then overlap in position, and only the contig change separates them."""
    rng, contigs = genome(seed)
    present = [contigs[c] for c in HEADER]
    recs = [r for r in random_records(rng, present, n, kinds=kinds, Lrange=(18, 32), flags_special=0.03) if r.pos > 0]
    for h, c in enumerate(present):
        recs.append(_edge_read(c, 1, 25, h % 2 == 1))
        recs.append(_edge_read(c, LENGTH - 24, 25, h % 2 == 0))
    hpos = {contigs[c][0]: h for h, c in enumerate(HEADER)}
    recs.sort(key=lambda r: (hpos[r.rname], r.pos))
    g = po.Genome(dict(contigs))
    ok = []
    for r in recs:
        try:
            po.pileup(to_py([r]), g, po.SnpDb([]), 1)
            po.profile(to_py([r]), g, 64)
            ok.append(r)
        except po.ReferenceWouldThrow:
            pass
    return contigs, ok


def record_max_key(recs, contigs):
    """(FASTA contig, alignment end) maximum of the records the pileup keys (PileupClusters.java:146-158), contigs
    compared in header order: what ps_pileup_max_key gives under that order."""
    index = {n: i for i, (n, _) in enumerate(contigs)}
    rank = {c: h for h, c in enumerate(HEADER)}
    best = None
    for r in recs:
        ops = po.parse_cigar(r.cigar)
        kinds = {op for op, _ in ops}
        if r.flag & 0x4 or r.pos == 0 or (kinds & {"I", "D"} and "N" in kinds):
            continue
        k = (index[r.rname], r.pos + sum(n for op, n in ops if op in "MDN=X") - 1)
        if best is None or (rank[k[0]], k[1]) > (rank[best[0]], best[1]):
            best = k
    return best


def transitions(recs, contigs):
    """Index of the first record of every header contig after the first one."""
    return [k for k in range(1, len(recs)) if recs[k].rname != recs[k - 1].rname]


def write_pair(tmp_path, contigs, recs, fmt):
    """FASTA, the file with the permuted header, and the same records under a FASTA-order header."""
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs)
    writer = write_bam if fmt == "bam" else write_sam
    perm, plain = str(tmp_path / f"perm.{fmt}"), str(tmp_path / f"plain.{fmt}")
    writer(perm, header_sq(contigs), recs)
    writer(plain, [(n, len(s)) for n, s in contigs], recs)
    return fa, perm, plain


@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_permuted_header_opens_and_reports_its_order(tmp_path, fmt):
    contigs, recs = permuted_records(51, n=500)
    fa, perm, plain = write_pair(tmp_path, contigs, recs, fmt)
    pf = PackedFasta(fa)
    b = BamBatcher(perm, pf, any_contig_order=True)
    assert b.contig_order == HEADER                       # chrUn is left out, FASTA contig 2 is not listed
    b.close()
    for any_order in (True, False):
        b = BamBatcher(plain, pf, any_contig_order=any_order)
        assert b.contig_order == list(range(len(contigs)))
        b.close()
    # without the flag the batcher keeps refusing the header by name: its caller keys the pileup in FASTA order
    with pytest.raises(abi.PsError) as e:
        BamBatcher(perm, pf)
    assert e.value.status == abi.PS_ERR_UNSUPPORTED and "PS_BAM_ANY_CONTIG_ORDER" in str(e.value)


@pytest.mark.parametrize("fmt,max_batch", [("bam", 0), ("bam", 700), ("sam", 0), ("sam", 333)])
def test_batches_equal_fasta_order_header(tmp_path, fmt, max_batch):
    from test_bamio_cpu import assert_batch_equal
    contigs, recs = permuted_records(52, kinds=("M", "clip", "indel", "splice"))
    fa, perm, plain = write_pair(tmp_path, contigs, recs, fmt)
    pf = PackedFasta(fa)
    got, exp = list(BamBatcher(perm, pf, max_batch, any_contig_order=True)), list(BamBatcher(plain, pf, max_batch))
    assert len(got) == len(exp) and sum(b.n_reads for b in got) == len(recs)
    ref = PackedReference.from_contigs(contigs)
    step = max_batch or len(recs)
    for k, (a, b) in enumerate(zip(got, exp)):
        assert_batch_equal(a, b, f"batch {k}")
        assert_batch_equal(a, ReadBatch.from_records(recs[k * step:(k + 1) * step], ref), f"batch {k} (Python packer)")


def test_record_on_a_contig_the_fasta_lacks(tmp_path):
    """A header contig the FASTA lacks keeps its place in the file but not in the order; its records carry
    PS_RF_REF_RANGE (getSubsequenceAt on an unknown contig throws)."""
    contigs, recs = permuted_records(53, n=200)
    k = next(i for i, r in enumerate(recs) if r.rname == contigs[HEADER[2]][0])      # first record after chrUn
    stray = Record(0, UNKNOWN[0], 10, "20M", b"ACGT" * 5, bytes([30] * 20))
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs)
    bam = str(tmp_path / "stray.bam")
    write_bam(bam, header_sq(contigs), recs[:k] + [stray] + recs[k:])
    b = BamBatcher(bam, PackedFasta(fa), any_contig_order=True)
    assert b.contig_order == HEADER
    batch = next(b)
    flags = batch.meta >> 24
    assert flags[k] & abi.PS_RF_REF_RANGE
    assert not np.any(np.delete(flags, k) & abi.PS_RF_REF_RANGE)


def test_unsorted_header_is_still_refused(tmp_path):
    contigs, recs = permuted_records(54, n=100)
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs)
    bam = str(tmp_path / "u.bam")
    write_bam(bam, header_sq(contigs), recs, sort_order="unsorted")
    with pytest.raises(abi.PsError) as e:
        BamBatcher(bam, PackedFasta(fa), any_contig_order=True)
    assert e.value.status == abi.PS_ERR_UNSORTED


# ---- the sharded pileup carry in the header's order -----------------------------------------------------------------
def test_exclusive_prefix_max_with_an_order():
    from parasuite_b200.distributed import exclusive_prefix_max
    keys = [(3, 2900), (0, 15), None, (5, 40), (1, 7), (4, 3000)]
    assert exclusive_prefix_max(keys, HEADER) == [None, (3, 2900), (0, 15), (0, 15), (5, 40), (1, 7)]
    assert exclusive_prefix_max(keys) == [None, (3, 2900), (3, 2900), (3, 2900), (5, 40), (5, 40)]     # FASTA order
    # contigs the order does not list come after the listed ones, in FASTA order
    assert exclusive_prefix_max([(2, 5), (4, 1), (6, 1), (2, 9)], [4]) == [None, (2, 5), (2, 5), (6, 1)]


def sharded_by_oracle(oracle, ref, recs, contigs, cuts, order):
    from parasuite_b200.distributed import exclusive_prefix_max
    from parasuite_b200.sharding import merge_pileup_shards
    bounds = [0] + list(cuts) + [len(recs)]
    parts = [recs[lo:hi] for lo, hi in zip(bounds[:-1], bounds[1:])]
    carries = exclusive_prefix_max([record_max_key(p, contigs) for p in parts], order)
    results = [oracle.pileup(ref, ReadBatch.from_records(p, ref), carry=c) for p, c in zip(parts, carries)]
    return merge_pileup_shards(results, bounds[:-1])


def test_prefix_max_carry_over_contig_changes(oracle):
    """Shards cut where the contig before the cut has a higher FASTA index than the one after it (and next to such
    places): the carry taken in header order gives the whole-stream result."""
    from test_sharding_cpu import assert_same
    contigs, recs = permuted_records(55)
    ref = PackedReference.from_contigs(contigs)
    whole = oracle.pileup(ref, ReadBatch.from_records(recs, ref))
    index = {n: i for i, (n, _) in enumerate(contigs)}
    down = [k for k in transitions(recs, contigs) if index[recs[k].rname] < index[recs[k - 1].rname]]
    assert len(down) == 2                                   # 3 -> 0 and 5 -> 1
    for cuts in ([down[0]], [down[1]], down, [down[0] + 1, down[1] - 1], [down[0] - 1, down[0], down[1] + 3],
                 [1, len(recs) // 2, len(recs) - 1]):
        assert_same(sharded_by_oracle(oracle, ref, recs, contigs, cuts, HEADER), whole, f"cuts {cuts}")


def _worker_ordered(rank, world, port, q):
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    repo = os.path.dirname(here)
    for p in (os.path.join(repo, "para-suite_b200"), os.path.join(repo, "oracle"), here):
        sys.path.insert(0, p)
    import torch.distributed as dist
    import oracle_lib
    from parasuite_b200.distributed import sharded_pileup
    from test_sharding_cpu import assert_same
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    contigs, recs = permuted_records(56)
    ref = PackedReference.from_contigs(contigs)
    t = transitions(recs, contigs)
    cuts = {2: [t[0]], 3: [t[0] + 5, t[2]]}[world]          # at the 3 -> 0 change; 5 reads into contig 0 and at 5 -> 1
    bounds = [0] + cuts + [len(recs)]
    lo, hi = bounds[rank], bounds[rank + 1]
    part = recs[lo:hi]
    res, merged = sharded_pileup(ReadBatch.from_records(part, ref), lambda b: record_max_key(part, contigs),
                                 lambda b, c: oracle_lib.pileup(ref, b, carry=c), lo, order=HEADER)
    if rank == 0:
        ok = True
        try:
            assert_same(merged, oracle_lib.pileup(ref, ReadBatch.from_records(recs, ref)), f"gloo, world {world}")
        except AssertionError as e:
            ok = False
            q.put(repr(e))
        q.put(ok)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_world_gloo_carry_in_header_order(oracle, world):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker_ordered, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    out = []
    while not q.empty():
        out.append(q.get())
    assert out and out[-1] is True, out
