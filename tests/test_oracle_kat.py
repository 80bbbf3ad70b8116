"""CPU: both oracle restatements against the hand-derived vectors of SURVEY.md 8(c), and against each other."""
import random

import numpy as np
import pytest

import py_oracle as po
from helpers import (assert_profile_equal, kat_records, py_profile_dict, random_genome, random_records, to_py)
from kat_vectors import (BASES, KAT_MAXLEN, KAT_REF, PILEUP_DOUBLE_STRANDED, PILEUP_EXPECT, PILEUP_READS, PILEUP_REF,
                         PROFILE_KATS, parse_conv)
from parasuite_b200 import PackedReference, ReadBatch, abi


def expected_profile(k):
    m = KAT_MAXLEN
    conv = np.zeros((m, 4, 4), dtype=np.int32)
    for (i, a, b), v in parse_conv(k["conv"]).items():
        conv[i, a, b] = v
    return conv


def check_kat(kid, got):
    k = PROFILE_KATS[kid]
    assert np.array_equal(got["position_conversions"], expected_profile(k)), kid
    if "qsum" in k:
        qs = np.zeros((4, 4), dtype=np.int32)
        for key, v in k["qsum"].items():
            a, b = key.split(">")
            qs[BASES.index(a), BASES.index(b)] = v
        assert np.array_equal(got["quality_per_mismatch"], qs), kid
    ins = np.zeros(KAT_MAXLEN)
    dele = np.zeros(KAT_MAXLEN)
    for i, v in k.get("ins", {}).items():
        ins[i] = v
    for i, v in k.get("dels", {}).items():
        dele[i] = v
    assert np.array_equal(got["insertions_per_pos"], ins), kid
    assert np.array_equal(got["deletions_per_pos"], dele), kid
    for name, v in k.get("counters", {}).items():
        assert got["counters"][abi.PS_PC_NAMES.index(name)] == v, (kid, name)


@pytest.mark.parametrize("kid", sorted(PROFILE_KATS))
def test_profile_kat_python(kid):
    g = po.Genome({"chr1": KAT_REF.encode()})
    st = po.profile(to_py(kat_records(PROFILE_KATS[kid]["reads"])), g, KAT_MAXLEN)
    check_kat(kid, py_profile_dict(st))


@pytest.mark.parametrize("kid", sorted(PROFILE_KATS))
def test_profile_kat_cpp(kid, oracle):
    ref = PackedReference.from_contigs([("chr1", KAT_REF.encode())])
    batch = ReadBatch.from_records(kat_records(PROFILE_KATS[kid]["reads"]), ref)
    check_kat(kid, oracle.profile(ref, batch, KAT_MAXLEN))


def test_profile_kat_all_in_one_batch(oracle):
    """All KAT reads in one stream: sums of the individual expectations."""
    ref = PackedReference.from_contigs([("chr1", KAT_REF.encode())])
    recs = []
    for kid in sorted(PROFILE_KATS):
        recs += kat_records(PROFILE_KATS[kid]["reads"])
    got = oracle.profile(ref, ReadBatch.from_records(recs, ref), KAT_MAXLEN)
    exp = sum(expected_profile(PROFILE_KATS[k]) for k in PROFILE_KATS)
    assert np.array_equal(got["position_conversions"], exp)
    st = po.profile(to_py(recs), po.Genome({"chr1": KAT_REF.encode()}), KAT_MAXLEN)
    assert_profile_equal(got, py_profile_dict(st))


def _pileup_check(clusters, sites_of, double_stranded, open_start):
    assert len(clusters) == len(PILEUP_EXPECT)
    for c, e in zip(clusters, PILEUP_EXPECT):
        assert c["cluster_id"] == e["cluster_id"]
        assert (c["start"], c["end"], c["first_reverse"], c["num_reads"]) == \
            (e["start"], e["end"], e["first_reverse"], e["num_reads"])
        assert c["combined"] == e["combined"]
        if "num_t2c" in e:
            assert c["num_t2c"] == e["num_t2c"]
        if "sites" in e:
            assert sites_of(c) == e["sites"]
        if "mask" in e:
            assert c["mask"] == e["mask"]
    assert double_stranded == PILEUP_DOUBLE_STRANDED
    assert open_start == 40


def test_pileup_kat_python():
    g = po.Genome({"chr1": PILEUP_REF.encode()})
    st = po.pileup(to_py(kat_records(PILEUP_READS)), g, po.SnpDb([]), 1)
    cl = [dict(cluster_id=c.cluster_id, start=c.start, end=c.end, first_reverse=c.first_reverse,
               num_reads=c.num_reads, num_t2c=c.num_t2c, combined=c.combined_strand,
               mask=[i for i, m in enumerate(c.mask51) if m], sites={p: (t, v) for p, t, v in c.sites})
          for c in st.clusters]
    _pileup_check(cl, lambda c: c["sites"], st.double_stranded, st.open_cluster.start)
    assert st.clusters[0].fraction == pytest.approx(2 / 2 + 1 / 3)
    assert st.clusters[0].best_pos == 5


def cpp_clusters(res, names):
    strand = {0: "+", 1: "-", 2: "+/-"}
    out = []
    for c in res["clusters"]:
        s = res["sites"][int(c["site_begin"]):int(c["site_end"])]
        out.append(dict(cluster_id=f"cl_{c['running_id']}_{names[c['contig']]}", start=int(c["start"]),
                        end=int(c["end"]), first_reverse=bool(c["first_reverse"]), num_reads=int(c["num_reads"]),
                        num_t2c=int(c["num_t2c"]), combined=strand[int(c["combined_strand"])],
                        mask=[i for i in range(64) if (int(c["mask51"]) >> i) & 1],
                        sites={int(x["pos"]): (int(x["t2c"]), int(x["cov"])) for x in s},
                        order=[int(x["pos"]) for x in sorted(s, key=lambda x: int(x["order_key"]))]))
    return out


def test_pileup_kat_cpp(oracle):
    ref = PackedReference.from_contigs([("chr1", PILEUP_REF.encode())])
    batch = ReadBatch.from_records(kat_records(PILEUP_READS), ref)
    res = oracle.pileup(ref, batch)
    cl = cpp_clusters(res, ref.names)
    _pileup_check(cl, lambda c: c["sites"], res["counters"]["double_stranded"], int(res["open_cluster"]["start"]))


def test_struct_layouts():
    import ctypes
    assert np.dtype(abi.CLUSTER_DTYPE).itemsize == ctypes.sizeof(abi.ps_cluster) == 64
    assert np.dtype(abi.SITE_DTYPE).itemsize == ctypes.sizeof(abi.ps_site) == 24


@pytest.mark.parametrize("seed,kinds", [(1, ("M",)), (2, ("M", "clip")), (3, ("indel",)), (4, ("splice",)),
                                        (5, ("wild", "indel", "clip", "M", "splice"))])
def test_profile_cpp_vs_python_random(oracle, seed, kinds):
    """Two independent restatements must agree read by read, incl. which reads would kill the JVM."""
    rng = random.Random(seed)
    contigs = random_genome(rng)
    recs = random_records(rng, contigs, 300, kinds=kinds, flags_special=0.1)
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    max_len = 64
    n_fault = 0
    keep = []
    for r in recs:   # drop reads on which the JVM would die, but check both oracles agree on that
        b1 = ReadBatch.from_records([r], ref)
        try:
            po.profile(to_py([r]), g, max_len)
            py_fault = None
        except po.ReferenceWouldThrow as e:
            py_fault = e
        try:
            oracle.profile(ref, b1, max_len)
            cpp_fault = None
        except oracle.OracleFault as e:
            cpp_fault = e
        assert (py_fault is None) == (cpp_fault is None), (r, py_fault, cpp_fault)
        if py_fault is None:
            keep.append(r)
        else:
            n_fault += 1
    st = po.profile(to_py(keep), g, max_len)
    got = oracle.profile(ref, ReadBatch.from_records(keep, ref), max_len)
    assert_profile_equal(got, py_profile_dict(st), f"seed {seed}")
    got4 = oracle.profile(ref, ReadBatch.from_records(keep * 5, ref), max_len, threads=4)
    st5 = po.profile(to_py(keep * 5), g, max_len)
    assert_profile_equal(got4, py_profile_dict(st5), f"seed {seed} threads")
    if kinds != ("splice",):      # spliced reads are (almost) all skipped by the reference (quirk Q4)
        assert int(got["counters"][7]) > 0
    else:
        assert int(got["counters"][5]) > 0


@pytest.mark.parametrize("seed,kinds", [(11, ("M",)), (12, ("M", "clip", "indel")), (13, ("wild", "splice", "M"))])
def test_pileup_cpp_vs_python_random(oracle, seed, kinds):
    rng = random.Random(seed)
    contigs = random_genome(rng, n_contigs=2, length=6000, n_frac=0.003, lower_frac=0.05)
    recs = random_records(rng, contigs, 400, kinds=kinds, Lrange=(15, 30), flags_special=0.05)
    recs = [r for r in recs if r.pos > 0]
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    # drop records that would kill the JVM (both must agree)
    keep = []
    for r in recs:
        try:
            po.pileup(to_py([r]), g, po.SnpDb([]), 1)
            pf = False
        except po.ReferenceWouldThrow:
            pf = True
        try:
            oracle.pileup(ref, ReadBatch.from_records([r], ref))
            cf = False
        except oracle.OracleFault:
            cf = True
        assert pf == cf, r
        if not pf:
            keep.append(r)
    st = po.pileup(to_py(keep), g, po.SnpDb([]), 1)
    res = oracle.pileup(ref, ReadBatch.from_records(keep, ref))
    cl = cpp_clusters(res, ref.names)
    assert len(cl) == len(st.clusters) > 10
    for a, b in zip(cl, st.clusters):
        assert a["cluster_id"] == b.cluster_id
        assert (a["start"], a["end"], a["first_reverse"], a["num_reads"], a["num_t2c"], a["combined"]) == \
            (b.start, b.end, b.first_reverse, b.num_reads, b.num_t2c, b.combined_strand)
        assert a["mask"] == [i for i, m in enumerate(b.mask51) if m]
        assert a["sites"] == {p: (t, v) for p, t, v in b.sites}
        assert a["order"] == [p for p, _, _ in b.sites]      # HashMap.put order
    assert res["counters"]["double_stranded"] == st.double_stranded
    assert res["counters"]["skipped_due_indel"] == st.skipped_due_indel
    assert res["counters"]["num_reads_processed"] == st.num_reads_processed
    assert int(res["open_cluster"]["start"]) == st.open_cluster.start


def full_range_records(seed, n, kinds, Lrange):
    """Random records with quality bytes over the whole range 0..254: Java reads them as signed bytes (values 128..254
    are negative, ErrorProfiling.java:301); 0xFF is left out, as the first byte it would mean "no qualities"."""
    from parasuite_b200 import Record
    rng = random.Random(seed)
    contigs = random_genome(rng, n_contigs=2, length=700)
    recs = random_records(rng, contigs, n, kinds=kinds, Lrange=Lrange, flags_special=0.05)
    recs = [Record(r.flag, r.rname, r.pos, r.cigar, r.seq, bytes(rng.randint(0, 254) for _ in r.seq)) for r in recs]
    assert any(q >= 128 for r in recs for q in r.qual)
    return contigs, recs


@pytest.mark.parametrize("infer_q", [False, True])
@pytest.mark.parametrize("seed,kinds", [(21, ("M",)), (22, ("M", "clip", "indel", "wild"))])
def test_profile_cpp_vs_python_full_range_qualities(oracle, seed, kinds, infer_q):
    """The signed-byte rule, and the -q histogram (C++: by byte value 0..255, Python: by the signed Java byte)."""
    contigs, recs = full_range_records(seed, 400, kinds, (1, 60))
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    max_len = 64
    keep = []
    for r in recs:
        try:
            po.profile(to_py([r]), g, max_len, infer_q)
            keep.append(r)
        except po.ReferenceWouldThrow:
            with pytest.raises(oracle.OracleFault):
                oracle.profile(ref, ReadBatch.from_records([r], ref), max_len, infer_q)
    assert len(keep) > 300
    st = po.profile(to_py(keep), g, max_len, infer_q)
    got = oracle.profile(ref, ReadBatch.from_records(keep, ref), max_len, infer_q)
    assert_profile_equal(got, py_profile_dict(st), f"seed {seed} -q {infer_q}")
    assert (got["quality_per_mismatch"] < 0).any()         # the bytes above 127 do go in as negative numbers
    if infer_q:
        hist = np.zeros((max_len, 256), dtype=np.int64)
        for i, d in enumerate(st.qual_hist):
            for q, c in d.items():
                hist[i, q & 0xFF] += c
        assert np.array_equal(got["quality_hist"], hist)
        assert hist[:, 128:].sum() > 0


@pytest.mark.parametrize("seed,kinds", [(31, ("M",)), (32, ("M", "clip", "indel", "wild", "splice"))])
def test_read_t2c_masks_cpp_vs_python(oracle, seed, kinds):
    """oracle.read_t2c_masks (the per-read T>C masks the profile kernel hands the pileup) against the Python pileup's
    per-read mutation map (calculateClusterInformation, PileupClusters.java:637-661) with room for 64 indices."""
    contigs, recs = full_range_records(seed, 500, kinds, (1, 60))
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    got = oracle.read_t2c_masks(ref, ReadBatch.from_records(recs, ref))
    n_set = 0
    for k, (r, p) in enumerate(zip(recs, to_py(recs))):
        exp = 0
        has_id = any(op in "ID" for op, _ in p.cigar)
        if not p.unmapped and p.pos > 0 and not (has_id and any(op == "N" for op, _ in p.cigar)):
            mask = po.JArray(64)
            try:
                po._cluster_information(k, p, g, [False], po.JHashMap(), po.JHashMap(), mask, 0)
                exp = sum(1 << i for i, m in enumerate(mask.a) if m)
            except po.ReferenceWouldThrow:
                pass
        assert int(got[k]) == exp, (k, r, hex(int(got[k])), hex(exp))
        n_set += exp != 0
    assert n_set > 50
