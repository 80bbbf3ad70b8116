"""CPU: the native host batcher (FASTA -> packed reference, BGZF/BAM -> SoA batches) against the record-by-record
Python packers, on files written by the pure-Python writers.  No GPU needed (the batcher is host code)."""
import os
import random

import numpy as np
import pytest

from helpers import random_genome, random_records
from parasuite_b200 import PackedReference, ReadBatch, Record, abi
from parasuite_b200.bamio import BamBatcher, PackedFasta, batch_to_records, write_bam, write_fasta

pytestmark = pytest.mark.skipif(not os.path.exists(abi.lib_path()), reason="library not built")

STREAMS = ("meta", "ref_start", "tile_base_off", "tile_qual_off", "tile_cigar_off", "tile_exc_off")


def assert_batch_equal(a: ReadBatch, b: ReadBatch, what=""):
    assert a.n_reads == b.n_reads, what
    for f in ("uniform_len", "uniform_ncigar", "bases_bytes", "qual_bytes", "cigar_count", "exc_count"):
        assert getattr(a, f) == getattr(b, f), (what, f, getattr(a, f), getattr(b, f))
    for f in STREAMS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), (what, f)
    assert np.array_equal(a.bases2[:a.bases_bytes], b.bases2[:b.bases_bytes]), (what, "bases2")
    assert np.array_equal(a.qual[:a.qual_bytes], b.qual[:b.qual_bytes]), (what, "qual")
    assert np.array_equal(a.cigar[:a.cigar_count], b.cigar[:b.cigar_count]), (what, "cigar")
    assert np.array_equal(a.exc[:a.exc_count], b.exc[:b.exc_count]), (what, "exc")


@pytest.mark.parametrize("width", [60, 7, 1000])
def test_fasta_pack_matches_python_packer(tmp_path, width):
    rng = random.Random(width)
    contigs = random_genome(rng, n_contigs=4, length=3000 + width, n_frac=0.05, lower_frac=0.2)
    contigs.append(("tiny", b"ACGTN"))
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs, line_width=width)
    pf = PackedFasta(fa)
    got, exp = pf.reference(), PackedReference.from_contigs(contigs)
    assert got.names == exp.names and got.lengths == exp.lengths
    assert np.array_equal(got.contig_off, exp.contig_off)
    assert np.array_equal(got.seq2, exp.seq2) and np.array_equal(got.inv, exp.inv)
    pf.close()


def test_fasta_errors(tmp_path):
    fa = str(tmp_path / "x.fa")
    with open(fa, "w") as f:
        f.write(">a\nACGT\n")
    with pytest.raises(abi.PsError) as e:
        PackedFasta(fa)                       # no .fai
    assert e.value.status == abi.PS_ERR_IO
    with open(fa + ".fai", "w") as f:
        f.write("a\t400\t3\t60\t61\n")        # index claims more than the file holds
    with pytest.raises(abi.PsError) as e:
        PackedFasta(fa)
    assert e.value.status == abi.PS_ERR_FORMAT


@pytest.mark.parametrize("seed,kinds,max_batch", [(1, ("M",), 0), (2, ("M", "clip", "indel", "splice", "wild"), 700),
                                                  (3, ("wild", "indel"), 256), (4, ("M",), 1)])
def test_bam_batches_match_python_packer(tmp_path, seed, kinds, max_batch):
    rng = random.Random(seed)
    contigs = random_genome(rng, n_contigs=3, length=5000, n_frac=0.01, lower_frac=0.1)
    recs = random_records(rng, contigs, 1800 if max_batch != 1 else 40, kinds=kinds, Lrange=(1, 60), flags_special=0.08)
    # a record on a contig the FASTA does not hold, one without sequence, one with missing qualities
    recs.append(Record(0, "chrUn", 5, "4M", b"ACGT", bytes([30] * 4)))
    recs.append(Record(4, "*", 0, "*", b"", b""))
    recs.append(Record(16, contigs[2][0], 10, "3M", b"ACN", b"\xff\xff\xff"))
    fa, bam = str(tmp_path / "ref.fa"), str(tmp_path / "x.bam")
    write_fasta(fa, contigs)
    write_bam(bam, [(n, len(s)) for n, s in contigs] + [("chrUn", 1000)], recs, block_bytes=3000)
    pf = PackedFasta(fa)
    ref = pf.reference()
    got = list(BamBatcher(bam, pf, max_batch_reads=max_batch, threads=3))
    step = max_batch or len(recs)
    assert sum(b.n_reads for b in got) == len(recs)
    assert len(got) == (len(recs) + step - 1) // step
    for k, b in enumerate(got):
        assert_batch_equal(b, ReadBatch.from_records(recs[k * step:(k + 1) * step], ref), f"batch {k}")


def test_bam_header_checks(tmp_path):
    rng = random.Random(9)
    contigs = random_genome(rng, n_contigs=2, length=500)
    recs = random_records(rng, contigs, 20)
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, contigs)
    pf = PackedFasta(fa)
    sq = [(n, len(s)) for n, s in contigs]
    bam = str(tmp_path / "u.bam")
    write_bam(bam, sq, recs, sort_order="unsorted")
    with pytest.raises(abi.PsError) as e:
        BamBatcher(bam, pf)
    assert e.value.status == abi.PS_ERR_UNSORTED and "sorted" in str(e.value)      # ErrorProfiling.java:128-131
    write_bam(bam, sq[::-1], recs)                                                   # @SQ order != FASTA order
    with pytest.raises(abi.PsError) as e:
        BamBatcher(bam, pf)
    assert e.value.status == abi.PS_ERR_UNSUPPORTED
    write_bam(bam, sq, recs)
    data = open(bam, "rb").read()
    open(bam, "wb").write(data[:len(data) // 2])                                     # truncated file
    with pytest.raises(abi.PsError) as e:
        list(BamBatcher(bam, pf))
    assert e.value.status == abi.PS_ERR_FORMAT
    open(bam, "wb").write(b"not a bam")
    with pytest.raises(abi.PsError):
        BamBatcher(bam, pf)
    with pytest.raises(abi.PsError) as e:
        BamBatcher(str(tmp_path / "missing.bam"), pf)
    assert e.value.status == abi.PS_ERR_IO


def test_empty_bam(tmp_path):
    contigs = [("chr1", b"ACGT" * 50)]
    fa, bam = str(tmp_path / "ref.fa"), str(tmp_path / "e.bam")
    write_fasta(fa, contigs)
    write_bam(bam, [("chr1", 200)], [])
    assert list(BamBatcher(bam, PackedFasta(fa))) == []


def test_synthetic_batch_round_trip(tmp_path):
    """synthetic SoA batch -> records -> BAM -> native batcher gives the batch back."""
    from parasuite_b200 import synth
    ref = synth.synth_reference(5, [300_000, 200_000], n_run=500)
    batch = synth.synth_reads(ref, 3000, 36, seed=3, special_ppm=20000)
    # the BAM carries contig names: give the packed reference a FASTA twin
    codes = np.zeros(ref.n_bases, dtype=np.uint8)
    for k in range(16):
        codes[k::16] = ((ref.seq2[: (ref.n_bases + 15) // 16] >> (2 * k)) & 3)[: len(codes[k::16])]
    ascii_ = np.frombuffer(b"ACGT", dtype=np.uint8)[codes].copy()
    invbits = np.unpackbits(ref.inv.view(np.uint8), bitorder="little")[: ref.n_bases].astype(bool)
    ascii_[invbits] = ord("N")
    contigs = [(n, ascii_[int(ref.contig_off[i]):int(ref.contig_off[i + 1])].tobytes()) for i, n in enumerate(ref.names)]
    fa, bam = str(tmp_path / "s.fa"), str(tmp_path / "s.bam")
    write_fasta(fa, contigs)
    recs = batch_to_records(batch, ref)
    write_bam(bam, [(n, len(s)) for n, s in contigs], recs)
    pf = PackedFasta(fa)
    assert np.array_equal(pf.reference().seq2, ref.seq2) and np.array_equal(pf.reference().inv, ref.inv)
    got = list(BamBatcher(bam, pf))
    assert len(got) == 1
    assert_batch_equal(got[0], ReadBatch.from_records(recs, ref), "synthetic via records")
    # and against the generator's own arrays (unmapped / POS==0 records lose their coordinates in a BAM)
    g = got[0]
    assert np.array_equal(g.bases2[:g.bases_bytes], batch.bases2[:batch.bases_bytes])
    assert np.array_equal(g.qual[:g.qual_bytes], batch.qual[:batch.qual_bytes])


REF_FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config1", "reference_chr1.fa.gz")


def test_reference_fixture_fasta(tmp_path):
    """The reference's own example genome (chr1, 483 300 bp, N runs, soft-masked; kept byte for byte, gzipped, in the
    config-1 fixture): native pack == Python pack."""
    import gzip
    text = gzip.open(REF_FIXTURE, "rb").read()
    raw = text.split(b"\n")
    name = raw[0][1:].split()[0].decode()
    seq = b"".join(raw[1:])
    fa = str(tmp_path / "chr1.fa")
    write_fasta(fa, [(name, seq)], line_width=len(raw[1]))
    assert open(fa, "rb").read().rstrip(b"\n") == text.rstrip(b"\n")   # same bytes as the fixture
    pf = PackedFasta(fa)
    got, exp = pf.reference(), PackedReference.from_contigs([(name, seq)])
    assert got.lengths == [483300]
    assert np.array_equal(got.seq2, exp.seq2) and np.array_equal(got.inv, exp.inv)
    assert int(np.unpackbits(got.inv.view(np.uint8)).sum()) == seq.upper().count(b"N")


def test_more_than_255_cigar_ops_is_refused_by_name(tmp_path):
    """htsjdk takes any number of CIGAR elements (ErrorProfiling.java:206-207); the SoA keeps 8 bits per record.  The
    batcher refuses such a file with PS_ERR_UNSUPPORTED and the ordinal of the record instead of dropping its CIGAR."""
    contigs = [("chr1", b"ACGT" * 400)]
    cig = "".join("1M1I" for _ in range(130)) + "1M"
    recs = [Record(0, "chr1", 5, "20M", b"ACGT" * 5, bytes([30] * 20)),
            Record(0, "chr1", 10, cig, b"A" * 261, bytes([30] * 261))]
    fa, bam = str(tmp_path / "ref.fa"), str(tmp_path / "x.bam")
    write_fasta(fa, contigs)
    write_bam(bam, [("chr1", 1600)], recs)
    pf = PackedFasta(fa)
    with pytest.raises(abi.PsError) as e:
        list(BamBatcher(bam, pf))
    assert e.value.status == abi.PS_ERR_UNSUPPORTED and "record 1 " in str(e.value)
    pf.close()


def test_sam_text_gives_the_same_batches_as_bam(tmp_path):
    """htsjdk opens SAM and BAM through one factory (ErrorProfiling.java:104-107): the batcher takes SAM text too and
    hands the loops the same SoA (bases upper-cased, '.' as N, QUAL '*' as missing, POS 0 as getAlignmentStart() == 0)."""
    from parasuite_b200.bamio import write_sam
    rng = random.Random(77)
    contigs = random_genome(rng, n_contigs=3, length=4000, n_frac=0.01, lower_frac=0.1)
    # (reads of one base are left out: a lone quality 9 is "*" in SAM text, which means "no qualities")
    recs = random_records(rng, contigs, 1500, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(2, 50), flags_special=0.08)
    recs.append(Record(4, "*", 0, "*", b"", b""))
    recs.append(Record(16, contigs[2][0], 10, "3M", b"ACN", b"\xff\xff\xff"))
    fa, bam, sam = str(tmp_path / "ref.fa"), str(tmp_path / "x.bam"), str(tmp_path / "x.sam")
    write_fasta(fa, contigs)
    hdr = [(n, len(s)) for n, s in contigs]
    write_bam(bam, hdr, recs)
    write_sam(sam, hdr, recs)
    pf = PackedFasta(fa)
    a = list(BamBatcher(bam, pf, max_batch_reads=400, threads=2))
    b = list(BamBatcher(sam, pf, max_batch_reads=400, threads=2))
    assert len(a) == len(b) == 4
    for k, (x, y) in enumerate(zip(a, b)):
        assert_batch_equal(y, x, f"SAM vs BAM, batch {k}")
    # lower-case bases and '.' in the text are what SAMRecord.setReadString normalises
    low = str(tmp_path / "low.sam")
    with open(low, "w") as f:
        f.write("@HD\tVN:1.4\tSO:coordinate\n@SQ\tSN:%s\tLN:%d\n" % hdr[0])
        f.write("r\t0\t%s\t5\t30\t6M\t*\t0\t0\tac.gtN\tIIIIII\n" % hdr[0][0])
    got = list(BamBatcher(low, pf))[0]
    exp = ReadBatch.from_records([Record(0, hdr[0][0], 5, "6M", b"ACNGTN", bytes([40] * 6))], pf.reference())
    assert_batch_equal(got, exp, "lower case / dot")
    with open(low, "w") as f:
        f.write("@HD\tVN:1.4\tSO:unsorted\n@SQ\tSN:%s\tLN:%d\n" % hdr[0])
    with pytest.raises(abi.PsError) as e:
        BamBatcher(low, pf)
    assert e.value.status == abi.PS_ERR_UNSORTED
    pf.close()


def test_hand_encoded_bam_bytes(tmp_path):
    """A BAM assembled here byte by byte from the SAM specification (section 4.2), NOT by bamio.write_bam: magic, header
    text, one reference, two records with hand-packed nibbles, two BGZF members plus the EOF marker, written with zlib at
    raw-deflate level 0 (stored blocks) -- a reader that shares a misreading with our writer would not survive this."""
    import struct
    import zlib

    def bgzf(data: bytes) -> bytes:
        c = zlib.compressobj(0, zlib.DEFLATED, -15)
        comp = c.compress(data) + c.flush()
        bsize = len(comp) + 25
        return (b"\x1f\x8b\x08\x04" + b"\x00" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize) + comp +
                struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))

    text = b"@HD\tVN:1.0\tSO:coordinate\n@SQ\tSN:chrQ\tLN:40\n"
    head = b"BAM\x01" + struct.pack("<i", len(text)) + text + struct.pack("<i", 1) + struct.pack("<i", 5) + b"chrQ\x00" + struct.pack("<i", 40)

    def rec(pos0, flag, cigar, seq_nibbles, l_seq, qual, name=b"q1\x00"):
        body = struct.pack("<iiBBHHHiiii", 0, pos0, len(name), 30, 4680, len(cigar), flag, l_seq, -1, -1, 0) + name
        body += b"".join(struct.pack("<I", (n << 4) | op) for n, op in cigar) + seq_nibbles + qual
        return struct.pack("<i", len(body)) + body

    # read 1: pos 3 (0-based 2), 5M, ACGTN -> nibbles 1,2,4,8,15 ; read 2: reverse, 2S3M, GGTCA, qualities missing
    r1 = rec(2, 0, [(5, 0)], bytes([0x12, 0x48, 0xF0]), 5, bytes([10, 20, 30, 40, 41]))
    r2 = rec(6, 16, [(2, 4), (3, 0)], bytes([0x44, 0x82, 0x10]), 5, b"\xff" * 5)
    blob = bgzf(head + r1[:7]) + bgzf(r1[7:] + r2) + bgzf(b"")          # a record split across two BGZF members
    fa, bam = str(tmp_path / "q.fa"), str(tmp_path / "hand.bam")
    write_fasta(fa, [("chrQ", b"ACGTACGTAC" * 4)])
    open(bam, "wb").write(blob)
    pf = PackedFasta(fa)
    got = list(BamBatcher(bam, pf))
    assert len(got) == 1
    exp = ReadBatch.from_records([Record(0, "chrQ", 3, "5M", b"ACGTN", bytes([10, 20, 30, 40, 41])),
                                  Record(16, "chrQ", 7, "2S3M", b"GGTCA", b"")], pf.reference())
    assert_batch_equal(got[0], exp, "hand-encoded BAM")
    pf.close()


def test_parallel_record_location_equals_serial(tmp_path):
    """More than 8 MB of records at hand: the batcher cuts them into one span per thread, finds a plausible chain start
    in every span and walks all spans at once (bam_batcher.cpp: locate).  Same batches as the one-thread walk, also when
    a batch boundary falls inside the bytes at hand."""
    from parasuite_b200 import synth
    from parasuite_b200.bamio import batch_to_records
    ref = synth.synth_reference(77, [1_000_000, 500_000], n_run=500)
    recs = batch_to_records(synth.synth_reads(ref, 110_000, 36, seed=3, special_ppm=5000), ref)
    fa, bam = str(tmp_path / "r.fa"), str(tmp_path / "r.bam")
    import numpy as np
    k = np.arange(ref.n_bases, dtype=np.int64)
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[(ref.seq2[k >> 4] >> ((k & 15) * 2).astype(np.uint32)) & 3].tobytes()
    write_fasta(fa, [(ref.names[0], seq[:ref.lengths[0]]), (ref.names[1], seq[ref.lengths[0]:])])
    write_bam(bam, list(zip(ref.names, ref.lengths)), recs)
    pf = PackedFasta(fa)
    for max_batch in (0, 40_000):
        got = {}
        for threads in (1, 6):
            got[threads] = list(BamBatcher(bam, pf, max_batch_reads=max_batch, threads=threads))
        assert len(got[1]) == len(got[6]) == (1 if max_batch == 0 else 3)
        for a, b in zip(got[1], got[6]):
            assert a.n_reads == b.n_reads
            for f in ("meta", "ref_start", "bases2", "qual", "cigar", "exc"):
                assert np.array_equal(getattr(a, f), getattr(b, f)), f
