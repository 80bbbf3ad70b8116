"""CPU: the per-position T>C conversion and coverage track (tool `track`).  Hand-derived rows on the SURVEY 8(c)
reference against the Python restatement, the Python and C++ restatements against each other on random records of every
CIGAR kind, the file texts and the counter invariants."""
import random

import numpy as np
import pytest

import py_oracle as po
import track_oracle as to
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, Record, abi

REF = "ACGTTGCAAGGCTTACGATCGGATCCTTAGNNacgtTTGACC"

# (flag, pos, cigar, seq) -> plus runs, minus runs (0-based half-open), sites (pos, strand, t2c, cov)
WORKED = [
    ((0, 3, "8M", "GTCGCAAG"), [(2, 10, 1)], [], [(5, "+", 1, 1)]),
    ((16, 3, "8M", "GTCGCAAG"), [], [(2, 10, 1)], []),                          # T>C on the genome is A>G on this strand
    ((0, 3, "4M1D4M", "GTTGAAGG"), [(2, 6, 1), (7, 11, 1)], [], []),            # no coverage at 7 (clust puts block 2 there)
    ((0, 3, "4M10N4M", "GTTGGACC"), [(2, 6, 1), (16, 20, 1)], [], [(19, "+", 1, 1)]),   # nothing across the gap
    ((0, 3, "2M2I4M", "GCAATGCA"), [(2, 8, 1)], [], [(4, "+", 1, 1)]),           # inserted bases take no position
    ((0, 5, "2S6M", "AACGCAAG"), [(4, 10, 1)], [], [(5, "+", 1, 1)]),            # clipped bases take no position
    # over NN and acgt: coverage everywhere, no T>C at N, lower-case t counts
    ((0, 29, "10M", "AGCCACGCCC"), [(28, 38, 1)], [], [(36, "+", 1, 1), (37, "+", 1, 1), (38, "+", 1, 1)]),
    ((16, 29, "10M", "GGGAGCGTTT"), [], [(28, 38, 1)], [(29, "-", 1, 1), (33, "-", 1, 1)]),
]


def _recs(rows):
    return [Record(f, "chr1", p, c, s.encode(), bytes([30] * len(s))) for f, p, c, s in rows]


@pytest.mark.parametrize("k", range(len(WORKED)))
def test_worked_rows(k):
    row, plus, minus, sites = WORKED[k]
    g = po.Genome({"chr1": REF.encode()})
    got = to.track(to_py(_recs([row])), g)
    assert [tuple(r[1:]) for r in got["runs_plus"]] == plus
    assert [tuple(r[1:]) for r in got["runs_minus"]] == minus
    assert [tuple(s[1:]) for s in got["sites"]] == sites
    ref = PackedReference.from_contigs([("chr1", REF.encode())])
    _same(got, to.track_cpp(ref, ReadBatch.from_records(_recs([row]), ref)), ["chr1"])


def test_worked_rows_together_and_file_texts():
    rows = sorted((w[0] for w in WORKED), key=lambda r: r[1])
    g = po.Genome({"chr1": REF.encode()})
    got = to.track(to_py(_recs(rows)), g)
    f = got["files"]
    assert f["t2c.tsv"].splitlines()[0] == "chrom\tpos\tstrand\tt2c\tcoverage"
    assert "chr1\t5\t+\t2\t5\n" in f["t2c.tsv"]            # rows 1 and 6 convert position 5, five plus reads cover it
    assert f["minus.bedGraph"] == "chr1\t2\t10\t1\nchr1\t28\t38\t1\n"
    for line in f["plus.bedGraph"].splitlines():
        c, a, b, v = line.split("\t")
        assert c == "chr1" and int(a) < int(b) and int(v) > 0
    plus = [tuple(r[1:]) for r in got["runs_plus"]]
    assert all(plus[i][1] < plus[i + 1][0] or plus[i][2] != plus[i + 1][2] for i in range(len(plus) - 1))   # maximal
    ref = PackedReference.from_contigs([("chr1", REF.encode())])
    _same(got, to.track_cpp(ref, ReadBatch.from_records(_recs(rows), ref)), ["chr1"])


def _same(py, cpp, names):
    """track_oracle.track against track_oracle.track_cpp (contigs as names there, FASTA indices here)."""
    for name in ("runs_plus", "runs_minus"):
        a = [(c, s, e, v) for c, s, e, v in py[name]]
        b = [(names[int(x["contig"])], int(x["start0"]), int(x["end0"]), int(x["cov"])) for x in cpp[name]]
        assert a == b, name
    b = [(names[int(x["contig"])], int(x["pos"]), "+-"[int(x["strand"])], int(x["t2c"]), int(x["cov"])) for x in cpp["sites"]]
    assert list(py["sites"]) == b
    for k in ("num_reads_processed", "unmapped", "skipped_due_indel", "reads_counted", "aligned_bases", "t2c_events",
              "n_runs", "n_sites"):
        assert py["counters"][k] == cpp["counters"][k], k


def _invariants(res):
    c = res["counters"]
    for s, name in ((0, "runs_plus"), (1, "runs_minus")):
        a = res[name]
        assert int(((a["end0"].astype(np.int64) - a["start0"]) * a["cov"]).sum()) == c["aligned_bases"][s]
        assert int(res["sites"]["t2c"][res["sites"]["strand"] == s].sum()) == c["t2c_events"][s]


@pytest.mark.parametrize("seed", range(6))
def test_python_and_cpp_oracles_agree(seed):
    rng = random.Random(9100 + seed)
    contigs = random_genome(rng, n_contigs=3, length=500, n_frac=0.03, lower_frac=0.2)
    recs = random_records(rng, contigs, 400, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 90),
                          flags_special=0.05)
    names = [c for c, _ in contigs]
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    batch = ReadBatch.from_records(recs, ref)
    try:
        py = to.track(to_py(recs), g)
    except to.TrackFault as e:
        with pytest.raises(to.TrackFault) as ei:
            to.track_cpp(ref, batch)
        assert (ei.value.code, ei.value.ordinal) == (e.code, e.ordinal)
        recs = [r for i, r in enumerate(recs) if i != e.ordinal and r.pos > 0]
        batch = ReadBatch.from_records(recs, ref)
        py = to.track(to_py(recs), g)
    cpp = to.track_cpp(ref, batch)
    _same(py, cpp, names)
    _invariants(cpp)
    assert cpp["counters"]["reads_counted"] > 300
    assert cpp["counters"]["t2c_events"][0] > 0 and cpp["counters"]["t2c_events"][1] > 0


def test_faults_and_unsorted():
    ref = PackedReference.from_contigs([("chr1", REF.encode())])
    g = po.Genome({"chr1": REF.encode()})
    past_end = [(0, 3, "8M", "GTCGCAAG"), (0, 38, "8M", "TTGACCAA")]           # second read runs off the contig
    with pytest.raises(to.TrackFault) as e:
        to.track(to_py(_recs(past_end)), g)
    assert (e.value.code, e.value.ordinal) == (abi.PS_THROW_REF_RANGE, 1)
    with pytest.raises(to.TrackFault) as e2:
        to.track_cpp(ref, ReadBatch.from_records(_recs(past_end), ref))
    assert (e2.value.code, e2.value.ordinal) == (abi.PS_THROW_REF_RANGE, 1)
    backwards = [(0, 5, "8M", "GTCGCAAG"), (0, 3, "8M", "GTCGCAAG")]
    with pytest.raises(to.TrackUnsorted):
        to.track(to_py(_recs(backwards)), g)
    with pytest.raises(to.TrackUnsorted):
        to.track_cpp(ref, ReadBatch.from_records(_recs(backwards), ref))
    # a read with every T converted, up to position 38: no 51-position limit on the positions of a read
    long = [(0, 1, "42M", REF.replace("T", "C").replace("N", "A").upper())]
    res = to.track_cpp(ref, ReadBatch.from_records(_recs(long), ref))
    assert int(res["sites"]["pos"].max()) == 38
