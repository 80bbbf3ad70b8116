"""CPU: the track's per-position base counts (ps_track_opts.base_counts).  The Python and C++ restatements against each
other on random records of every CIGAR kind under several masks and thresholds, the mask parsing of the Python binding,
and the invariants that tie the base counts to the track's own outputs."""
import random

import numpy as np
import pytest

import py_oracle as po
import track_bases_oracle as tb
import track_oracle as to
from helpers import random_genome, random_records, to_py
from parasuite_b200 import PackedReference, ReadBatch, abi
from parasuite_b200.runtime import substitution_mask, track_opts

T2C = 1 << (4 * 3 + 1)
# (substitutions, min_coverage, min_events)
SETTINGS = [(0, 1, 1), (0, 0, 0), (T2C, 1, 1), (T2C, 3, 2), (1 << (4 * 2 + 0), 1, 1), ((1 << 2) | T2C, 2, 1),
            (0, 5, 3), (0x8421, 1, 1)]


def _case(seed):
    rng = random.Random(9700 + seed)
    contigs = random_genome(rng, n_contigs=3, length=400, n_frac=0.05, lower_frac=0.2)
    recs = random_records(rng, contigs, 500, kinds=("M", "clip", "indel", "splice", "wild"), Lrange=(12, 90),
                          err=0.08, flags_special=0.05)
    # N calls in the reads: the batch lists them in `exc`
    for r in recs[::7]:
        s = bytearray(r.seq)
        for _ in range(rng.randint(1, 3)):
            s[rng.randrange(len(s))] = ord("N")
        r.seq = bytes(s)
    g = po.Genome(dict(contigs))
    ref = PackedReference.from_contigs(contigs)
    while True:                             # drop the records the pileup's loop would die on
        try:
            to.track(to_py(recs), g)
            break
        except to.TrackFault as e:
            recs = [r for i, r in enumerate(recs) if i != e.ordinal]
    return contigs, g, ref, recs


def _rows_of(cpp, names):
    return [(names[int(x["contig"])], int(x["pos"]), "+-"[int(x["strand"])], "ACGT"[int(x["ref"])], int(x["cov"]),
             *map(int, x["n"])) for x in cpp["base_rows"]]


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("setting", range(len(SETTINGS)))
def test_python_and_cpp_restatements_agree(seed, setting):
    mask, mc, me = SETTINGS[setting]
    contigs, g, ref, recs = _case(seed)
    names = [c for c, _ in contigs]
    py = tb.track_bases(to_py(recs), g, min_coverage=mc, min_events=me, substitutions=mask)
    cpp = tb.track_bases_cpp(ref, ReadBatch.from_records(recs, ref), min_coverage=mc, min_events=me, substitutions=mask)
    assert _rows_of(cpp, names) == py["base_rows"]
    assert np.array_equal(cpp["base_totals"], py["base_totals"])
    text = "chrom\tpos\tstrand\tref\tcoverage\tA\tC\tG\tT\tN\n" + "".join(
        "\t".join(map(str, r)) + "\n" for r in _rows_of(cpp, names))
    assert text == py["files"]["bases.tsv"]
    # the track's own outputs are those of the plain restatement
    plain = to.track_cpp(ref, ReadBatch.from_records(recs, ref))
    for k in ("runs_plus", "runs_minus", "sites"):
        assert np.array_equal(plain[k], cpp[k]), k
    assert plain["counters"] == cpp["counters"]
    assert py["files"]["t2c.tsv"] == to.track(to_py(recs), g)["files"]["t2c.tsv"]
    if mask == 0x8421:                      # only diagonal bits: nothing is selected
        assert py["base_rows"] == []
    else:
        assert len(py["base_rows"]) > 0


@pytest.mark.parametrize("seed", range(4))
def test_invariants(seed):
    contigs, g, ref, recs = _case(seed)
    cpp = tb.track_bases_cpp(ref, ReadBatch.from_records(recs, ref))
    c, tot, rows = cpp["counters"], cpp["base_totals"], cpp["base_rows"]
    assert np.array_equal(rows["n"].sum(axis=1), rows["cov"])
    assert [int(tot[s, 3, 1]) for s in (0, 1)] == c["t2c_events"]
    # the matrix holds every aligned base at an ACGT reference position: the coverage of the other positions is the rest
    seqs = {i: s for i, (_, s) in enumerate(contigs)}
    for s, name in ((0, "runs_plus"), (1, "runs_minus")):
        off_acgt = sum(int(r["cov"]) for r in cpp[name] for p in range(int(r["start0"]), int(r["end0"]))
                       if seqs[int(r["contig"])][p] not in b"ACGTacgt")
        assert int(tot[s].sum()) == c["aligned_bases"][s] - off_acgt
    # every row's coverage is the strand's coverage at that position
    cov = {}
    for s, name in ((0, "runs_plus"), (1, "runs_minus")):
        for r in cpp[name]:
            for p in range(int(r["start0"]), int(r["end0"])):
                cov[(int(r["contig"]), p + 1, s)] = int(r["cov"])
    assert all(cov[(int(x["contig"]), int(x["pos"]), int(x["strand"]))] == int(x["cov"]) for x in rows)
    assert (rows["n"][:, :4].sum(axis=1) > rows["n"][np.arange(rows.size), rows["ref"]]).all()   # an event in every row


@pytest.mark.parametrize("seed", range(4))
def test_t2c_mask_rows_are_the_sites(seed):
    contigs, g, ref, recs = _case(seed)
    cpp = tb.track_bases_cpp(ref, ReadBatch.from_records(recs, ref), substitutions=T2C)
    rows, sites = cpp["base_rows"], cpp["sites"]
    assert rows.size == sites.size > 0
    for k in ("contig", "pos", "strand", "cov"):
        assert np.array_equal(rows[k].astype(np.int64), sites[k].astype(np.int64)), k
    assert (rows["ref"] == 3).all()
    assert np.array_equal(rows["n"][:, 1], sites["t2c"])


def test_faults_and_unsorted_give_no_rows():
    contigs, g, ref, recs = _case(0)
    bad = list(recs)
    bad.insert(3, bad[-1])                  # a record far ahead, then back
    with pytest.raises(to.TrackUnsorted):
        tb.track_bases_cpp(ref, ReadBatch.from_records(bad, ref))
    with pytest.raises(to.TrackUnsorted):
        tb.track_bases(to_py(bad), g)


def test_mask_parsing():
    assert substitution_mask(None) == 0
    assert substitution_mask(["T>C"]) == T2C
    assert substitution_mask("T>C") == T2C
    assert substitution_mask(["g>a", "A>G"]) == (1 << 8) | (1 << 2)
    assert substitution_mask(["T>C", "T>C"]) == T2C
    all12 = [f"{a}>{b}" for a in "ACGT" for b in "ACGT" if a != b]
    assert substitution_mask(all12) == 0xFFFF & ~0x8421
    for bad in (["T>T"], ["T-C"], ["X>C"], ["TC"], ["T>C>A"], [], [""]):
        with pytest.raises(ValueError):
            substitution_mask(bad)
    assert track_opts(False, 1, 1, ["T>C"]) is None
    o = track_opts(True, 3, 2, ["T>C"])
    assert (o.base_counts, o.min_coverage, o.min_events, o.substitutions) == (1, 3, 2, T2C)
    with pytest.raises(ValueError):
        track_opts(True, -1, 1, None)


def test_abi_layouts():
    import ctypes as C
    assert C.sizeof(abi.ps_track_base_row) == 36 == np.dtype(abi.TRACK_BASE_ROW_DTYPE).itemsize
    assert C.sizeof(abi.ps_track_opts) == 16
    assert C.sizeof(abi.ps_track_base_totals) == 8 * 41
    for f, _ in abi.ps_track_base_row._fields_:
        assert getattr(abi.ps_track_base_row, f).offset == np.dtype(abi.TRACK_BASE_ROW_DTYPE).fields[f][1], f
