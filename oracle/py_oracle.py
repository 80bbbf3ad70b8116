"""
TEST INFRASTRUCTURE ONLY -- parity unpinned.

Literal pure-Python transliteration of the two PARA-suite hot loops, working on the same
objects the Java code sees (ASCII read bases, raw FASTA bytes, BAM flags/CIGAR):

  * error profile : src/src/utils/errorprofile/ErrorProfiling.java:146-409 (+ :633-664)
  * T>C pileup    : src/src/utils/pileupclusters/PileupClusters.java:137-500, 585-673
                    (+ StrandOrientation.java:14-56, SNPCalling.java:49-69)

It exists to cross-check the C++ oracle (oracle/parasuite_oracle.cpp) on small inputs: the
reference jar cannot run (no JVM in this image), so two independently written restatements
agreeing on the hand-derived vectors of SURVEY.md 8(c) is the strongest pin available.
"parity unpinned": the reference ships no tests/golden outputs for this path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module.
htsjdk 1.128 semantics (Cigar.getReferenceLength, SAMRecord.getAlignmentEnd,
SAMUtils.getAlignmentBlocks, SequenceUtil.reverseComplement, IndexedFastaSequenceFile
.getSubsequenceAt) are restated from their published behaviour; the jar is bytecode only.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

CIGAR_OPS = "MIDNSHP=X"
CONSUMES_READ = {"M": 1, "I": 1, "D": 0, "N": 0, "S": 1, "H": 0, "P": 0, "=": 1, "X": 1}
CONSUMES_REF = {"M": 1, "I": 0, "D": 1, "N": 1, "S": 0, "H": 0, "P": 0, "=": 1, "X": 1}


class ReferenceWouldThrow(Exception):
    """The Java tool would die here with an uncaught RuntimeException."""

    def __init__(self, ordinal: int, what: str):
        super().__init__(f"record {ordinal}: {what}")
        self.ordinal = ordinal
        self.what = what


class AIOOBE(Exception):
    pass


PS_FAULT_PAST_END = 10


class PastContigEnd(Exception):
    """A mapped record that consumes no reference and starts past its contig's end: the SoA batch holds no contig per
    record, so the library refuses it (ps_fault.code PS_FAULT_PAST_END) where the JVM would keep it."""

    def __init__(self, ordinal: int):
        super().__init__(f"record {ordinal}: no reference span, POS past its contig's end")
        self.ordinal = ordinal
        self.code = PS_FAULT_PAST_END


def past_contig_end(r: "Rec", genome: "Genome") -> bool:
    return r.ref_len() == 0 and r.rname in genome.contigs and r.pos > len(genome.contigs[r.rname])


class JArray:
    """Java array: fixed length, zero filled, bounds checked (no negative indexing)."""

    def __init__(self, n_or_data):
        if isinstance(n_or_data, int):
            self.a = [0] * n_or_data
        else:
            self.a = list(n_or_data)

    def __len__(self):
        return len(self.a)

    def __getitem__(self, i):
        if i < 0 or i >= len(self.a):
            raise AIOOBE(i)
        return self.a[i]

    def __setitem__(self, i, v):
        if i < 0 or i >= len(self.a):
            raise AIOOBE(i)
        self.a[i] = v


@dataclass
class Rec:
    """What htsjdk hands the Java loops for one BAM record."""
    flag: int
    rname: str
    pos: int                      # getAlignmentStart(): 1-based, 0 = none
    cigar: List[Tuple[str, int]]  # [(op, len)]
    seq: bytes                    # getReadBases(): upper-case ASCII from the nibble table
    qual: bytes                   # getBaseQualities(): raw phred; b"" when missing

    @property
    def unmapped(self):
        return bool(self.flag & 0x4)

    @property
    def reverse(self):
        return bool(self.flag & 0x10)

    @property
    def duplicate(self):
        return bool(self.flag & 0x400)

    def cigar_string(self):
        if not self.cigar:
            return "*"
        return "".join(f"{n}{op}" for op, n in self.cigar)

    def ref_len(self):
        return sum(n for op, n in self.cigar if op in "MDN=X")

    def end(self):
        # SAMRecord.getAlignmentEnd
        if self.unmapped:
            return 0
        return self.pos + self.ref_len() - 1

    def alignment_blocks(self):
        # SAMUtils.getAlignmentBlocks: (readStart1, refStart1, len) for M/=/X
        out = []
        rd = 1
        rf = self.pos
        for op, n in self.cigar:
            if op in "HP":
                continue
            if op in "SI":
                rd += n
            elif op in "DN":
                rf += n
            elif op in "M=X":
                out.append((rd, rf, n))
                rd += n
                rf += n
        return out


def parse_cigar(s: str) -> List[Tuple[str, int]]:
    if s == "*" or s == "":
        return []
    out = []
    num = ""
    for ch in s:
        if ch.isdigit():
            num += ch
        else:
            out.append((ch, int(num)))
            num = ""
    return out


class Genome:
    """IndexedFastaSequenceFile.getSubsequenceAt on in-memory contigs (raw bytes, case kept)."""

    def __init__(self, contigs: Dict[str, bytes]):
        self.contigs = contigs

    def fetch(self, name: str, start: int, stop: int) -> bytes:
        if name not in self.contigs:
            raise KeyError("SAMException: contig not found " + name)
        seq = self.contigs[name]
        if start > stop + 1:
            raise KeyError("SAMException: start after stop")
        if stop > len(seq):
            raise KeyError("SAMException: query asks for data past end of contig")
        if start < 1:
            raise KeyError("SAMException: start < 1")
        return seq[start - 1:stop]


_COMP = {65: 84, 67: 71, 71: 67, 84: 65, 97: 116, 99: 103, 103: 99, 116: 97}


def reverse_complement(a: JArray):
    # htsjdk SequenceUtil.reverseComplement: in place, only ACGTacgt mapped
    n = len(a.a)
    a.a = [_COMP.get(b, b) for b in reversed(a.a)]
    assert len(a.a) == n


def array_pos(b: int) -> int:
    # ErrorProfiling.java:633-664 / PileupClusters.java:690-721
    return {65: 0, 67: 1, 71: 2, 84: 3, 97: 0, 99: 1, 103: 2, 116: 3}.get(b, -1)


def _i32(x: int) -> int:
    x &= 0xFFFFFFFF
    return x - (1 << 32) if x & 0x80000000 else x


def _i8(b: int) -> int:
    return b - 256 if b >= 128 else b


# ------------------------------------------------------------------------------------------
# error profile
# ------------------------------------------------------------------------------------------
@dataclass
class ProfileState:
    max_len: int
    pos_conv: List[List[List[int]]] = field(default_factory=list)   # [maxLen][4][4]
    qual_mm: List[List[int]] = field(default_factory=list)          # [4][4]
    qual_mm_cnt: List[List[int]] = field(default_factory=list)
    ins_per_pos: List[float] = field(default_factory=list)
    del_per_pos: List[float] = field(default_factory=list)
    qual_hist: List[Dict[int, int]] = field(default_factory=list)   # -q: per position value->count
    total_bases_checked: int = 0
    num_reads_processed: int = 0
    unmapped: int = 0
    duplicates: int = 0
    start_zero: int = 0
    indel_read: int = 0
    skipped_reads: int = 0
    longer_indels: int = 0

    def __post_init__(self):
        m = self.max_len
        self.pos_conv = [[[0] * 4 for _ in range(4)] for _ in range(m)]
        self.qual_mm = [[0] * 4 for _ in range(4)]
        self.qual_mm_cnt = [[0] * 4 for _ in range(4)]
        self.ins_per_pos = [0.0] * m
        self.del_per_pos = [0.0] * m
        self.qual_hist = [dict() for _ in range(m)]

    def wrapped(self):
        """Java int fields after two's-complement wrap-around (SURVEY Q8)."""
        return {
            "pos_conv": [[[_i32(v) for v in r] for r in p] for p in self.pos_conv],
            "qual_mm": [[_i32(v) for v in r] for r in self.qual_mm],
            "qual_mm_cnt": [[_i32(v) for v in r] for r in self.qual_mm_cnt],
            "ins_per_pos": list(self.ins_per_pos),
            "del_per_pos": list(self.del_per_pos),
            "counters": [_i32(self.num_reads_processed), _i32(self.unmapped), _i32(self.duplicates),
                         _i32(self.start_zero), _i32(self.indel_read), _i32(self.skipped_reads),
                         _i32(self.longer_indels), _i32(self.total_bases_checked)],
        }


def profile_read(st: ProfileState, ordinal: int, r: Rec, genome: Genome, infer_qual: bool = False):
    """One iteration of ErrorProfiling.java:146-409."""
    if r.unmapped:                                    # :155
        st.unmapped += 1
        return
    if r.duplicate:                                   # :159
        st.duplicates += 1
        return
    if r.pos == 0:                                    # :163
        st.start_zero += 1
        return
    read_seq = JArray(r.seq)                          # :168
    try:
        ref_seq = JArray(genome.fetch(r.rname, r.pos, r.end()))   # :169-172
    except KeyError as e:
        raise ReferenceWouldThrow(ordinal, str(e))
    st.num_reads_processed += 1                       # :174
    try:
        if ref_seq[0] == 0:                           # :180
            return
    except AIOOBE:
        raise ReferenceWouldThrow(ordinal, "refSequenceForRead[0] on empty array")
    skip = False
    ml = max(len(read_seq), len(ref_seq))             # :189-193
    if len(read_seq) != len(ref_seq):                 # :194
        ref_t = JArray(ml)
        read_t = JArray(ml)
        p_ref = p_read = p_m = 0
        for op, n in r.cigar:                         # :206
            if op in "MX=":                           # :214-216
                for z in range(n):
                    try:
                        ref_t[z + p_m] = ref_seq[z + p_ref]
                        read_t[z + p_m] = read_seq[z + p_read]
                    except AIOOBE:
                        skip = True                   # :230-242
                p_m += n
                p_ref += n
                p_read += n
            elif op == "N":                           # :247-251 (sic: read cursor moves too)
                p_ref += n
                p_read += n
            elif op == "I":                           # :252-270
                try:
                    for z in range(n):
                        ref_t[p_m + z] = 45
                except AIOOBE:
                    raise ReferenceWouldThrow(ordinal, "I fill beyond mappingLength")
                p_m += n
                p_read += n
                for q in range(1, n + 1):
                    if p_m + q >= st.max_len:
                        raise ReferenceWouldThrow(ordinal, "insertionsPerPos index >= maxReadLength")
                    st.ins_per_pos[p_m + q] += 1.0
                if n > 1:
                    st.longer_indels += 1
            elif op == "D":                           # :272-294
                try:
                    for z in range(n):
                        read_t[p_m + z] = 45
                except AIOOBE:
                    raise ReferenceWouldThrow(ordinal, "D fill beyond mappingLength")
                p_m += n
                p_ref += n
                for q in range(1, n + 1):
                    if p_m + q >= st.max_len:
                        raise ReferenceWouldThrow(ordinal, "deletionsPerPos index >= maxReadLength")
                    st.del_per_pos[p_m + q] += 1.0
                if n > 1:
                    st.longer_indels += 1
            # S, H, P: no branch at all
        st.indel_read += 1                            # :296
        ref_seq = ref_t
        read_seq = read_t
    quals = JArray([_i8(b) for b in r.qual])          # :301 (byte[] is signed)
    if skip:                                          # :303
        st.skipped_reads += 1
        return
    if r.reverse:                                     # :311-316
        reverse_complement(read_seq)
        reverse_complement(ref_seq)
    # :320-348 dead filter loop (isFilter == false): no observable effect
    cs = r.cigar_string()
    has_indel = ("D" in cs) or ("I" in cs)            # :379-382
    for i in range(len(read_seq)):                    # :349
        a = array_pos(ref_seq[i])
        b = array_pos(read_seq[i])
        if a >= 0 and b >= 0:                         # :376
            if i >= st.max_len:
                raise ReferenceWouldThrow(ordinal, "positionConversions index >= maxReadLength")
            st.pos_conv[i][a][b] += 1
            if not has_indel:
                try:
                    q = quals[i]
                except AIOOBE:
                    raise ReferenceWouldThrow(ordinal, "readQualities index out of range")
                st.qual_mm[a][b] += q
                st.qual_mm_cnt[a][b] += 1
            st.total_bases_checked += 1
        if infer_qual:                                # :402-407
            if i >= st.max_len:
                raise ReferenceWouldThrow(ordinal, "baseQualitiesPerPos index >= maxReadLength")
            try:
                q = quals[i]
            except AIOOBE:
                raise ReferenceWouldThrow(ordinal, "readQualities index out of range (-q)")
            st.qual_hist[i][q] = st.qual_hist[i].get(q, 0) + 1


def profile(records: List[Rec], genome: Genome, max_len: int, infer_qual: bool = False) -> ProfileState:
    st = ProfileState(max_len)
    for k, r in enumerate(records):
        profile_read(st, k, r, genome, infer_qual)
    return st


# ------------------------------------------------------------------------------------------
# java.util.HashMap<Integer,Integer> (Java 8+) iteration-order emulation (SURVEY P8)
# ------------------------------------------------------------------------------------------
class JHashMap:
    """Order-faithful model of java.util.HashMap with Integer keys, JDK 8+.

    hash(key) = key ^ (key >>> 16); bucket = hash & (cap-1); new nodes appended at the bucket tail;
    resize (double) when ++size > 0.75*cap, order-preserving lo/hi split; clear() keeps capacity.
    Treeification (>= 8 nodes in a bucket with cap >= 64) is not modelled: raises.
    """

    def __init__(self, initial_capacity: Optional[int] = None):
        self.table: Optional[List[List[List[int]]]] = None
        self.size = 0
        if initial_capacity is None:
            self.threshold = 0          # default ctor: table allocated lazily with cap 16
        else:
            self.threshold = self._table_size_for(initial_capacity)

    @staticmethod
    def _table_size_for(c: int) -> int:
        n = 1
        while n < c:
            n <<= 1
        return max(1, min(n, 1 << 30))

    @staticmethod
    def _hash(k: int) -> int:
        h = k & 0xFFFFFFFF
        return h ^ (h >> 16)

    def _resize(self):
        if self.table is None:
            cap = self.threshold if self.threshold > 0 else 16
            self.table = [[] for _ in range(cap)]
            self.threshold = int(cap * 0.75)
            return
        old = self.table
        ocap = len(old)
        ncap = ocap * 2
        new = [[] for _ in range(ncap)]
        for j, bucket in enumerate(old):
            for node in bucket:
                if self._hash(node[0]) & ocap:
                    new[j + ocap].append(node)
                else:
                    new[j].append(node)
        self.table = new
        self.threshold = int(ncap * 0.75)

    def put(self, k: int, v: int):
        if self.table is None:
            self._resize()
        b = self.table[self._hash(k) & (len(self.table) - 1)]
        for node in b:
            if node[0] == k:
                node[1] = v
                return
        b.append([k, v])
        if len(b) >= 9:
            # 9th node in one bucket: JDK treeifies (cap >= 64) or force-resizes (cap < 64)
            raise NotImplementedError("HashMap treeifyBin path not modelled")
        self.size += 1
        if self.size > self.threshold:
            self._resize()

    def get(self, k: int):
        if self.table is None:
            return None
        for node in self.table[self._hash(k) & (len(self.table) - 1)]:
            if node[0] == k:
                return node[1]
        return None

    def contains(self, k: int) -> bool:
        return self.get(k) is not None

    def remove(self, k: int):
        if self.table is None:
            return
        b = self.table[self._hash(k) & (len(self.table) - 1)]
        for j, node in enumerate(b):
            if node[0] == k:
                del b[j]
                self.size -= 1
                return

    def clear(self):
        if self.table is not None:
            for b in self.table:
                b.clear()
        self.size = 0

    def keys(self) -> List[int]:
        if self.table is None:
            return []
        return [node[0] for b in self.table for node in b]

    def put_all(self, other: "JHashMap"):
        # HashMap.putMapEntries: pre-size when the table is unallocated, else resize if s > threshold
        s = other.size
        if s > 0:
            if self.table is None:
                ft = s / 0.75 + 1.0
                t = int(ft) if ft < (1 << 30) else (1 << 30)
                if t > self.threshold:
                    self.threshold = self._table_size_for(t)
            elif s > self.threshold:
                self._resize()
            for k in other.keys():
                self.put(k, other.get(k))


# ------------------------------------------------------------------------------------------
# T>C pileup
# ------------------------------------------------------------------------------------------
class SnpDb:
    """SNPCalling.querySNP (SNPCalling.java:49-69) over an in-memory list of VCF rows."""

    def __init__(self, rows: List[Tuple[str, int, str, str]]):
        self.rows = rows  # (chrom, pos, ref, alt0)

    def query(self, chrom: str, position: int, ref_base: str, alt_base: str) -> bool:
        if chrom.startswith("chr"):
            chrom = chrom[3:]
        for c, p, rf, al in self.rows:
            # tabix query(chr, position, position+1) returns overlapping records; the body re-checks
            if c == chrom and p == position and ref_base in rf and alt_base in al:
                return True
        return False


@dataclass
class ClusterRecord:
    """State of one cluster at the moment the Java loop would flush it (before the SNP filter)."""
    cluster_id: str
    running_id: int
    chrom: str
    start: int
    end: int
    first_reverse: bool
    num_reads: int
    num_t2c: int
    combined_strand: str                  # isReverse.getStrandOrientation() at flush time
    mask51: List[bool]
    sites: List[Tuple[int, int, int]]     # (pos, t2c, cov) in mutationMap insertion order
    # flush results (only when num_reads >= minCov)
    emitted: bool = False
    num_t2c_sites: int = 0
    fraction: float = 0.0
    best_pos: int = -1
    best_value: float = 0.0
    best_count: Optional[int] = None
    sites_after_snp: List[int] = field(default_factory=list)  # iteration order of filtered map


@dataclass
class PileupState:
    clusters: List[ClusterRecord] = field(default_factory=list)   # every closed cluster, in order
    open_cluster: Optional[ClusterRecord] = None                  # never flushed by the reference
    num_reads_processed: int = 0
    skipped_due_indel: int = 0
    double_stranded: int = 0
    snp_hit: int = 0
    high_frequent_error: int = 0
    num_crosslinked_clusters: int = 0
    num_allele_positions: int = 0
    allele_positions: List[int] = field(default_factory=lambda: [0] * 51)
    allele_frequency_information: List[float] = field(default_factory=list)


def _cluster_information(ordinal, r: Rec, genome: Genome, is_reverse: list, mutation_map: JHashMap,
                         covered_map: JHashMap, mask: JArray, num_t2c: int) -> int:
    """PileupClusters.java:585-673. is_reverse is a 1-element list holding True/False/None."""
    tmp = r.seq
    read_seq: List[int] = []
    ref_seq: List[int] = []
    for rd1, rf1, n in r.alignment_blocks():                      # :593-604
        lo, hi = rd1 - 1, rd1 - 1 + n
        if hi > len(tmp) or lo < 0:
            raise ReferenceWouldThrow(ordinal, "alignment block beyond read bases")
        read_seq += list(tmp[lo:hi])
        try:
            ref_seq += list(genome.fetch(r.rname, rf1, rf1 + n - 1))
        except KeyError as e:
            raise ReferenceWouldThrow(ordinal, str(e))
    read_a = JArray(read_seq)
    ref_a = JArray(ref_seq)
    if r.reverse:                                                 # :606-613
        reverse_complement(read_a)
        reverse_complement(ref_a)
        is_reverse[0] = True
    for i in range(len(read_a)):                                  # :637
        check = (r.end() - i) if r.reverse else (r.pos + i)
        if array_pos(ref_a[i]) == 3 and array_pos(read_a[i]) == 1:
            num_t2c += 1
            try:
                mask[i] = True                                    # :654 (array of 51)
            except AIOOBE:
                raise ReferenceWouldThrow(ordinal, "mutationMapInRead index >= 51")
            if mutation_map.contains(check):
                mutation_map.put(check, mutation_map.get(check) + 1)
            else:
                mutation_map.put(check, 1)
        if covered_map.contains(check):
            covered_map.put(check, covered_map.get(check) + 1)
        else:
            covered_map.put(check, 1)
    return num_t2c


def _strand_str(v) -> str:
    return "+/-" if v is None else ("-" if v else "+")


def pileup(records: List[Rec], genome: Genome, snps: SnpDb, min_cov: int) -> PileupState:
    """PileupClusters.java:108-545 without the FASTA-derived text columns (P5/P9 sequences)."""
    st = PileupState()
    t_start = 0
    t_end = 0
    t_chr = ""
    n_reads = 0
    n_t2c = 0
    mutation_map = JHashMap()
    covered_map = JHashMap()
    is_reverse = [False]
    t_is_reverse = False
    cluster_id = ""
    running_id = 1
    mask = JArray(51)
    insertion_order: List[int] = []   # not Java state; recorded for the device contract

    def snapshot(emit_ok: bool) -> ClusterRecord:
        sites = [(k, mutation_map.get(k), covered_map.get(k)) for k in insertion_order]
        return ClusterRecord(cluster_id, running_id, t_chr, t_start, t_end, t_is_reverse, n_reads, n_t2c,
                             _strand_str(is_reverse[0]), [bool(x) for x in mask.a], sites)

    have_cluster = False
    for ordinal, r in enumerate(records):                         # :137
        st.num_reads_processed += 1
        if r.unmapped:
            continue
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):          # :152-157
            st.skipped_due_indel += 1
            continue
        if r.pos and past_contig_end(r, genome):
            raise PastContigEnd(ordinal)
        if (t_end - r.pos) < 5 or r.rname != t_chr:               # :175-176
            if have_cluster:      # before the first read numReads==0 < minCov: nothing to flush
                rec = snapshot(True)
                if n_reads >= min_cov:                            # :180
                    rec.emitted = True
                    rec.num_t2c_sites = mutation_map.size          # :181
                    best_pos = -1
                    best_val = 0.0
                    tmp_map = JHashMap()
                    tmp_map.put_all(mutation_map)                 # :187-188
                    for key in mutation_map.keys():               # :189
                        if snps.query(t_chr, key, "T", "C"):
                            tmp_map.remove(key)
                            st.snp_hit += 1
                        if mutation_map.get(key) == 1:
                            st.high_frequent_error += 1
                    mutation_map.clear()                          # :200
                    mutation_map.put_all(tmp_map)                 # :201
                    fraction = 0.0
                    if rec.num_t2c_sites > 0:                     # :203
                        sorted_amounts: List[float] = []
                        for key in mutation_map.keys():           # :206
                            v = float(mutation_map.get(key)) / covered_map.get(key)
                            if v >= best_val:
                                best_val = v
                                best_pos = key
                            sorted_amounts.append(v)
                        sorted_amounts.sort(reverse=True)         # stable; equal doubles indistinguishable
                        if len(sorted_amounts) == 0:
                            pass
                        else:
                            s = 0.0
                            for v in sorted_amounts:
                                s += v
                            if s >= 0.2:                          # :232
                                afi = st.allele_frequency_information
                                for k in range(len(sorted_amounts)):
                                    if len(afi) > k:
                                        afi[k] = afi[k] + sorted_amounts[k]
                                    elif len(afi) == 0:
                                        afi.extend(sorted_amounts)
                                    else:
                                        afi.append(sorted_amounts[k])
                                st.num_crosslinked_clusters += 1
                                for j in range(51):
                                    if mask[j]:
                                        st.allele_positions[j] += 1
                                        st.num_allele_positions += 1
                        for v in sorted_amounts:                  # :258-260
                            fraction += v
                    rec.fraction = fraction
                    rec.best_pos = best_pos
                    rec.best_value = best_val
                    rec.best_count = mutation_map.get(best_pos) if best_pos > 0 else None
                    rec.sites_after_snp = mutation_map.keys()
                st.clusters.append(rec)
            t_start = r.pos                                       # :346-357
            t_end = r.end()
            t_chr = r.rname
            n_reads = 1
            n_t2c = 0
            is_reverse[0] = False
            mutation_map.clear()
            covered_map.clear()
            running_id += 1
            cluster_id = "cl_" + str(running_id) + "_" + t_chr
            mask = JArray(51)
            insertion_order = []
            have_cluster = True
            n_t2c = _cluster_information(ordinal, r, genome, is_reverse, mutation_map, covered_map, mask, n_t2c)
            t_is_reverse = is_reverse[0]                          # :364
        else:
            t_chr = r.rname                                       # :419
            if r.end() > t_end:
                t_end = r.end()                                   # :480 (net effect, see DESIGN.md)
            n_reads += 1
            n_t2c = _cluster_information(ordinal, r, genome, is_reverse, mutation_map, covered_map, mask, n_t2c)
            if is_reverse[0] is not None and t_is_reverse != is_reverse[0]:   # :494-498
                st.double_stranded += 1
                is_reverse[0] = None
        # record first-insertion order of T>C sites (device contract, SURVEY "first-insertion rank")
        seen = set(insertion_order)
        # keys are appended in the order calculateClusterInformation inserted them: i ascending
        blocks_len = sum(n for _, _, n in r.alignment_blocks())
        for i in range(blocks_len):
            check = (r.end() - i) if r.reverse else (r.pos + i)
            if check not in seen and mutation_map.contains(check):
                # a key present now but unseen was inserted by this read; order by i
                insertion_order.append(check)
                seen.add(check)
    if have_cluster:
        st.open_cluster = snapshot(False)
    return st


# ------------------------------------------------------------------------------------------
# Post-loop of the `error` tool: the six output files (ErrorProfiling.java:410-591), literally
# ------------------------------------------------------------------------------------------
def _jdiv(a: float, b: float) -> float:
    """Java double division (no exceptions: x/0 = +-Infinity, 0/0 = NaN)."""
    a, b = float(a), float(b)
    if b == 0.0:
        if a == 0.0 or a != a:
            return float("nan")
        return float("inf") if a > 0 else float("-inf")
    return a / b


def profile_outputs(st: ProfileState, infer_qual: bool, fmt) -> Dict[str, str]:
    """Text of <bam>.errorprofile, .errorprofile.vcf, .qualityPerMismatch, .indels, .indelprofile, .qualities and the
    'Averaged T2C' log value.  `fmt` = Double.toString.  Loops and statement order follow the Java."""
    w = st.wrapped()
    pc, qmm, qcnt = w["pos_conv"], w["qual_mm"], w["qual_mm_cnt"]
    n_proc = w["counters"][0]
    m = st.max_len
    base = ["A", "C", "G", "T"]
    out = {k: "" for k in ("errorprofile", "errorprofile.vcf", "qualityPerMismatch", "indels", "indelprofile", "qualities")}
    nl = "\n"
    if infer_qual:                                                   # :421-437
        for i in range(m):
            vals = []
            for q, c in sorted(st.qual_hist[i].items()):
                vals += [q] * c
            n = len(vals)
            mean = _jdiv(float(sum(vals)), n)
            tmp = 0.0
            for v in vals:
                tmp += (v - mean) ** 2
            sd = math.sqrt(_jdiv(tmp, n)) if n else float("nan")
            out["qualities"] += fmt(mean) + "\t" + fmt(sd) + nl
    qpct = [[_jdiv(qmm[i][j], qcnt[i][j]) for j in range(4)] for i in range(4)]      # :439-446
    total_err = [[0.0] * 4 for _ in range(4)]
    total_base = [0.0] * 4
    total_pos = [0] * m
    for i in range(m):                                               # :448-459
        for j in range(4):
            for k in range(4):
                total_err[j][k] += pc[i][j][k]
                total_base[j] += pc[i][j][k]
                total_pos[i] = _i32(total_pos[i] + pc[i][j][k])
    t2c = [0.0] * m
    for i in range(m):                                               # :464-502
        t2c[i] = _jdiv(float(pc[i][3][1]), n_proc) * 100
    for j in range(4):                                               # :504-531
        for k in range(4):
            out["errorprofile.vcf"] += base[j] + "\t" + base[k] + "\t" + fmt(total_err[j][k]) + nl
            total_err[j][k] = _jdiv(total_err[j][k], total_base[j])
            out["errorprofile"] += fmt(total_err[j][k]) + "\t"
            out["qualityPerMismatch"] += fmt(qpct[j][k]) + "\t"
        out["errorprofile"] += nl
        out["qualityPerMismatch"] += nl
        out["errorprofile.vcf"] += nl
    avg = 0.0                                                        # :532-542
    for j in range(m):
        if t2c[j] > 0:
            avg += t2c[j]
        else:
            avg = avg / (j + 1)
            break
    ins, dele = list(w["ins_per_pos"]), list(w["del_per_pos"])
    ins_all = del_all = 0.0
    ins_zero = del_zero = 0
    for i in range(m):                                               # :553-578
        if total_pos[i] == 0:
            ins[i] = 0.0
            dele[i] = 0.0
            ins_zero += 1
            del_zero += 1
        else:
            ins[i] = ins[i] / total_pos[i]
            if ins[i] > 0:
                ins_all += ins[i]
            else:
                ins_zero += 1
            dele[i] = dele[i] / total_pos[i]
            if dele[i] > 0:
                del_all += dele[i]
            else:
                del_zero += 1
        out["indels"] += fmt(ins[i]) + "\t" + fmt(dele[i]) + nl
    if m == ins_zero and m == del_zero:                              # :579-589
        ins_all = del_all = 0.0
    else:
        ins_all = _jdiv(ins_all, m - ins_zero)
        del_all = _jdiv(del_all, m - del_zero)
    out["indelprofile"] = fmt(ins_all) + "\t" + fmt(del_all)
    out["averaged_t2c_epr"] = fmt(avg)
    return out


# ------------------------------------------------------------------------------------------
# Output files of the `clust` tool, literally (PileupClusters.java:62-545): the record loop again, this time WITH the
# cluster sequence (tempClusterBytes :367-414, :421-487) and every writer.  TEST INFRASTRUCTURE: the native writer
# (csrc/clust_writer.cpp) is compared with these texts byte for byte.
# ------------------------------------------------------------------------------------------
def java_double_str(x: float) -> str:
    """Double.toString (shortest round-trip digits; decimal for 1e-3 <= |x| < 1e7, else d.dddE<exp>)."""
    if x != x:
        return "NaN"
    if x == float("inf"):
        return "Infinity"
    if x == float("-inf"):
        return "-Infinity"
    if x == 0:
        return "-0.0" if math.copysign(1.0, x) < 0 else "0.0"
    sign = "-" if x < 0 else ""
    a = abs(x)
    mant, exp = f"{a:.17e}".split("e")
    # shortest repr digits
    r = repr(a)
    if "e" in r:
        m, e = r.split("e")
        e10 = int(e)
    else:
        m, e10 = r, 0
    ip, _, fp = m.partition(".")
    raw = ip + fp
    lead = len(raw) - len(raw.lstrip("0"))
    digits = raw.lstrip("0").rstrip("0") or "0"
    point = len(ip) + e10 - lead            # number of digits in front of the decimal point
    if 1e-3 <= a < 1e7:
        if point <= 0:
            return sign + "0." + "0" * (-point) + digits
        if point >= len(digits):
            return sign + digits + "0" * (point - len(digits)) + ".0"
        return sign + digits[:point] + "." + digits[point:]
    return sign + digits[0] + "." + (digits[1:] or "0") + "E" + str(point - 1)


def _rc_bytes(b: bytearray) -> bytearray:
    a = JArray(list(b))
    reverse_complement(a)
    return bytearray(a.a)


class JvmWouldDie(Exception):
    """An exception the Java code does not catch (SAMException outside a try block)."""


def clust_files(records: List[Rec], genome: Genome, snps: SnpDb, min_cov: int) -> Dict[str, str]:
    """Returns the text of <out>, <out>.ccr.fasta, <out>.ccr.tsv, <out>.report, <bam>.sitefrequency.tsv and
    <bam>.sitepositions.tsv as the Java tool writes them."""
    nl = "\n"
    fmt = java_double_str
    out = {"pileup": "ClusterID\tChr\tStart\tEnd\tStrand\t#reads\t#T2C\t#T2C sites\tT2C Fraction\tSeqenece\tCombStrand\tSeqLength" + nl,
           "ccr.fasta": "",
           "ccr.tsv": "Protein_Group\tCluster ID\tStrand\tChromosome\tCluster_Begin\tCluster_End\tAnchor_FlankSeq_Begin"
                      "\tAnchor_FlankSeq_End\tAnchor_FlankSeq\tAnchor_Position\tCluster_Clone_Count\tNumber_of_T2C_Positions"
                      "\tT2C_Freq_at_Anchor_Position\tT2C_Fract_at_Anchor_Position\tT2C_Freq_Whole_Cluster"
                      "\tT2C_Fract_Whole_Cluster" + nl,
           "report": "", "sitefrequency": "", "sitepositions": ""}
    num_crosslinked = 0
    num_allele_positions = 0
    afi: List[float] = []
    allele_positions = [0] * 51
    mask = JArray(51)
    t_start = t_end = 0
    t_chr = ""
    t_bytes = bytearray()
    n_reads = n_t2c = n_t2c_sites = 0
    double_stranded = 0
    mutation_map = JHashMap()
    covered_map = JHashMap()
    is_reverse = [False]
    t_is_reverse = False
    cluster_id = ""
    running_id = 1
    snp_count = 0                      # `SNPs`: declared, printed, never incremented (:135, :504)
    snp_hit = high_frequent_error = skipped_due_indel = 0

    def fetch(chrom, a, b):
        try:
            return genome.fetch(chrom, a, b)
        except KeyError as e:
            raise JvmWouldDie(str(e))

    for ordinal, r in enumerate(records):
        if r.unmapped:
            continue
        cs = r.cigar_string()
        if (("I" in cs) or ("D" in cs)) and ("N" in cs):
            skipped_due_indel += 1
            continue
        if (t_end - r.pos) < 5 or r.rname != t_chr:
            fraction = 0.0
            if n_reads >= min_cov:                                              # :180
                n_t2c_sites = mutation_map.size
                best_pos, best_val = -1, 0.0
                tmp = JHashMap()
                tmp.put_all(mutation_map)
                for key in mutation_map.keys():
                    if snps.query(t_chr, key, "T", "C"):
                        tmp.remove(key)
                        snp_hit += 1
                    if mutation_map.get(key) == 1:
                        high_frequent_error += 1
                mutation_map.clear()
                mutation_map.put_all(tmp)
                if n_t2c_sites > 0:
                    amounts: List[float] = []
                    for key in mutation_map.keys():
                        v = float(mutation_map.get(key)) / covered_map.get(key)
                        if v >= best_val:
                            best_val, best_pos = v, key
                        amounts.append(v)
                    amounts.sort(reverse=True)
                    if amounts:
                        s = 0.0
                        for v in amounts:
                            s += v
                        if s >= 0.2:
                            for k in range(len(amounts)):
                                if len(afi) > k:
                                    afi[k] = afi[k] + amounts[k]
                                elif len(afi) == 0:
                                    afi.extend(amounts)
                                else:
                                    afi.append(amounts[k])
                            num_crosslinked += 1
                            for j in range(51):
                                if mask[j]:
                                    allele_positions[j] += 1
                                    num_allele_positions += 1
                    for v in amounts:
                        fraction += v
                    if best_pos > 0:                                            # :262
                        strand = _strand_str(is_reverse[0])
                        try:
                            ccr = bytearray(genome.fetch(t_chr, best_pos - 20, best_pos + 20))
                            if strand == "-":
                                ccr = _rc_bytes(ccr)
                        except KeyError:                                        # catch (SAMException e)
                            ccr = bytearray()
                        ccr_seq = "".join(chr(c).upper() for c in ccr)
                        out["ccr.fasta"] += (">" + cluster_id + " 20-anchor-20 " + t_chr + ":" + strand + ":" +
                                             str(best_pos - 20) + "-" + str(best_pos + 20) + nl + ccr_seq + nl)
                        out["ccr.tsv"] += ("Gene\t" + cluster_id + "\t" + strand + "\t" + t_chr + "\t" + str(t_start) + "\t" +
                                           str(t_end) + "\t" + str(best_pos - 20) + "\t" + str(best_pos + 20) + "\t" + ccr_seq +
                                           "\t" + str(best_pos) + "\t" + str(n_reads) + "\t" + str(n_t2c_sites) + "\t" +
                                           str(mutation_map.get(best_pos)) + "\t" + fmt(best_val) + "\t" + str(n_t2c) + "\t" +
                                           fmt(fraction) + nl)
                seq = _rc_bytes(t_bytes) if t_is_reverse else t_bytes           # :318-321
                seq_s = "".join(chr(c) for c in seq)
                out["pileup"] += (cluster_id + "\t" + t_chr + "\t" + str(t_start) + "\t" + str(t_end) + "\t" +
                                  ("-" if t_is_reverse else "+") + "\t" + str(n_reads) + "\t" + str(n_t2c) + "\t" +
                                  str(n_t2c_sites) + "\t" + fmt(fraction) + "\t" + seq_s + "\t" + _strand_str(is_reverse[0]) +
                                  "\t" + str(len(seq_s)) + nl)
            t_start, t_end, t_chr = r.pos, r.end(), r.rname                     # :346-357
            n_reads, n_t2c, n_t2c_sites = 1, 0, 0
            is_reverse[0] = False
            mutation_map.clear()
            covered_map.clear()
            running_id += 1
            cluster_id = "cl_" + str(running_id) + "_" + t_chr
            mask = JArray(51)
            n_t2c = _cluster_information(ordinal, r, genome, is_reverse, mutation_map, covered_map, mask, n_t2c)
            t_is_reverse = is_reverse[0]
            t_bytes = bytearray()                                               # :367
            cur = r.pos
            for op, n in r.cigar:                                               # :374-414
                if op == "D" or op == "M":
                    t_bytes = t_bytes + bytearray(fetch(r.rname, cur, cur + n - 1))
                if op != "I":
                    cur += n
        else:
            t_chr = r.rname                                                     # :419
            if r.end() > t_end:                                                 # :421
                cur = r.pos
                for op, n in r.cigar:
                    if (cur + n - 1) < t_end:                                   # :429-436
                        if op != "I":
                            cur += n
                        continue
                    if op == "D" or op == "M":
                        add = bytearray(fetch(r.rname, cur, cur + n - 1))
                        overhang = t_end - cur + 1
                        if overhang > 0:                                        # mergeByteSubArrays (:453-457)
                            t_bytes = t_bytes + add[overhang:n]
                        else:                                                   # mergeByteArrays(additionalNucs, tempClusterBytes)
                            t_bytes = add + t_bytes
                    t_end = r.end()                                             # :480
                    if op != "I":
                        cur += n
            n_reads += 1
            n_t2c = _cluster_information(ordinal, r, genome, is_reverse, mutation_map, covered_map, mask, n_t2c)
            if is_reverse[0] is not None and t_is_reverse != is_reverse[0]:
                double_stranded += 1
                is_reverse[0] = None
    out["report"] = ("Double stranded clusters found: " + str(double_stranded) + nl +
                     "Loci found that are SNPs: " + str(snp_count) + nl +
                     str(skipped_due_indel) + " insertion or deletion skipped" + nl +
                     "T-C mutations identified as SNPs: " + str(snp_hit) + nl +
                     "T-C mutations identified as SNVs (100% T-C in 1 site): " + str(high_frequent_error) + nl)
    for v in afi:                                                               # :531-536
        out["sitefrequency"] += fmt(_jdiv(v, num_crosslinked)) + nl
    for j in range(51):                                                         # :538-543
        out["sitepositions"] += fmt(_jdiv(float(allele_positions[j]), num_allele_positions)) + nl
    return out


# ---------------------------------------------------------------------------------------------------------
# CombineGenomeTranscript (utils/postprocessing/CombineGenomeTranscript.java): transcript hits lifted to genomic
# coordinates (cigars with N across introns) and merged with the genomic hits.  Literal restatement, statement by
# statement; test infrastructure like everything in this file.
# ---------------------------------------------------------------------------------------------------------
def java_split(s: str, sep: str) -> List[str]:
    """String.split(regex) for a one-character literal separator: trailing empty strings are removed."""
    parts = s.split(sep)
    while parts and parts[-1] == "":
        parts.pop()
    return parts if parts else ([""] if s == "" else [])


def java_parse_int(s: str) -> int:
    """Integer.parseInt: optional sign, decimal digits only, 32-bit range; anything else kills the tool."""
    body = s[1:] if s[:1] in "+-" else s
    if not body or not all("0" <= c <= "9" for c in body):
        raise ReferenceWouldThrow(-1, f"NumberFormatException: {s!r}")
    v = int(s)
    if not -2 ** 31 <= v < 2 ** 31:
        raise ReferenceWouldThrow(-1, f"NumberFormatException: {s!r}")
    return v


def liftover_hit(ref_name: str, aln_start: int, aln_end: int, read_len: int, cigar: str):
    """One transcript hit (CombineGenomeTranscript.java:146-474).  -> (newGenomicPositionStart or -1, newGenomicCigar,
    missedTranscriptAlignments increment)."""
    f = java_split(ref_name, "|")                                          # :148
    if len(f) < 6:
        raise ReferenceWouldThrow(-1, "ArrayIndexOutOfBoundsException: transcript name without six |-separated fields")
    exon_starts = sorted(java_split(f[3], ";"))                            # :172-175 Arrays.sort on STRINGS
    exon_ends = sorted(java_split(f[4], ";"))
    strand = f[5]
    new_start, new_cigar, missed = -1, "", 0
    length_passed = 0
    has_indel = "D" in cigar or "I" in cigar
    n = len(exon_starts)

    def st(i):
        return java_parse_int(exon_starts[i])

    def en(i):
        if i >= len(exon_ends):
            raise ReferenceWouldThrow(-1, "ArrayIndexOutOfBoundsException: fewer exon ends than starts")
        return java_parse_int(exon_ends[i])

    if strand == "1":                                                      # :219-391
        for i in range(n):
            tmp = length_passed
            length_passed += en(i) - st(i) + 1
            if aln_start <= length_passed:
                if new_start == -1:
                    new_start = st(i) + (aln_start - tmp) - 1
            if aln_end <= length_passed:
                if new_start >= st(i):
                    new_cigar = cigar
                else:
                    new_cigar += str(aln_end - tmp) + "M"
                break
            elif new_start != -1:
                if has_indel:
                    missed += 1
                    break
                if new_start >= st(i):
                    new_cigar += str(en(i) - new_start + 1) + "M"
                else:
                    new_cigar += str(en(i) - st(i) + 1) + "M"
                if i < n - 1:
                    intron = st(i + 1) - en(i) - 1
                    if intron <= 0:
                        break
                    new_cigar += str(intron) + "N"
                else:
                    break
    elif strand == "-1":                                                   # :392-473
        new_end = -1
        for i in range(n - 1, -1, -1):
            tmp = length_passed
            length_passed += en(i) - st(i) + 1
            if aln_start <= length_passed:
                if new_end == -1:
                    new_end = en(i) - (aln_start - tmp) + 1
            if aln_end <= length_passed:
                if new_end <= en(i):
                    new_cigar = cigar
                    new_start = new_end - read_len + 1
                else:
                    if has_indel:
                        missed += 1
                        break
                    new_cigar = str(aln_end - tmp) + "M" + new_cigar
                    new_start = en(i) - (aln_end - tmp) + 1
                break
            elif new_end != -1:
                if has_indel:
                    missed += 1
                    break
                if new_end < en(i):
                    new_cigar = str(new_end - st(i) + 1) + "M" + new_cigar
                else:
                    new_cigar = str(en(i) - st(i) + 1) + "M" + new_cigar
                if i >= 1:
                    intron = st(i) - en(i - 1) - 1
                    if intron <= 0:
                        break
                    new_cigar = str(intron) + "N" + new_cigar
                else:
                    break
    return new_start, new_cigar, missed


_RC = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")          # SequenceUtil.complement: other symbols stay as they are


def combine(genome_names: List[str], sort_order: str, genome_recs: List[dict], transcript_recs: List[dict]):
    """combine() + printReadsToBamFile (CombineGenomeTranscript.java:36-666) on records given as dicts
    {name, flag, rname, pos, cigar, seq, qual, mapq}; the transcript records are name-grouped as in a queryname-sorted
    BAM.  -> (output records in the order htsjdk's writer emits them, stats dict)."""
    out = [dict(r) for r in genome_recs]                                   # :53-60
    mapped, spliced, missed_total = len(out), 0, 0
    index = {n: i for i, n in enumerate(genome_names)}
    lifted = []

    def flush(group):                                                      # printReadsToBamFile :598-666
        nonlocal mapped
        if not group:
            return
        if any(p != group["pos"][0] for p in group["pos"]):
            return
        rec = dict(group["recs"][group["primary"]])
        f = java_split(rec["rname"], "|")
        if "chr" + f[2] not in index:
            return
        chrom = "M" if f[2] == "MT" else f[2]
        rec["rname"] = "chr" + chrom if "chr" + chrom in index else "*"
        rec["pos"] = group["pos"][group["primary"]]
        rec["cigar"] = group["cigars"][group["primary"]]
        rec["mapq"] = 10
        if f[5] == "-1":
            rec["flag"] = rec["flag"] - 16 if rec["flag"] & 16 else rec["flag"] + 16
            rec["seq"] = rec["seq"].translate(_RC)[::-1]
        lifted.append(rec)
        mapped += 1

    group, name_tmp = None, ""
    for r in transcript_recs:
        if r["rname"] == "*":                                              # :105
            continue
        if name_tmp != r["name"]:                                          # :137-144
            flush(group)
            group, name_tmp = None, r["name"]
        aln_end = r["pos"] + ref_length(r["cigar"]) - 1 if not (r["flag"] & 4) else 0
        new_start, new_cigar, missed = liftover_hit(r["rname"], r["pos"], aln_end, len(r["seq"]), r["cigar"])
        missed_total += missed
        if new_start == -1:                                                # :476
            continue
        if "N" in new_cigar:
            spliced += 1
        if group is None:
            group = {"genes": [], "pos": [], "cigars": [], "recs": [], "primary": 0}
        if not (r["flag"] & 0x100):
            group["primary"] = len(group["genes"])
        group["genes"].append(java_split(r["rname"], "|")[0])
        group["pos"].append(new_start)
        group["cigars"].append(new_cigar)
        group["recs"].append(r)
    flush(group)
    out += lifted
    if sort_order == "coordinate":
        def key(r):       # SAMRecordCoordinateComparator: reference index (unmapped last), start, strand, name, flags, mapq
            ri = index.get(r["rname"], -1)
            return (ri if ri >= 0 else 1 << 31, r["pos"], 1 if r["flag"] & 16 else 0, r["name"], r["flag"], r["mapq"])
        out.sort(key=key)
    return out, {"mapped_reads": mapped, "spliced_reads": spliced, "missed_transcript_alignments": missed_total,
                 "lifted": len(lifted)}


def ref_length(cigar: str) -> int:
    return sum(n for op, n in parse_cigar(cigar) if op in "MDN=X") if cigar and cigar != "*" else 0
