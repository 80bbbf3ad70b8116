"""Host-side SoA containers: the packed reference and the read batch of include/parasuite_b200.h.

These hold numpy arrays and hand out the C structs.  The record-by-record packers here are the
small-input path (tests, golden vectors); bulk inputs come from the native batcher (BAM -> SoA)
and the synthetic generator, which fill the same arrays.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import abi

CIGAR_OPS = "MIDNSHP=X"
_CODE = np.full(256, 255, dtype=np.uint8)
for _ch, _v in (("A", 0), ("C", 1), ("G", 2), ("T", 3), ("a", 0), ("c", 1), ("g", 2), ("t", 3)):
    _CODE[ord(_ch)] = _v

PAD_WORDS = 8  # >= 16 readable bytes past the last used word (header contract)


def _ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


class PackedReference:
    """2-bit + invalid-bit packing of all contigs in one global coordinate space."""

    def __init__(self, names: List[str], lengths: List[int], seq2: np.ndarray, inv: np.ndarray):
        self.names = list(names)
        self.lengths = [int(x) for x in lengths]
        self.contig_off = np.zeros(len(names) + 1, dtype=np.uint64)
        self.contig_off[1:] = np.cumsum(np.asarray(self.lengths, dtype=np.uint64))
        self.n_bases = int(self.contig_off[-1])
        if self.n_bases >= (1 << 32):
            raise ValueError("reference longer than 2^32 bases is not supported (uint32 global offsets)")
        self.seq2 = np.ascontiguousarray(seq2, dtype=np.uint32)
        self.inv = np.ascontiguousarray(inv, dtype=np.uint32)
        self._index = {n: i for i, n in enumerate(self.names)}

    @staticmethod
    def words_for(n_bases: int) -> Tuple[int, int]:
        return (n_bases + 15) // 16 + PAD_WORDS, (n_bases + 31) // 32 + PAD_WORDS

    @classmethod
    def from_contigs(cls, contigs: Sequence[Tuple[str, bytes]]) -> "PackedReference":
        names = [n for n, _ in contigs]
        lengths = [len(s) for _, s in contigs]
        raw = np.frombuffer(b"".join(s for _, s in contigs), dtype=np.uint8)
        return cls.from_ascii(names, lengths, raw)

    @classmethod
    def from_ascii(cls, names, lengths, raw: np.ndarray) -> "PackedReference":
        n = int(raw.size)
        w2, w1 = cls.words_for(n)
        code = _CODE[raw]
        invalid = code == 255
        code = np.where(invalid, 0, code).astype(np.uint32)
        pad2 = np.zeros(w2 * 16, dtype=np.uint32)
        pad2[:n] = code
        seq2 = np.zeros(w2, dtype=np.uint32)
        lanes = pad2.reshape(w2, 16)
        for k in range(16):
            seq2 |= lanes[:, k] << np.uint32(2 * k)
        pad1 = np.zeros(w1 * 32, dtype=np.uint8)
        pad1[:n] = invalid
        inv = np.packbits(pad1.reshape(w1, 32), axis=1, bitorder="little").view("<u4").reshape(w1)
        return cls(names, lengths, seq2, inv)

    def contig_index(self, name: str) -> int:
        return self._index[name]

    def as_struct(self) -> abi.ps_reference:
        s = abi.ps_reference()
        s.n_bases = self.n_bases
        s.seq2 = _ptr(self.seq2)
        s.inv = _ptr(self.inv)
        s.n_contigs = len(self.names)
        s.contig_off = _ptr(self.contig_off)
        return s


@dataclass
class Record:
    """One alignment record as htsjdk presents it (the fields the two loops read)."""
    flag: int
    rname: str          # "*" when none
    pos: int            # 1-based, 0 = none
    cigar: str          # SAM text, "*" when none
    seq: bytes          # ASCII
    qual: bytes         # raw phred bytes; b"" or first byte 0xFF = missing


def parse_cigar(text: str) -> List[Tuple[int, int]]:
    if text in ("*", ""):
        return []
    out, num = [], 0
    for ch in text:
        if ch.isdigit():
            num = num * 10 + ord(ch) - 48
        else:
            out.append((CIGAR_OPS.index(ch), num))
            num = 0
    return out


class ReadBatch:
    """SoA read batch on the host (numpy) -- see ps_read_batch in include/parasuite_b200.h."""

    FIELDS = ("meta", "ref_start", "bases2", "qual", "cigar", "tile_base_off", "tile_qual_off", "tile_cigar_off",
              "tile_exc_off", "exc")

    def __init__(self, n_reads, meta, ref_start, bases2, qual, cigar, tile_base_off, tile_qual_off, tile_cigar_off,
                 tile_exc_off, exc, uniform_len=0, uniform_ncigar=0, bases_bytes=None, qual_bytes=None,
                 cigar_count=None, exc_count=None, past_end=0):
        self.n_reads = int(n_reads)
        self.past_end = int(past_end)      # 1 + ordinal of the first record past its contig's end (ps_read_batch.past_end)
        self.meta = meta
        self.ref_start = ref_start
        self.bases2 = bases2
        self.qual = qual
        self.cigar = cigar
        self.tile_base_off = tile_base_off
        self.tile_qual_off = tile_qual_off
        self.tile_cigar_off = tile_cigar_off
        self.tile_exc_off = tile_exc_off
        self.exc = exc
        self.uniform_len = int(uniform_len)
        self.uniform_ncigar = int(uniform_ncigar)
        self.bases_bytes = int(tile_base_off[-1]) if bases_bytes is None else int(bases_bytes)
        self.qual_bytes = int(tile_qual_off[-1]) if qual_bytes is None else int(qual_bytes)
        self.cigar_count = int(tile_cigar_off[-1]) if cigar_count is None else int(cigar_count)
        self.exc_count = int(tile_exc_off[-1]) if exc_count is None else int(exc_count)
        # longest read: a hint for the kernels' choice of row geometry on ragged batches
        self.max_len = self.uniform_len or (int((np.asarray(meta[:self.n_reads]) & 0xFFFF).max()) if self.n_reads else 0)

    @property
    def n_tiles(self) -> int:
        return (self.n_reads + abi.PS_TILE_READS - 1) // abi.PS_TILE_READS

    def as_struct(self) -> abi.ps_read_batch:
        s = abi.ps_read_batch()
        s.n_reads = self.n_reads
        for f in self.FIELDS:
            setattr(s, f, _ptr(getattr(self, f)))
        s.uniform_len = self.uniform_len
        s.uniform_ncigar = self.uniform_ncigar
        s.bases_bytes = self.bases_bytes
        s.qual_bytes = self.qual_bytes
        s.cigar_count = self.cigar_count
        s.exc_count = self.exc_count
        s.max_len = self.max_len
        s.past_end = self.past_end
        return s

    def algorithmic_bytes(self, with_qual: bool = True) -> int:
        """SURVEY 8(d): ceil(L/4) + L + 4*n_cigar + 4 + 4 + ceil(R/4) summed over reads."""
        L = (self.meta & 0xFFFF).astype(np.int64)
        total = int(((L + 3) // 4).sum()) + 4 * self.cigar_count + 8 * self.n_reads
        if with_qual:
            total += int(L.sum())
        op = self.cigar[: self.cigar_count] & 15
        ln = (self.cigar[: self.cigar_count] >> 4).astype(np.int64)
        refc = np.isin(op, (0, 2, 3, 7, 8))
        if self.uniform_ncigar:
            R = (ln * refc).reshape(self.n_reads, self.uniform_ncigar).sum(axis=1)
        else:
            ncig = ((self.meta >> 16) & 0xFF).astype(np.int64)
            idx = np.repeat(np.arange(self.n_reads), ncig)
            R = np.bincount(idx, weights=(ln * refc), minlength=self.n_reads).astype(np.int64)
        total += int(((R + 3) // 4).sum())
        return total

    @classmethod
    def from_records(cls, records: Sequence[Record], ref: PackedReference) -> "ReadBatch":
        """Pack records exactly as the native BAM batcher does (small inputs; pure Python loop)."""
        n = len(records)
        T = abi.PS_TILE_READS
        n_tiles = (n + T - 1) // T
        past_end = 0
        meta = np.zeros(n, dtype=np.uint32)
        ref_start = np.zeros(n, dtype=np.uint32)
        bases = bytearray()
        quals = bytearray()
        cig: List[int] = []
        exc: List[int] = []
        tb = np.zeros(n_tiles + 1, dtype=np.uint64)
        tq = np.zeros(n_tiles + 1, dtype=np.uint64)
        tc = np.zeros(n_tiles + 1, dtype=np.uint64)
        te = np.zeros(n_tiles + 1, dtype=np.uint32)
        lens = set()
        ncigs = set()
        for r, rec in enumerate(records):
            if r % T == 0:
                t = r // T
                tb[t], tq[t], tc[t], te[t] = len(bases), len(quals), len(cig), len(exc)
            ops = parse_cigar(rec.cigar)
            L = len(rec.seq)
            fl = 0
            if rec.flag & 0x4:
                fl |= abi.PS_RF_UNMAPPED
            if rec.flag & 0x10:
                fl |= abi.PS_RF_REVERSE
            if rec.flag & 0x400:
                fl |= abi.PS_RF_DUPLICATE
            if rec.pos == 0:
                fl |= abi.PS_RF_POS_ZERO
            if len(rec.qual) == 0 or rec.qual[0] == 0xFF:
                fl |= abi.PS_RF_QUAL_MISSING
            if len(ops) > 255:
                fl |= abi.PS_RF_CIGAR_OVERFLOW
                ops = []
            codes = _CODE[np.frombuffer(rec.seq, dtype=np.uint8)] if L else np.zeros(0, np.uint8)
            bad = np.nonzero(codes == 255)[0]
            if bad.size:
                fl |= abi.PS_RF_HAS_INVALID
                exc.extend(((r % T) << 16) | int(p) for p in bad)
            codes = np.where(codes == 255, 0, codes).astype(np.uint8)
            padded = np.zeros((L + 3) // 4 * 4, dtype=np.uint8)
            padded[:L] = codes
            q4 = padded.reshape(-1, 4)
            bases += (q4[:, 0] | (q4[:, 1] << 2) | (q4[:, 2] << 4) | (q4[:, 3] << 6)).astype(np.uint8).tobytes()
            qb = bytes(rec.qual) if len(rec.qual) == L else bytes([0xFF]) * L
            quals += qb
            cig.extend((ln << 4) | op for op, ln in ops)
            R = sum(ln for op, ln in ops if op in (0, 2, 3, 7, 8))
            if not (fl & (abi.PS_RF_UNMAPPED | abi.PS_RF_POS_ZERO)):
                if rec.rname not in ref._index:
                    fl |= abi.PS_RF_REF_RANGE
                else:
                    ci = ref.contig_index(rec.rname)
                    g = int(ref.contig_off[ci]) + rec.pos - 1
                    # htsjdk getSubsequenceAt(chr, pos, pos+R-1) throws iff stop > contig length
                    if rec.pos - 1 + R > ref.lengths[ci]:
                        fl |= abi.PS_RF_REF_RANGE
                    if R == 0 and rec.pos > ref.lengths[ci] and not fl & abi.PS_RF_CIGAR_OVERFLOW:
                        # no reference span, POS past the contig's end: as the native batcher (ps_read_batch.past_end)
                        g = int(ref.contig_off[ci]) + ref.lengths[ci] - 1
                        past_end = past_end or r + 1
                    ref_start[r] = min(g, 0xFFFFFFFF)
            meta[r] = (L & 0xFFFF) | ((len(ops) & 0xFF) << 16) | (fl << 24)
            lens.add(L)
            ncigs.add(len(ops))
        tb[n_tiles], tq[n_tiles], tc[n_tiles], te[n_tiles] = len(bases), len(quals), len(cig), len(exc)
        pad = 64
        bases2 = np.frombuffer(bytes(bases) + bytes(pad), dtype=np.uint8).copy()
        qual = np.frombuffer(bytes(quals) + bytes(pad), dtype=np.uint8).copy()
        cigar = np.asarray(cig + [0] * 16, dtype=np.uint32)
        exc_a = np.asarray(exc + [0] * 16, dtype=np.uint32)
        ul = lens.pop() if len(lens) == 1 else 0
        uc = ncigs.pop() if len(ncigs) == 1 else 0
        return cls(n, meta, ref_start, bases2, qual, cigar, tb, tq, tc, te, exc_a, uniform_len=ul, uniform_ncigar=uc,
                   bases_bytes=len(bases), qual_bytes=len(quals), cigar_count=len(cig), exc_count=len(exc),
                   past_end=past_end)
