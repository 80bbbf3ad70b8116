"""File formats either side of the hot path.

* writers (test / workload tooling, pure Python): FASTA + .fai, BGZF/BAM -- so that coordinate-sorted inputs for the
  tools can be produced in an image that has no samtools;
* readers: thin wrappers over the native host batcher of libparasuite_b200.so (csrc/bam_batcher.cpp): FASTA -> packed
  reference, BAM -> SoA batches.  The batcher is host code and works without a GPU.
"""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import abi
from .batch import CIGAR_OPS, PackedReference, ReadBatch, Record, parse_cigar

_NIB = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}


# ---- writers ------------------------------------------------------------------------------------------------
def write_fasta(path: str, contigs: Sequence[Tuple[str, bytes]], line_width: int = 60) -> None:
    """FASTA with `line_width` bases per line plus the .fai index htsjdk / ps_fasta_pack need."""
    fai = []
    with open(path, "wb") as f:
        for name, seq in contigs:
            f.write(b">" + name.encode() + b"\n")
            off = f.tell()
            for k in range(0, len(seq), line_width):
                f.write(seq[k:k + line_width] + b"\n")
            fai.append((name, len(seq), off, line_width, line_width + 1))
    with open(path + ".fai", "w") as f:
        for e in fai:
            f.write("\t".join(str(x) for x in e) + "\n")


def _bgzf_block(data: bytes, level: int = 6) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    bsize = len(comp) + 25
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize) + comp +
            struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def _reg2bin(beg: int, end: int) -> int:
    end -= 1
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return base + (beg >> shift)
    return 0


def encode_bam_record(rec: Record, ref_ids: dict, name: bytes = b"r", mapq: int = 255) -> bytes:
    ops = parse_cigar(rec.cigar)
    L = len(rec.seq)
    ref_id = ref_ids.get(rec.rname, -1)
    pos = rec.pos - 1
    rlen = sum(n for op, n in ops if op in (0, 2, 3, 7, 8))
    bin_ = _reg2bin(max(pos, 0), max(pos, 0) + max(rlen, 1))
    seq = bytearray((L + 1) // 2)
    for k, ch in enumerate(rec.seq):
        nib = _NIB.get(chr(ch).upper(), 15)
        seq[k >> 1] |= nib << (4 if k % 2 == 0 else 0)
    qual = bytes(rec.qual) if len(rec.qual) == L else b"\xff" * L
    body = struct.pack("<iiBBHHHIiii", ref_id, pos, len(name) + 1, mapq, bin_, len(ops), rec.flag & 0xFFFF, L, -1, -1, 0)
    body += name + b"\0" + b"".join(struct.pack("<I", (n << 4) | op) for op, n in ops) + bytes(seq) + qual
    return struct.pack("<I", len(body)) + body


def write_bam(path: str, contigs: Sequence[Tuple[str, int]], records: Iterable[Record], sort_order: str = "coordinate",
              block_bytes: int = 0xFF00, level: int = 1, names: Optional[Sequence[bytes]] = None) -> int:
    """Minimal BAM writer (one read group-less header; records in the order given; read names r<k> unless `names` gives
    them).  Returns the record count."""
    text = f"@HD\tVN:1.4\tSO:{sort_order}\n" + "".join(f"@SQ\tSN:{n}\tLN:{ln}\n" for n, ln in contigs)
    hdr = b"BAM\1" + struct.pack("<I", len(text)) + text.encode() + struct.pack("<I", len(contigs))
    for n, ln in contigs:
        hdr += struct.pack("<I", len(n) + 1) + n.encode() + b"\0" + struct.pack("<I", ln)
    ref_ids = {n: i for i, (n, _) in enumerate(contigs)}
    count = 0
    with open(path, "wb") as f:
        pend = bytearray(hdr)

        def flush(final=False):
            nonlocal pend
            while len(pend) >= block_bytes or (final and pend):
                f.write(_bgzf_block(bytes(pend[:block_bytes]), level))
                del pend[:block_bytes]

        for k, rec in enumerate(records):
            pend += encode_bam_record(rec, ref_ids, names[k] if names is not None else b"r%d" % k)
            count += 1
            flush()
        flush(final=True)
        f.write(_bgzf_block(b""))       # EOF marker
    return count


def read_bam_records(path: str):
    """Pure-Python BAM decoder for tests and small files: -> (header text, [(name, length)], [record dict]).  A record
    dict holds name, flag, rname, pos (1-based), mapq, cigar, seq, qual (bytes), mate fields and the raw tag bytes."""
    import gzip
    data = gzip.open(path, "rb").read()
    assert data[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<I", data, 4)
    text = data[8:8 + l_text].rstrip(b"\0").decode()
    o = 8 + l_text
    n_ref, = struct.unpack_from("<I", data, o)
    o += 4
    refs = []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<I", data, o)
        name = data[o + 4:o + 4 + ln - 1].decode()
        length, = struct.unpack_from("<I", data, o + 4 + ln)
        refs.append((name, length))
        o += 8 + ln
    nib = "=ACMGRSVTWYHKDBN"
    recs = []
    while o + 4 <= len(data):
        bs, = struct.unpack_from("<I", data, o)
        ref_id, pos, l_name, mapq, _bin, n_cig, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHIiii", data, o + 4)
        q = o + 36
        name = data[q:q + l_name - 1].decode()
        q += l_name
        ops = struct.unpack_from("<%dI" % n_cig, data, q)
        q += 4 * n_cig
        sb = data[q:q + (l_seq + 1) // 2]
        q += (l_seq + 1) // 2
        seq = "".join(nib[(sb[k >> 1] >> (4 if k % 2 == 0 else 0)) & 15] for k in range(l_seq))
        qual = data[q:q + l_seq]
        q += l_seq
        recs.append({"name": name, "flag": flag, "rname": refs[ref_id][0] if ref_id >= 0 else "*", "pos": pos + 1, "mapq": mapq,
                     "cigar": "".join(f"{c >> 4}{CIGAR_OPS[c & 15]}" for c in ops) or "*", "seq": seq.encode(), "qual": qual,
                     "next_ref": nref, "next_pos": npos + 1, "tlen": tlen, "tags": data[q:o + 4 + bs]})
        o += 4 + bs
    return text, refs, recs


def write_sam(path: str, contigs: Sequence[Tuple[str, int]], records: Iterable[Record], sort_order: str = "coordinate") -> None:
    """The same records as SAM text (htsjdk opens SAM and BAM through one factory, ErrorProfiling.java:104-107)."""
    with open(path, "w") as f:
        f.write(f"@HD\tVN:1.4\tSO:{sort_order}\n")
        for name, length in contigs:
            f.write(f"@SQ\tSN:{name}\tLN:{length}\n")
        for k, r in enumerate(records):
            q = bytes(r.qual)
            missing = len(q) == 0 or q[0] == 0xFF
            qual = "*" if missing else "".join(chr(33 + (b & 0xFF)) if (b & 0xFF) + 33 < 127 else "~" for b in q)
            seq = r.seq.decode() if len(r.seq) else "*"
            f.write("\t".join([f"r{k}", str(r.flag), r.rname, str(r.pos), "30", r.cigar if r.cigar else "*", "*", "0", "0", seq,
                               qual]) + "\n")


def batch_to_records(batch: ReadBatch, ref: PackedReference) -> List[Record]:
    """Inverse of the packers for uniform or ragged batches (used to write synthetic workloads as BAM files)."""
    out = []
    T = abi.PS_TILE_READS
    exc = {}
    for t in range(batch.n_tiles):
        for e in batch.exc[int(batch.tile_exc_off[t]):int(batch.tile_exc_off[t + 1])]:
            exc.setdefault(t * T + (int(e) >> 16), set()).add(int(e) & 0xFFFF)
    ob = oq = oc = 0
    coff = ref.contig_off
    for r in range(batch.n_reads):
        m = int(batch.meta[r])
        L, nc, fl = m & 0xFFFF, (m >> 16) & 0xFF, m >> 24
        if r % T == 0 and not (batch.uniform_len and batch.uniform_ncigar):
            t = r // T
            ob, oq, oc = int(batch.tile_base_off[t]), int(batch.tile_qual_off[t]), int(batch.tile_cigar_off[t])
        elif batch.uniform_len and batch.uniform_ncigar:
            ob, oq, oc = r * ((L + 3) // 4), r * L, r * nc
        codes = [(int(batch.bases2[ob + (k >> 2)]) >> (2 * (k & 3))) & 3 for k in range(L)]
        seq = bytearray(b"ACGT"[c] for c in codes)
        for p in exc.get(r, ()):
            seq[p] = ord("N")
        qual = bytes(batch.qual[oq:oq + L])
        cig = "".join(f"{int(c) >> 4}{CIGAR_OPS[int(c) & 15]}" for c in batch.cigar[oc:oc + nc]) or "*"
        flag = (0x4 if fl & abi.PS_RF_UNMAPPED else 0) | (0x10 if fl & abi.PS_RF_REVERSE else 0) | \
               (0x400 if fl & abi.PS_RF_DUPLICATE else 0)
        if fl & abi.PS_RF_POS_ZERO:
            rname, pos = ref.names[0], 0
        else:
            g = int(batch.ref_start[r])
            ci = int(np.searchsorted(coff, g, side="right")) - 1
            ci = min(max(ci, 0), len(ref.names) - 1)
            rname, pos = ref.names[ci], g - int(coff[ci]) + 1
        out.append(Record(flag, rname, pos, cig, bytes(seq), qual))
        ob += (L + 3) // 4
        oq += L
        oc += nc
    return out


# ---- readers (native) -----------------------------------------------------------------------------------------
class PackedFasta:
    """ps_packed_fasta: the packed reference built natively from FASTA + .fai (host memory)."""

    def __init__(self, path: str):
        self.lib = abi.load_library()
        h = C.c_void_p()
        st = self.lib.ps_fasta_pack(path.encode(), C.byref(h))
        self.h = h
        if st != abi.PS_OK:
            msg = self.lib.ps_fasta_error(h).decode() if h else self.lib.ps_strerror(st).decode()
            self.close()
            raise abi.PsError(st, msg)
        v = self.lib.ps_fasta_reference(h).contents
        self.n_contigs = int(v.n_contigs)
        self.names = [self.lib.ps_fasta_contig_name(h, i).decode() for i in range(self.n_contigs)]
        off = np.ctypeslib.as_array(C.cast(v.contig_off, C.POINTER(C.c_uint64)), shape=(self.n_contigs + 1,)).copy()
        self.lengths = [int(off[i + 1] - off[i]) for i in range(self.n_contigs)]
        self._view = v

    def reference(self) -> PackedReference:
        """Copy into the numpy container the rest of the Python layer uses."""
        v = self._view
        w2, w1 = PackedReference.words_for(int(v.n_bases))
        seq2 = np.ctypeslib.as_array(C.cast(v.seq2, C.POINTER(C.c_uint32)), shape=(w2,)).copy()
        inv = np.ctypeslib.as_array(C.cast(v.inv, C.POINTER(C.c_uint32)), shape=(w1,)).copy()
        return PackedReference(self.names, self.lengths, seq2, inv)

    def close(self):
        if getattr(self, "h", None):
            self.lib.ps_fasta_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BamBatcher:
    """ps_bam: iterate a coordinate-sorted BAM as SoA batches (numpy copies of the native slabs).
    any_contig_order=True: take a header that lists the contigs in another order than the FASTA (contig_order gives it,
    Context.set_contig_order keys the pileup in it); otherwise such a file raises PS_ERR_UNSUPPORTED."""

    def __init__(self, path: str, fasta: PackedFasta, max_batch_reads: int = 0, threads: int = 0,
                 any_contig_order: bool = False):
        self.lib = abi.load_library()
        self._fasta = fasta
        h = C.c_void_p()
        flags = abi.PS_BAM_ANY_CONTIG_ORDER if any_contig_order else 0
        st = self.lib.ps_bam_open_ex(C.byref(h), path.encode(), fasta.h, max_batch_reads, threads, flags)
        self.h = h
        if st != abi.PS_OK:
            msg = self.lib.ps_bam_error(h).decode() if h else self.lib.ps_strerror(st).decode()
            self.close()
            raise abi.PsError(st, msg)

    @property
    def contig_order(self) -> List[int]:
        """FASTA indices of the header's @SQ contigs in header order, contigs the FASTA lacks left out: the order the
        records of a coordinate-sorted file follow (Context.set_contig_order)."""
        n = int(self.lib.ps_bam_contig_order(self.h, None, 0))
        if n < 0:
            raise abi.PsError(n, self.lib.ps_strerror(n).decode())
        a = np.zeros(max(n, 1), dtype=np.uint32)
        self.lib.ps_bam_contig_order(self.h, a.ctypes.data, n)
        return [int(x) for x in a[:n]]

    def __iter__(self):
        return self

    def __next__(self) -> ReadBatch:
        s = abi.ps_read_batch()
        k = self.lib.ps_bam_next(self.h, C.byref(s))
        if k < 0:
            raise abi.PsError(k, self.lib.ps_bam_error(self.h).decode())
        if k == 0:
            raise StopIteration
        n = int(s.n_reads)
        nt = (n + abi.PS_TILE_READS - 1) // abi.PS_TILE_READS

        def arr(ptr, ctype, count):
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(count,)).copy()

        return ReadBatch(
            n, arr(s.meta, C.c_uint32, n), arr(s.ref_start, C.c_uint32, n), arr(s.bases2, C.c_uint8, s.bases_bytes + 64),
            arr(s.qual, C.c_uint8, s.qual_bytes + 64), arr(s.cigar, C.c_uint32, s.cigar_count + 16),
            arr(s.tile_base_off, C.c_uint64, nt + 1), arr(s.tile_qual_off, C.c_uint64, nt + 1),
            arr(s.tile_cigar_off, C.c_uint64, nt + 1), arr(s.tile_exc_off, C.c_uint32, nt + 1),
            arr(s.exc, C.c_uint32, s.exc_count + 16), uniform_len=int(s.uniform_len), uniform_ncigar=int(s.uniform_ncigar),
            bases_bytes=int(s.bases_bytes), qual_bytes=int(s.qual_bytes), cigar_count=int(s.cigar_count),
            exc_count=int(s.exc_count), past_end=int(s.past_end))

    def close(self):
        if getattr(self, "h", None):
            self.lib.ps_bam_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
