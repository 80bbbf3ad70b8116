"""Context + batch-level calls over the C ABI (host side of the drop-in boundary).

`Context` owns one GPU (one process per GPU under torch.distributed).  All compute goes through
libparasuite_b200.so; there is no CPU path here.  torch is used only as plumbing: device memory for
resident batches, streams, and the NCCL all-reduce of the count vector.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import abi
from .batch import PackedReference, ReadBatch


def _check(lib, ctx, st, fault=None):
    if st == abi.PS_OK:
        return
    msg = lib.ps_last_error(ctx).decode() if ctx else lib.ps_strerror(st).decode()
    if st == abi.PS_ERR_REFERENCE_WOULD_THROW:
        raise abi.ReferenceWouldThrow(st, msg, fault)
    raise abi.PsError(st, msg or lib.ps_strerror(st).decode(), fault)


_BASE_CODE = {"A": 0, "C": 1, "G": 2, "T": 3}


def substitution_mask(substitutions) -> int:
    """ps_track_opts.substitutions of an iterable of "X>Y" strings (X != Y, both of ACGT, strand orientation); None: 0,
    which selects all twelve."""
    if substitutions is None:
        return 0
    if isinstance(substitutions, str):
        substitutions = [substitutions]
    mask = 0
    for t in substitutions:
        parts = str(t).strip().upper().split(">")
        if len(parts) != 2 or parts[0] not in _BASE_CODE or parts[1] not in _BASE_CODE or parts[0] == parts[1]:
            raise ValueError(f"not a substitution: {t!r} (expected X>Y with X != Y of A, C, G, T)")
        mask |= 1 << (4 * _BASE_CODE[parts[0]] + _BASE_CODE[parts[1]])
    if not mask:
        raise ValueError("no substitution selected")
    return mask


def track_opts(base_counts: bool, min_coverage: int, min_events: int, substitutions) -> Optional[abi.ps_track_opts]:
    """The ps_track_opts of the keywords of Context.track, or None for the plain track"""
    if not base_counts:
        return None
    if min(int(min_coverage), int(min_events)) < 0:
        raise ValueError("min_coverage and min_events must be >= 0")
    return abi.ps_track_opts(1, int(min_coverage), int(min_events), substitution_mask(substitutions))


def track_indel_opts(indel_counts: bool, min_indel_depth: int, min_indel_events: int) -> Optional[abi.ps_track_indel_opts]:
    """The ps_track_indel_opts of the indel keywords of Context.track, or None without indel counts"""
    if not indel_counts:
        return None
    if min(int(min_indel_depth), int(min_indel_events)) < 0:
        raise ValueError("min_indel_depth and min_indel_events must be >= 0")
    return abi.ps_track_indel_opts(1, int(min_indel_depth), int(min_indel_events), 0)


def track_filter_opts(min_mapq: int, require_flags: int, exclude_flags: int,
                      min_base_quality: int) -> Optional[abi.ps_track_filter_opts]:
    """The ps_track_filter_opts of the filter keywords of Context.track, or None when all four are 0 (no filter)"""
    vals = (int(min_mapq), int(require_flags), int(exclude_flags), int(min_base_quality))
    if not any(vals):
        return None
    if not 0 <= vals[0] <= 255:
        raise ValueError("min_mapq must be in 0..255")
    if not 0 <= vals[3] <= 255:
        raise ValueError("min_base_quality must be in 0..255")
    if not (0 <= vals[1] <= 0xFFFF and 0 <= vals[2] <= 0xFFFF):
        raise ValueError("require_flags and exclude_flags must be 16-bit flag masks")
    return abi.ps_track_filter_opts(*vals)


def _base_totals_dict(tot) -> dict:
    return {"base_totals": np.array(tot.bases, dtype=np.uint64).reshape(2, 4, 5), "n_base_rows": int(tot.n_rows)}


class DeviceBatch:
    """A ReadBatch resident in HBM (torch tensors hold the memory; the kernels see raw pointers)."""

    def __init__(self, host: ReadBatch, device):
        import torch
        self.n_reads = host.n_reads
        self.host = host
        self._t = {}
        for f in ReadBatch.FIELDS:
            a = getattr(host, f)
            if a is None:
                self._t[f] = None
                continue
            t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8))
            self._t[f] = t.to(device, non_blocking=False)
        s = host.as_struct()
        for f in ReadBatch.FIELDS:
            setattr(s, f, None if self._t[f] is None else self._t[f].data_ptr())
        self.struct = s
        self.nbytes = sum(t.numel() for t in self._t.values() if t is not None)
        # the aux arrays of the track's read filters, when the host batch has them
        aux = {}
        for f in ("sam_flags", "mapq"):
            a = getattr(host, f, None)
            aux[f] = None if a is None else torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).to(device)
        self._aux = aux
        self.aux = abi.ps_read_aux(*(None if aux[f] is None else aux[f].data_ptr() for f in ("sam_flags", "mapq")))


class UploadedBatch:
    """Device-resident view returned by ps_batch_upload (memory owned by the context's staging slots)."""

    def __init__(self, struct, n_reads, source):
        self.struct = struct
        self.n_reads = n_reads
        self._source = source        # keeps the host buffers alive until the copy has completed


class PinnedBatch:
    """A ReadBatch copied into page-locked host memory (what the native batcher fills)."""

    def __init__(self, host: ReadBatch, compact: bool = False):
        """compact=True: the compact host form of ps_read_batch where the batch allows it (uniform length, one cigar op
        per read, the same op everywhere): one flag byte per read instead of the meta word, no cigar stream (7 bytes per
        read less over the host link), and qualities packed 6 bits each when none exceeds 63 (a quarter of their bytes
        less); the upload expands all three on the device."""
        import torch
        self.n_reads = host.n_reads
        self.host = host             # the aux arrays of the track's read filters stay on the host
        self._t = {}
        s = host.as_struct()
        n = host.n_reads
        skip = set()
        self.compact = False
        if compact and n and host.uniform_len and host.uniform_ncigar == 1:
            op = int(host.cigar[0])
            if bool(np.all(np.asarray(host.cigar[:n]) == op)) and op != 0:
                flags = (np.asarray(host.meta[:n]) >> np.uint32(24)).astype(np.uint8)
                t = torch.from_numpy(flags).clone().pin_memory()
                self._t["flags8"] = t
                s.flags8 = t.data_ptr()
                s.uniform_cigar = op
                s.meta = None
                s.cigar = None
                skip = {"meta", "cigar"}
                self.compact = True
        start_sent = 4 * n
        self.compact_start = False
        if compact and n:
            T = abi.PS_TILE_READS
            st = np.asarray(host.ref_start[:n]).astype(np.int64)
            fl = (np.asarray(host.meta[:n]) >> np.uint32(24))
            live = (fl & (abi.PS_RF_UNMAPPED | abi.PS_RF_POS_ZERO)) == 0       # the others carry no defined start
            nt = (n + T - 1) // T
            big = np.int64(1) << 40
            padded = np.full(nt * T, big, dtype=np.int64)
            padded[:n] = np.where(live, st, big)
            base = padded.reshape(nt, T).min(axis=1)
            base = np.where(base == big, 0, base)
            delta = np.where(live, st - np.repeat(base, T)[:n], 0)
            if int(delta.max(initial=0)) <= 0xFFFF and int(delta.min(initial=0)) >= 0 and bool(np.all(st[~live] == st[~live])):
                # reads without a defined start get the tile's base: nothing looks at their start
                t16 = torch.from_numpy(delta.astype(np.uint16).view(np.uint8)).clone().pin_memory()
                tb = torch.from_numpy(base.astype(np.uint32).view(np.uint8)).clone().pin_memory()
                self._t["start16"], self._t["tile_start"] = t16, tb
                s.start16, s.tile_start = t16.data_ptr(), tb.data_ptr()
                s.ref_start = None
                skip = skip | {"ref_start"}
                start_sent = 2 * n + 4 * nt
                self.compact_start = True
        qual_sent = host.qual_bytes
        self.packed_qual = False
        if compact and n and host.uniform_len:
            L = host.uniform_len
            q = np.asarray(host.qual[:n * L]).reshape(n, L)
            missing = ((np.asarray(host.meta[:n]) >> np.uint32(24)) & abi.PS_RF_QUAL_MISSING) != 0
            if int(q.max()) <= 63 and not bool(missing.any()):
                g = (L + 3) // 4
                qp = np.zeros((n, g * 4), dtype=np.uint32)
                qp[:, :L] = q
                qp = qp.reshape(n, g, 4)
                w = qp[:, :, 0] | (qp[:, :, 1] << 6) | (qp[:, :, 2] << 12) | (qp[:, :, 3] << 18)
                packed = np.stack((w & 255, (w >> 8) & 255, w >> 16), axis=2).astype(np.uint8).reshape(-1)
                t = torch.from_numpy(np.ascontiguousarray(packed)).clone().pin_memory()
                self._t["qual6"] = t
                s.qual6 = t.data_ptr()
                s.qual = None
                skip = skip | {"qual"}
                qual_sent = int(packed.size)
                self.packed_qual = True
        for f in ReadBatch.FIELDS:
            a = getattr(host, f)
            if a is None or f in skip:
                continue
            t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).clone().pin_memory()
            self._t[f] = t
            setattr(s, f, t.data_ptr())
        self.struct = s
        per_read = 1 if self.compact else 4 + 4 * host.cigar_count / max(n, 1)
        self.h2d_bytes = int(n * per_read + start_sent + host.bases_bytes + qual_sent + host.exc_count * 4 + (host.n_tiles + 1) * 28)


class Context:
    def __init__(self, device: int = 0):
        self.lib = abi.load_library()
        h = C.c_void_p()
        st = self.lib.ps_create(C.byref(h), device)
        if st != abi.PS_OK:
            raise abi.PsError(st, self.lib.ps_strerror(st).decode())
        self.h = h
        self.device = device
        self.ref: Optional[PackedReference] = None
        self._max_len = 0
        self._infer_q = False
        self._keep = []
        self._pinned_bufs = {}
        self._result_plans = {}

    def close(self):
        if self.h:
            self.lib.ps_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference ------------------------------------------------------------------------------
    def upload_reference(self, ref: PackedReference):
        s = ref.as_struct()
        _check(self.lib, self.h, self.lib.ps_reference_upload(self.h, C.byref(s)))
        self.ref = ref

    def load_fasta(self, path: str):
        """FASTA + .fai -> packed reference resident in HBM (replaces IndexedFastaSequenceFile, ErrorProfiling.java:109)."""
        _check(self.lib, self.h, self.lib.ps_reference_load_fasta(self.h, path.encode()))
        self.ref = None

    def set_contig_order(self, order=None):
        """The contig order the records of the following pileup calls take: order[k] = FASTA index of the k-th contig
        (BamBatcher.contig_order gives a file's), contigs not listed after the listed ones in FASTA order; None or []:
        FASTA order, the state after every reference upload.  Records whose contig goes backwards against it raise
        PS_ERR_UNSORTED.  Carry tuples and pileup_max_key keep FASTA indices; the device keys follow the order."""
        a = np.ascontiguousarray(order if order is not None else [], dtype=np.uint32)
        _check(self.lib, self.h, self.lib.ps_reference_set_contig_order(self.h, a.ctypes.data if a.size else None, a.size))

    # ---- whole-tool loops from files ------------------------------------------------------------------
    def profile_bam(self, bam_path: str, max_read_length: int, infer_qualities: bool = False) -> dict:
        """The record loop of the `error` tool (ErrorProfiling.java:104-409) on a coordinate-sorted BAM."""
        self._max_len, self._infer_q = max_read_length, infer_qualities
        out, r = self._profile_result_arrays()
        o = abi.ps_profile_opts(max_read_length, int(infer_qualities), 0, 0)
        st = self.lib.ps_profile_bam(self.h, bam_path.encode(), C.byref(o), C.byref(r))
        _check(self.lib, self.h, st, fault=(r.fault.code, r.fault.read_ordinal))
        return out

    def pileup_bam(self, bam_path: str, first_running_id: int = 1) -> "PileupResult":
        """The record loop of the `clust` tool (PileupClusters.java:62-500) on a coordinate-sorted BAM."""
        opts = abi.ps_pileup_opts(first_running_id, 0, 0, 0, 0, None, None)
        h = C.c_void_p()
        st = self.lib.ps_pileup_bam(self.h, bam_path.encode(), C.byref(opts), C.byref(h))
        res = PileupResult(self, h, None)
        try:
            if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED) and h:
                f = abi.ps_fault()
                self.lib.ps_pileup_fault(h, C.byref(f))
                _check(self.lib, self.h, st, fault=(f.code, f.read_ordinal))
            _check(self.lib, self.h, st)
        except Exception:
            res.close()
            raise
        return res

    def clust_bam(self, bam_path: str, out_path: str, snp_vcf: Optional[str] = None, min_read_coverage: int = 1) -> dict:
        """The whole `clust` tool from files (PileupClusters.java:62-584): writes <out>, <out>.ccr.fasta, <out>.ccr.tsv,
        <out>.report, <bam>.sitefrequency.tsv and <bam>.sitepositions.tsv; returns the run's counters."""
        ctr, f = abi.ps_pileup_counters(), abi.ps_fault()
        st = self.lib.ps_clust_bam(self.h, bam_path.encode(), out_path.encode(), snp_vcf.encode() if snp_vcf else None,
                                   min_read_coverage, C.byref(ctr), C.byref(f))
        _check(self.lib, self.h, st, fault=(f.code, f.read_ordinal))
        return {k: getattr(ctr, k) for k, _ in abi.ps_pileup_counters._fields_}

    def error_bam(self, bam_path: str, max_read_length: int, infer_qualities: bool = False) -> np.ndarray:
        """The whole `error` tool from files (ErrorProfiling.inferErrorProfile): writes <bam>.errorprofile,
        .errorprofile.vcf, .qualityPerMismatch, .indels, .indelprofile, .qualities; returns the run counters."""
        o = abi.ps_profile_opts(max_read_length, int(infer_qualities), 0, 0)
        ctr = (C.c_int32 * abi.PS_PC_COUNT)()
        f = abi.ps_fault()
        st = self.lib.ps_error_bam(self.h, bam_path.encode(), C.byref(o), ctr, C.byref(f))
        _check(self.lib, self.h, st, fault=(f.code, f.read_ordinal))
        return np.array(list(ctr), dtype=np.int32)

    def track_bam(self, bam_path: str, out_prefix: str, *, base_counts: bool = False, min_coverage: int = 1,
                  min_events: int = 1, substitutions=None, indel_counts: bool = False, min_indel_depth: int = 1,
                  min_indel_events: int = 1, min_mapq: int = 0, require_flags: int = 0, exclude_flags: int = 0,
                  min_base_quality: int = 0) -> dict:
        """The `track` tool from files: writes <out_prefix>.plus.bedGraph, <out_prefix>.minus.bedGraph and
        <out_prefix>.t2c.tsv (per-position coverage and T>C events by strand); returns the run's counters.
        base_counts: also <out_prefix>.bases.tsv (keywords as Context.track), and the counters gain "base_totals"
        ((2, 4, 5) uint64: strand, reference base, read base A C G T N) and "n_base_rows".
        indel_counts: also <out_prefix>.indels.tsv (keywords as Context.track), and the counters gain "indel_totals".
        min_mapq, require_flags, exclude_flags, min_base_quality: the read and base filters of Context.track; with any
        of them set the counters gain "filter_counters"."""
        opts = track_opts(base_counts, min_coverage, min_events, substitutions)
        iopts = track_indel_opts(indel_counts, min_indel_depth, min_indel_events)
        fopts = track_filter_opts(min_mapq, require_flags, exclude_flags, min_base_quality)
        ctr, f, tot, itot = abi.ps_track_counters(), abi.ps_fault(), abi.ps_track_base_totals(), abi.ps_track_indel_totals()
        fctr = abi.ps_track_filter_counters()
        if fopts is None:
            st = self.lib.ps_track_bam_ex2(self.h, bam_path.encode(), out_prefix.encode(), C.byref(opts) if opts else None,
                                           C.byref(iopts) if iopts else None, C.byref(ctr), C.byref(tot), C.byref(itot),
                                           C.byref(f))
        else:
            st = self.lib.ps_track_bam_ex3(self.h, bam_path.encode(), out_prefix.encode(), C.byref(opts) if opts else None,
                                           C.byref(iopts) if iopts else None, C.byref(fopts), C.byref(ctr), C.byref(tot),
                                           C.byref(itot), C.byref(fctr), C.byref(f))
        _check(self.lib, self.h, st, fault=(f.code, f.read_ordinal))
        out = ctr.as_dict()
        if opts:
            out.update(_base_totals_dict(tot))
        if iopts:
            out["indel_totals"] = itot.as_dict()
        if fopts is not None:
            out["filter_counters"] = fctr.as_dict()
        return out

    # ---- batches ---------------------------------------------------------------------------------
    def upload(self, batch) -> UploadedBatch:
        """One H2D copy of a host batch (ReadBatch / PinnedBatch); both tools can then run on the device view
        (pass stream=0 so they are ordered after the copy on the context's stream)."""
        s = batch.struct if hasattr(batch, "struct") else batch.as_struct()
        v = abi.ps_read_batch()
        _check(self.lib, self.h, self.lib.ps_batch_upload(self.h, C.byref(s), C.byref(v)))
        return UploadedBatch(v, batch.n_reads, batch)

    # ---- error profile (ErrorProfiling.java:146-409) ---------------------------------------------
    def profile_begin(self, max_read_length: int, infer_qualities: bool = False, emit_t2c_masks: bool = False):
        """emit_t2c_masks: device-resident batches of the PAR-CLIP shape leave one T>C mask word per read in HBM
        (profile_masks()), which a pileup call on the same batch takes instead of decoding the reads again."""
        o = abi.ps_profile_opts(max_read_length, int(infer_qualities), int(emit_t2c_masks), 0)
        _check(self.lib, self.h, self.lib.ps_profile_begin(self.h, C.byref(o)))
        self._max_len = max_read_length
        self._infer_q = infer_qualities

    def profile_batch(self, batch):
        """Host-resident batch (ReadBatch or PinnedBatch): H2D inside the call."""
        s = batch.struct if hasattr(batch, "struct") else batch.as_struct()
        self._keep.append(batch)
        _check(self.lib, self.h, self.lib.ps_profile_batch(self.h, C.byref(s)))

    def profile_batch_device(self, dbatch, stream: int = 0):
        _check(self.lib, self.h, self.lib.ps_profile_batch_device(self.h, C.byref(dbatch.struct), stream or None))

    def profile_masks(self):
        """(device pointer, n) of the T>C mask words of the last profile_batch_device call, or None."""
        p, n = C.c_void_p(), C.c_uint64()
        _check(self.lib, self.h, self.lib.ps_profile_masks_device(self.h, C.byref(p), C.byref(n)))
        return (p.value, n.value) if p.value else None

    def profile_acc_tensor(self):
        """The int64 accumulator vector as a torch tensor aliasing library memory (for dist.all_reduce)."""
        import torch
        p = C.c_void_p()
        n = C.c_size_t()
        _check(self.lib, self.h, self.lib.ps_profile_acc_device(self.h, C.byref(p), C.byref(n)))

        class _Alias:
            __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<i8", "data": (p.value, False), "version": 3}

        return torch.as_tensor(_Alias(), device=f"cuda:{self.device}")

    def profile_set_stream(self, stream: int):
        """The accumulator vector is next touched on `stream` (an all-reduce queued there): profile_end reads it back
        there and waits for that stream only."""
        _check(self.lib, self.h, self.lib.ps_profile_set_stream(self.h, stream or None))

    def _profile_result_plan(self):
        """(name, dtype, shape, count, byte offset) of every result array inside one allocation, cached per run shape."""
        key = (self._max_len, bool(self._infer_q))
        plan = self._result_plans.get(key)
        if plan is None:
            m = self._max_len
            wide_n = self.lib.ps_profile_acc_len(m, int(self._infer_q))
            parts = [("position_conversions", np.int32, (m, 4, 4)), ("quality_per_mismatch", np.int32, (4, 4)),
                     ("quality_per_mismatch_counts", np.int32, (4, 4)), ("counters", np.int32, (abi.PS_PC_COUNT,)),
                     ("insertions_per_pos", np.float64, (m,)), ("deletions_per_pos", np.float64, (m,)),
                     ("wide", np.int64, (wide_n,))]
            if self._infer_q:
                parts.append(("quality_hist", np.int64, (m, 256)))
            items, total = [], 0
            for name, dt, shape in parts:
                n = 1
                for d in shape:
                    n *= int(d)
                total = (total + 7) & ~7
                items.append((name, np.dtype(dt), shape, n, total))
                total += n * np.dtype(dt).itemsize
            plan = (items, total)
            self._result_plans[key] = plan
        return plan

    def _profile_result_arrays(self):
        """Fresh result arrays for one run, carved out of ONE allocation (per-array numpy / ctypes bookkeeping costs more
        than the copy itself on the small PAR-CLIP profile, and the device sits idle while the host does it)."""
        items, total = self._profile_result_plan()
        buf = np.zeros(total, dtype=np.uint8)
        base = buf.ctypes.data
        out, r = {}, abi.ps_profile_result()
        for name, dt, shape, n, off in items:
            out[name] = np.frombuffer(buf, dtype=dt, count=n, offset=off).reshape(shape)
            setattr(r, name, base + off)
        if not self._infer_q:
            r.quality_hist = None
        return out, r

    def profile_end(self) -> dict:
        out, r = self._profile_result_arrays()
        st = self.lib.ps_profile_end(self.h, C.byref(r))
        self._keep.clear()
        _check(self.lib, self.h, st, fault=(r.fault.code, r.fault.read_ordinal))
        return out

    def profile(self, batch: ReadBatch, max_read_length: int, infer_qualities: bool = False) -> dict:
        self.profile_begin(max_read_length, infer_qualities)
        self.profile_batch(batch)
        return self.profile_end()

    # ---- T>C pileup (PileupClusters.java:137-500, 585-673) ----------------------------------------
    def pileup_run(self, batch, first_running_id: int = 1, carry=None, stream: int = 0, carry_keys=None,
                   defer: bool = False, masks=None) -> "PileupResult":
        """Run the pileup kernels; the cluster and site records stay in HBM behind the returned handle.
        defer=True (device-resident batches): return right behind the kernel launches (ps_pileup_submit_device); the
        call is completed by PileupResult.wait(), which the first look at the counters / records does by itself.
        batch: ReadBatch / PinnedBatch (host buffers, H2D inside) or DeviceBatch / UploadedBatch (resident).
        carry = (contig_index, cluster_end) of the cluster left open by the preceding shard, or None;
        carry_keys = (device pointer, n): the keys of the n preceding shards left on the device (pileup_max_key_tensor +
        all-gather), an alternative to `carry` without a host round trip."""
        opts = abi.ps_pileup_opts(first_running_id, 0, 0, 0, 0, None, None)
        if masks is not None:          # profile_masks() of the SAME batch (same stream, or ordered behind it)
            if int(masks[1]) != batch.n_reads:
                raise ValueError("mask words belong to another batch")
            opts.t2c_masks_device = int(masks[0])
        if carry is not None:
            opts.carry_valid, opts.carry_contig, opts.carry_cluster_end = 1, int(carry[0]), int(carry[1])
        if carry_keys is not None and carry_keys[1] > 0:
            opts.carry_keys_device, opts.carry_keys_n = int(carry_keys[0]), int(carry_keys[1])
        h = C.c_void_p()
        if defer:
            if not isinstance(batch, (DeviceBatch, UploadedBatch)):
                raise TypeError("defer=True needs a device-resident batch")
            self._keep_opts = opts                     # the library copies it; kept for symmetry with the batch
            st = self.lib.ps_pileup_submit_device(self.h, C.byref(batch.struct), C.byref(opts), stream or None,
                                                  C.byref(h))
            _check(self.lib, self.h, st)
            return PileupResult(self, h, batch, pending=True)
        if isinstance(batch, (DeviceBatch, UploadedBatch)):
            st = self.lib.ps_pileup_batch_device(self.h, C.byref(batch.struct), C.byref(opts), stream or None,
                                                 C.byref(h))
        else:
            s = batch.struct if hasattr(batch, "struct") else batch.as_struct()
            st = self.lib.ps_pileup_batch(self.h, C.byref(s), C.byref(opts), C.byref(h))
        res = PileupResult(self, h, batch)
        try:
            if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED) and h:
                f = abi.ps_fault()
                self.lib.ps_pileup_fault(h, C.byref(f))
                _check(self.lib, self.h, st, fault=(f.code, f.read_ordinal))
            _check(self.lib, self.h, st)
        except Exception:
            res.close()
            raise
        return res

    def pileup_max_key(self, dbatch, stream: int = 0):
        """(contig, end) maximum over the kept records of a device-resident batch, or None (region sharding carry).  Contigs
        compare by their position in the context's contig order (set_contig_order); the contig returned is a FASTA index."""
        v, c, e = C.c_uint32(), C.c_uint32(), C.c_int32()
        _check(self.lib, self.h, self.lib.ps_pileup_max_key(self.h, C.byref(dbatch.struct), stream or None, C.byref(v),
                                                             C.byref(c), C.byref(e)))
        return (int(c.value), int(e.value)) if v.value else None

    def pileup_max_key_tensor(self, dbatch, stream: int = 0):
        """The same maximum as a 1-element int64 CUDA tensor aliasing library memory, computed asynchronously on `stream`:
        (position of the contig in the context's contig order + 1) << 32 | end, 0 = none -- the position is the FASTA index
        unless set_contig_order changed the order, and keys of two contexts compare only under the same order.  Feed it
        to an all-gather and hand the gathered keys to pileup_run(carry_keys=)."""
        import torch
        p = C.c_void_p()
        _check(self.lib, self.h, self.lib.ps_pileup_max_key_device(self.h, C.byref(dbatch.struct), stream or None, C.byref(p)))

        class _Alias:
            __cuda_array_interface__ = {"shape": (1,), "typestr": "<i8", "data": (p.value, False), "version": 3}

        return torch.as_tensor(_Alias(), device=f"cuda:{self.device}")

    def pileup(self, batch, first_running_id: int = 1, carry=None, stream: int = 0) -> dict:
        """pileup_run + fetch of every record into host arrays."""
        with self.pileup_run(batch, first_running_id, carry, stream) as res:
            return res.fetch()

    # ---- T>C conversion and coverage track ---------------------------------------------------------
    def track(self, batch, stream: int = 0, *, base_counts: bool = False, min_coverage: int = 1, min_events: int = 1,
              substitutions=None, indel_counts: bool = False, min_indel_depth: int = 1, min_indel_events: int = 1,
              min_mapq: int = 0, require_flags: int = 0, exclude_flags: int = 0, min_base_quality: int = 0) -> dict:
        """Per-position coverage and T>C events by strand of one whole input: {"runs_plus", "runs_minus", "sites",
        "counters"}, runs and sites as numpy structured arrays (abi.TRACK_RUN_DTYPE / TRACK_SITE_DTYPE, contigs as FASTA
        indices).  batch: host (ReadBatch / PinnedBatch) or device-resident (DeviceBatch / UploadedBatch).
        base_counts: also "base_rows" (abi.TRACK_BASE_ROW_DTYPE: read bases A C G T N by position and strand, strand
        orientation) for the positions with coverage >= min_coverage and >= min_events of the selected substitutions
        (an iterable of "X>Y"; None: all twelve), and "base_totals" ((2, 4, 5) uint64: strand, reference base, read
        base) over every counted base.
        indel_counts: also "indel_rows" (abi.TRACK_INDEL_ROW_DTYPE: deletions over and insertions anchored at each
        position by strand) for the positions with deletions + insertions >= min_indel_events and coverage + deletions
        >= min_indel_depth, and "indel_totals" (abi.ps_track_indel_totals as a dict of [plus, minus] lists and
        "n_rows").
        Read and base filters (all off at 0; samtools view -q / -f / -F, mpileup -Q): records with MAPQ < min_mapq, or
        whose FLAG lacks a bit of require_flags or has one of exclude_flags, are left out; aligned bases with quality
        < min_base_quality count nowhere but in "filter_counters" ("filtered_flags", "filtered_mapq",
        "low_quality_bases" [plus, minus]), which the result gains when any filter is set.  The record filter reads
        the batch's FLAG and MAPQ arrays (ReadBatch.sam_flags / mapq: from_records fills them, DeviceBatch uploads
        them; PinnedBatch and UploadedBatch take them from the host batch they came from)."""
        opts = track_opts(base_counts, min_coverage, min_events, substitutions)
        iopts = track_indel_opts(indel_counts, min_indel_depth, min_indel_events)
        fopts = track_filter_opts(min_mapq, require_flags, exclude_flags, min_base_quality)
        po, pi = C.byref(opts) if opts else None, C.byref(iopts) if iopts else None
        h = C.c_void_p()
        if fopts is None:
            if isinstance(batch, (DeviceBatch, UploadedBatch)):
                st = self.lib.ps_track_batch_device_ex2(self.h, C.byref(batch.struct), po, pi, stream or None, C.byref(h))
            else:
                s = batch.struct if hasattr(batch, "struct") else batch.as_struct()
                st = self.lib.ps_track_batch_ex2(self.h, C.byref(s), po, pi, C.byref(h))
        elif isinstance(batch, DeviceBatch):
            st = self.lib.ps_track_batch_device_ex3(self.h, C.byref(batch.struct), po, pi, C.byref(batch.aux),
                                                    C.byref(fopts), stream or None, C.byref(h))
        elif isinstance(batch, UploadedBatch):
            # the upload holds no aux arrays: device copies of the host batch's, kept alive for the call
            import torch
            src = getattr(batch._source, "host", batch._source)
            keep = [None if getattr(src, f, None) is None else
                    torch.from_numpy(np.ascontiguousarray(getattr(src, f)).view(np.uint8)).to(f"cuda:{self.device}")
                    for f in ("sam_flags", "mapq")]
            aux = abi.ps_read_aux(*(None if t is None else t.data_ptr() for t in keep))
            torch.cuda.synchronize(self.device)
            st = self.lib.ps_track_batch_device_ex3(self.h, C.byref(batch.struct), po, pi, C.byref(aux), C.byref(fopts),
                                                    stream or None, C.byref(h))
        else:
            s = batch.struct if hasattr(batch, "struct") else batch.as_struct()
            host = getattr(batch, "host", batch)
            aux = host.aux_struct() if hasattr(host, "aux_struct") else abi.ps_read_aux()
            st = self.lib.ps_track_batch_ex3(self.h, C.byref(s), po, pi, C.byref(aux), C.byref(fopts), C.byref(h))
        try:
            if st != abi.PS_OK:
                fault = None
                if h:
                    f = abi.ps_fault()
                    self.lib.ps_track_fault(h, C.byref(f))
                    fault = (f.code, f.read_ordinal)
                msg = self.lib.ps_last_error(self.h).decode()
                if st == abi.PS_ERR_REFERENCE_WOULD_THROW:
                    raise abi.ReferenceWouldThrow(st, msg, fault)
                raise abi.PsError(st, msg, fault)
            ctr = abi.ps_track_counters()
            self.lib.ps_track_counters_get(h, C.byref(ctr))
            out = {"counters": ctr.as_dict()}
            for s_, name in ((0, "runs_plus"), (1, "runs_minus")):
                a = np.zeros(ctr.n_runs[s_], dtype=abi.TRACK_RUN_DTYPE)
                if a.size:
                    self.lib.ps_track_runs(h, s_, 0, a.ctypes.data, a.size)
                out[name] = a
            sites = np.zeros(ctr.n_sites, dtype=abi.TRACK_SITE_DTYPE)
            if sites.size:
                self.lib.ps_track_sites(h, 0, sites.ctypes.data, sites.size)
            out["sites"] = sites
            if opts:
                tot = abi.ps_track_base_totals()
                _check(self.lib, self.h, self.lib.ps_track_base_totals_get(h, C.byref(tot)))
                rows = np.zeros(tot.n_rows, dtype=abi.TRACK_BASE_ROW_DTYPE)
                if rows.size:
                    self.lib.ps_track_base_rows(h, 0, rows.ctypes.data, rows.size)
                out["base_rows"] = rows
                out["base_totals"] = _base_totals_dict(tot)["base_totals"]
            if iopts:
                itot = abi.ps_track_indel_totals()
                _check(self.lib, self.h, self.lib.ps_track_indel_totals_get(h, C.byref(itot)))
                rows = np.zeros(itot.n_rows, dtype=abi.TRACK_INDEL_ROW_DTYPE)
                if rows.size:
                    self.lib.ps_track_indel_rows(h, 0, rows.ctypes.data, rows.size)
                out["indel_rows"] = rows
                out["indel_totals"] = itot.as_dict()
            if fopts is not None:
                fctr = abi.ps_track_filter_counters()
                _check(self.lib, self.h, self.lib.ps_track_filter_counters_get(h, C.byref(fctr)))
                out["filter_counters"] = fctr.as_dict()
            return out
        finally:
            if h:
                self.lib.ps_track_close(h)

    def _pinned(self, key: str, nbytes: int) -> np.ndarray:
        """Reusable page-locked host buffer (grown on demand) viewed as uint8."""
        import torch
        t = self._pinned_bufs.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes + nbytes // 8, 4096), dtype=torch.uint8).pin_memory()
            self._pinned_bufs[key] = t
        return t.numpy()[:nbytes]

    # ---- instrumentation -------------------------------------------------------------------------
    def kernel_launches(self) -> int:
        return int(self.lib.ps_kernel_launches(self.h))

    def kernel_times_reset(self, enabled: bool = True):
        self.lib.ps_kernel_times_reset(self.h, int(enabled))

    def pileup_stage_ms(self) -> np.ndarray:
        """Device times of the last pileup call's kernels: flag scan, cluster kernel, site compaction."""
        buf = np.zeros(3, dtype=np.float32)
        st = self.lib.ps_pileup_stage_times(self.h, buf.ctypes.data)
        return buf if st == abi.PS_OK else np.full(3, np.nan, dtype=np.float32)

    def kernel_times_ms(self) -> np.ndarray:
        buf = np.zeros(512, dtype=np.float32)
        n = self.lib.ps_kernel_times(self.h, buf.ctypes.data, buf.size)
        return buf[:max(n, 0)].copy()


class PileupResult:
    """Handle of one pileup call: counters on the host, cluster / site records resident in HBM until fetched."""

    def __init__(self, ctx: Context, h, batch, pending: bool = False):
        self.ctx = ctx
        self.h = h
        self._batch = batch            # the records must outlive the halo-merge coverage query
        self._counters = None
        self._pending = pending        # submitted, not waited for (Context.pileup_run(defer=True))

    def wait(self):
        """Complete a deferred call (no-op otherwise); raises what the synchronous call would have raised."""
        if not self._pending:
            return self
        self._pending = False
        st = self.ctx.lib.ps_pileup_wait(self.h)
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED):
            f = abi.ps_fault()
            self.ctx.lib.ps_pileup_fault(self.h, C.byref(f))
            _check(self.ctx.lib, self.ctx.h, st, fault=(f.code, f.read_ordinal))
        _check(self.ctx.lib, self.ctx.h, st)
        return self

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def close(self):
        if self.h:
            self.ctx.lib.ps_pileup_close(self.h)
            self.h = None

    @property
    def counters(self) -> dict:
        if self._counters is None:
            self.wait()
            ctr = abi.ps_pileup_counters()
            self.ctx.lib.ps_pileup_counters_get(self.h, C.byref(ctr))
            self._counters = {f: getattr(ctr, f) for f, _ in abi.ps_pileup_counters._fields_}
        return self._counters

    def fetch(self, pinned: bool = False, boundary: bool = True) -> dict:
        """Copy the records to the host.  pinned=True: into page-locked buffers owned by the context and REUSED by the
        next pinned fetch (what a streaming caller does); otherwise into fresh arrays."""
        lib, ctx = self.ctx.lib, self.ctx
        c = self.counters
        nc, ns = c["n_clusters"], c["n_sites"]
        csz, ssz = np.dtype(abi.CLUSTER_DTYPE).itemsize, np.dtype(abi.SITE_DTYPE).itemsize
        if pinned:
            clusters = ctx._pinned("clusters", nc * csz).view(abi.CLUSTER_DTYPE)
            sites = ctx._pinned("sites", ns * ssz).view(abi.SITE_DTYPE)
        else:
            clusters = np.zeros(nc, dtype=abi.CLUSTER_DTYPE)
            sites = np.zeros(ns, dtype=abi.SITE_DTYPE)
        got = lib.ps_pileup_next(self.h, 0, clusters.ctypes.data, nc, sites.ctypes.data, ns)
        if got != nc:
            raise abi.PsError(int(got), "ps_pileup_next returned fewer clusters than announced")
        out = {"clusters": clusters, "sites": sites, "counters": dict(c)}
        if not boundary:
            return out
        open_c = np.zeros(1, dtype=abi.CLUSTER_DTYPE)
        open_s = np.zeros(1 << 16, dtype=abi.SITE_DTYPE)
        k = lib.ps_pileup_open_cluster(self.h, open_c.ctypes.data, open_s.ctypes.data, open_s.size)
        if k < 0:
            raise abi.PsError(k, "open cluster has too many sites")
        head_c = np.zeros(1, dtype=abi.CLUSTER_DTYPE)
        head_s = np.zeros(1 << 16, dtype=abi.SITE_DTYPE)
        kh = lib.ps_pileup_head_partial(self.h, head_c.ctypes.data, head_s.ctypes.data, head_s.size)
        if kh < 0:
            raise abi.PsError(kh, "head partial has too many sites")
        for which, name in ((0, "head_cov"), (1, "open_cov")):
            p0 = C.c_int32()
            ln = lib.ps_pileup_boundary_coverage(self.h, which, C.byref(p0), None, 0)
            if ln < 0:
                raise abi.PsError(int(ln), lib.ps_last_error(ctx.h).decode())
            a = np.zeros(max(int(ln), 0), dtype=np.uint32)
            if ln > 0:
                lib.ps_pileup_boundary_coverage(self.h, which, C.byref(p0), a.ctypes.data, a.size)
            out[name] = (int(p0.value), a)
        out.update({
            "open_cluster": open_c[0] if k > 0 else None,
            "open_sites": open_s[:int(open_c[0]["site_end"])].copy() if k > 0 else open_s[:0],
            "head_partial": head_c[0] if kh > 0 else None,
            "head_sites": head_s[:int(head_c[0]["site_end"])].copy() if kh > 0 else head_s[:0],
        })
        return out


class MultiContext:
    """Several GPUs behind one handle in ONE process (what a JVM uses: ps_create_multi): the file loops of both tools,
    batches / windows round-robin over the devices, results merged on the host."""

    def __init__(self, devices=None):
        self.lib = abi.load_library()
        h = C.c_void_p()
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            st = self.lib.ps_create_multi(C.byref(h), arr, len(devices))
        else:
            st = self.lib.ps_create_multi(C.byref(h), None, 0)          # PARASUITE_B200_DEVICES or device 0
        if st != abi.PS_OK:
            raise abi.PsError(st, self.lib.ps_strerror(st).decode())
        self.h = h

    def _check(self, st, fault=None):
        if st == abi.PS_OK:
            return
        msg = self.lib.ps_multi_last_error(self.h).decode() or self.lib.ps_strerror(st).decode()
        if st == abi.PS_ERR_REFERENCE_WOULD_THROW:
            raise abi.ReferenceWouldThrow(st, msg, fault)
        raise abi.PsError(st, msg, fault)

    @property
    def n_devices(self) -> int:
        return int(self.lib.ps_multi_device_count(self.h))

    def load_fasta(self, path: str):
        self._check(self.lib.ps_multi_load_fasta(self.h, path.encode()))

    def profile_bam(self, bam_path: str, max_read_length: int, infer_qualities: bool = False) -> dict:
        tmp = Context.__new__(Context)
        tmp.lib, tmp._max_len, tmp._infer_q, tmp._result_plans = self.lib, max_read_length, infer_qualities, {}
        out, r = Context._profile_result_arrays(tmp)
        o = abi.ps_profile_opts(max_read_length, int(infer_qualities), 0, 0)
        st = self.lib.ps_multi_profile_bam(self.h, bam_path.encode(), C.byref(o), C.byref(r))
        self._check(st, fault=(r.fault.code, r.fault.read_ordinal))
        return out

    def pileup_bam(self, bam_path: str, first_running_id: int = 1) -> "PileupResult":
        opts = abi.ps_pileup_opts(first_running_id, 0, 0, 0, 0, None, None)
        h = C.c_void_p()
        st = self.lib.ps_multi_pileup_bam(self.h, bam_path.encode(), C.byref(opts), C.byref(h))
        fault = None
        if st in (abi.PS_ERR_REFERENCE_WOULD_THROW, abi.PS_ERR_UNSUPPORTED) and h:
            f = abi.ps_fault()
            self.lib.ps_pileup_fault(h, C.byref(f))
            fault = (f.code, f.read_ordinal)
            self.lib.ps_pileup_close(h)
        self._check(st, fault=fault)
        holder = Context.__new__(Context)
        holder.lib, holder.h = self.lib, self.lib.ps_multi_context(self.h, 0)
        holder._pinned_bufs = {}
        holder.close = lambda: None
        return PileupResult(holder, h, None)

    def clust_bam(self, bam_path: str, out_path: str, snp_vcf: Optional[str] = None, min_read_coverage: int = 1) -> dict:
        ctr, f = abi.ps_pileup_counters(), abi.ps_fault()
        st = self.lib.ps_multi_clust_bam(self.h, bam_path.encode(), out_path.encode(), snp_vcf.encode() if snp_vcf else None,
                                         min_read_coverage, C.byref(ctr), C.byref(f))
        self._check(st, fault=(f.code, f.read_ordinal))
        return {k: getattr(ctr, k) for k, _ in abi.ps_pileup_counters._fields_}

    def track_bam(self, bam_path: str, out_prefix: str, *, base_counts: bool = False, min_coverage: int = 1,
                  min_events: int = 1, substitutions=None, indel_counts: bool = False, min_indel_depth: int = 1,
                  min_indel_events: int = 1, min_mapq: int = 0, require_flags: int = 0, exclude_flags: int = 0,
                  min_base_quality: int = 0) -> dict:
        """Context.track_bam with windows round-robin over the devices; the files are byte-identical."""
        opts = track_opts(base_counts, min_coverage, min_events, substitutions)
        iopts = track_indel_opts(indel_counts, min_indel_depth, min_indel_events)
        fopts = track_filter_opts(min_mapq, require_flags, exclude_flags, min_base_quality)
        ctr, f, tot, itot = abi.ps_track_counters(), abi.ps_fault(), abi.ps_track_base_totals(), abi.ps_track_indel_totals()
        fctr = abi.ps_track_filter_counters()
        if fopts is None:
            st = self.lib.ps_multi_track_bam_ex2(self.h, bam_path.encode(), out_prefix.encode(),
                                                 C.byref(opts) if opts else None, C.byref(iopts) if iopts else None,
                                                 C.byref(ctr), C.byref(tot), C.byref(itot), C.byref(f))
        else:
            st = self.lib.ps_multi_track_bam_ex3(self.h, bam_path.encode(), out_prefix.encode(),
                                                 C.byref(opts) if opts else None, C.byref(iopts) if iopts else None,
                                                 C.byref(fopts), C.byref(ctr), C.byref(tot), C.byref(itot),
                                                 C.byref(fctr), C.byref(f))
        self._check(st, fault=(f.code, f.read_ordinal))
        out = ctr.as_dict()
        if opts:
            out.update(_base_totals_dict(tot))
        if iopts:
            out["indel_totals"] = itot.as_dict()
        if fopts is not None:
            out["filter_counters"] = fctr.as_dict()
        return out

    def close(self):
        if getattr(self, "h", None):
            self.lib.ps_destroy_multi(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
