"""ctypes mirror of include/parasuite_b200.h (struct layouts, constants, library loader).

No compute happens here; this is the binding a Python caller uses where the Java toolkit would use
the JNI shim (INTEGRATION.md).  The CUDA library is mandatory: there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT_DIR = os.path.dirname(PKG_DIR)                 # para-suite_b200/
LIB_DIR = os.path.join(ROOT_DIR, "lib")
CSRC_DIR = os.path.join(ROOT_DIR, "csrc")
REPO_DIR = os.path.dirname(ROOT_DIR)
INCLUDE_DIR = os.path.join(REPO_DIR, "include")

PS_ABI_VERSION = 5
PS_OK = 0
PS_ERR_INVALID_ARG = -1
PS_ERR_NO_DEVICE = -2
PS_ERR_CUDA = -3
PS_ERR_OOM = -4
PS_ERR_IO = -5
PS_ERR_FORMAT = -6
PS_ERR_UNSORTED = -7
PS_ERR_REFERENCE_WOULD_THROW = -8
PS_ERR_STATE = -9
PS_ERR_UNSUPPORTED = -10

PS_THROW_NONE = 0
PS_THROW_REF_RANGE = 1
PS_THROW_EMPTY_REF = 2
PS_THROW_INDEL_FILL = 3
PS_THROW_INDEL_POS = 4
PS_THROW_POS_MAXLEN = 5
PS_THROW_QUAL_RANGE = 6
PS_THROW_MASK51 = 7
PS_THROW_BLOCK_RANGE = 8
PS_FAULT_CIGAR_OPS = 9
PS_FAULT_PAST_END = 10

PS_TILE_READS = 256
PS_RF_UNMAPPED = 0x01
PS_RF_REVERSE = 0x02
PS_RF_DUPLICATE = 0x04
PS_RF_POS_ZERO = 0x08
PS_RF_QUAL_MISSING = 0x10
PS_RF_HAS_INVALID = 0x20
PS_RF_REF_RANGE = 0x40
PS_RF_CIGAR_OVERFLOW = 0x80

PS_BAM_ANY_CONTIG_ORDER = 0x1

PS_PC_NAMES = ["num_reads_processed", "unmapped", "duplicates", "start_zero", "indel_read", "skipped_reads",
               "longer_indels", "total_bases_checked"]
PS_PC_COUNT = len(PS_PC_NAMES)

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)


class ps_reference(C.Structure):
    _fields_ = [("n_bases", C.c_uint64), ("seq2", C.c_void_p), ("inv", C.c_void_p), ("n_contigs", C.c_uint32),
                ("contig_off", C.c_void_p)]


class ps_read_batch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("meta", C.c_void_p), ("ref_start", C.c_void_p), ("bases2", C.c_void_p),
                ("qual", C.c_void_p), ("cigar", C.c_void_p), ("tile_base_off", C.c_void_p),
                ("tile_qual_off", C.c_void_p), ("tile_cigar_off", C.c_void_p), ("tile_exc_off", C.c_void_p),
                ("exc", C.c_void_p), ("uniform_len", C.c_uint32), ("uniform_ncigar", C.c_uint32),
                ("bases_bytes", C.c_uint64), ("qual_bytes", C.c_uint64), ("cigar_count", C.c_uint64),
                ("exc_count", C.c_uint64), ("max_len", C.c_uint32), ("uniform_cigar", C.c_uint32), ("flags8", C.c_void_p), ("qual6", C.c_void_p), ("start16", C.c_void_p),
                ("tile_start", C.c_void_p), ("past_end", C.c_uint64)]


class ps_comb_stats(C.Structure):
    _fields_ = [("genomic_records", C.c_uint64), ("transcript_records", C.c_uint64), ("lifted_records", C.c_uint64),
                ("mapped_reads", C.c_uint64), ("spliced_reads", C.c_uint64), ("missed_transcript_alignments", C.c_uint64)]


class ps_profile_opts(C.Structure):
    _fields_ = [("max_read_length", C.c_uint32), ("infer_qualities", C.c_uint32), ("emit_t2c_masks", C.c_uint32),
                ("reserved", C.c_uint32)]


class ps_fault(C.Structure):
    _fields_ = [("code", C.c_int32), ("read_ordinal", C.c_uint64)]


class ps_profile_result(C.Structure):
    _fields_ = [("position_conversions", C.c_void_p), ("quality_per_mismatch", C.c_void_p),
                ("quality_per_mismatch_counts", C.c_void_p), ("insertions_per_pos", C.c_void_p),
                ("deletions_per_pos", C.c_void_p), ("counters", C.c_void_p), ("quality_hist", C.c_void_p),
                ("wide", C.c_void_p), ("fault", ps_fault)]


class ps_cluster(C.Structure):
    _fields_ = [("first_read", C.c_uint64), ("running_id", C.c_uint32), ("contig", C.c_uint32),
                ("start", C.c_int32), ("end", C.c_int32), ("num_reads", C.c_uint32), ("num_t2c", C.c_uint32),
                ("minus_after_first", C.c_uint32), ("first_reverse", C.c_uint8), ("combined_strand", C.c_uint8),
                ("reserved", C.c_uint16), ("mask51", C.c_uint64), ("site_begin", C.c_uint64),
                ("site_end", C.c_uint64)]


class ps_site(C.Structure):
    _fields_ = [("pos", C.c_int32), ("t2c", C.c_uint32), ("cov", C.c_uint32), ("reserved", C.c_uint32),
                ("order_key", C.c_uint64)]


class ps_pileup_counters(C.Structure):
    _fields_ = [("num_reads_processed", C.c_uint64), ("skipped_due_indel", C.c_uint64),
                ("double_stranded", C.c_uint64), ("n_clusters", C.c_uint64), ("n_sites", C.c_uint64),
                ("has_open_cluster", C.c_uint8)]


class ps_pileup_opts(C.Structure):
    _fields_ = [("first_running_id", C.c_uint32), ("carry_valid", C.c_uint32), ("carry_contig", C.c_uint32),
                ("carry_cluster_end", C.c_int32), ("carry_keys_n", C.c_uint32), ("carry_keys_device", C.c_void_p),
                ("t2c_masks_device", C.c_void_p)]


class ps_track_counters(C.Structure):
    _fields_ = [("num_reads_processed", C.c_uint64), ("unmapped", C.c_uint64), ("skipped_due_indel", C.c_uint64),
                ("reads_counted", C.c_uint64), ("aligned_bases", C.c_uint64 * 2), ("t2c_events", C.c_uint64 * 2),
                ("n_runs", C.c_uint64 * 2), ("n_sites", C.c_uint64), ("fast_path_reads", C.c_uint64)]

    def as_dict(self) -> dict:
        return {f: (list(getattr(self, f)) if hasattr(getattr(self, f), "__len__") else int(getattr(self, f)))
                for f, _ in self._fields_}


class ps_flush_totals(C.Structure):
    _fields_ = [("snp_hit", C.c_uint64), ("high_frequent_error", C.c_uint64), ("num_crosslinked_clusters", C.c_uint64),
                ("num_allele_positions", C.c_uint64), ("allele_positions", C.c_uint64 * 51),
                ("n_allele_frequency", C.c_uint64)]


FLUSH_ROW_DTYPE = [("emitted", "u1"), ("has_ccr", "u1"), ("reserved", "<u2"), ("num_t2c_sites", "<u4"),
                   ("best_pos", "<i4"), ("best_count", "<u4"), ("best_value", "<f8"), ("fraction", "<f8")]

# numpy dtypes with the same layout as ps_cluster / ps_site (checked in tests against ctypes.sizeof)
CLUSTER_DTYPE = [("first_read", "<u8"), ("running_id", "<u4"), ("contig", "<u4"), ("start", "<i4"), ("end", "<i4"),
                 ("num_reads", "<u4"), ("num_t2c", "<u4"), ("minus_after_first", "<u4"), ("first_reverse", "u1"),
                 ("combined_strand", "u1"), ("reserved", "<u2"), ("mask51", "<u8"), ("site_begin", "<u8"),
                 ("site_end", "<u8")]
SITE_DTYPE = [("pos", "<i4"), ("t2c", "<u4"), ("cov", "<u4"), ("reserved", "<u4"), ("order_key", "<u8")]
# ps_track_run / ps_track_site
TRACK_RUN_DTYPE = [("contig", "<u4"), ("start0", "<u4"), ("end0", "<u4"), ("cov", "<u4")]
TRACK_SITE_DTYPE = [("contig", "<u4"), ("pos", "<i4"), ("strand", "<u4"), ("t2c", "<u4"), ("cov", "<u4")]

# every symbol include/parasuite_b200.h declares: name -> (restype, argtypes)
VP = C.c_void_p
EXPORTS = {
    "ps_abi_version": (C.c_int, []),
    "ps_create": (C.c_int, [C.POINTER(VP), C.c_int]),
    "ps_destroy": (None, [VP]),
    "ps_last_error": (C.c_char_p, [VP]),
    "ps_strerror": (C.c_char_p, [C.c_int]),
    "ps_reference_upload": (C.c_int, [VP, C.POINTER(ps_reference)]),
    "ps_reference_load_fasta": (C.c_int, [VP, C.c_char_p]),
    "ps_reference_adopt_device": (C.c_int, [VP, C.POINTER(ps_reference), VP]),
    "ps_reference_set_contig_order": (C.c_int, [VP, VP, C.c_uint32]),
    "ps_batch_upload": (C.c_int, [VP, C.POINTER(ps_read_batch), C.POINTER(ps_read_batch)]),
    "ps_profile_acc_len": (C.c_size_t, [C.c_uint32, C.c_uint32]),
    "ps_clust_bam": (C.c_int, [VP, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.POINTER(ps_pileup_counters),
                               C.POINTER(ps_fault)]),
    "ps_profile_write_files": (C.c_int, [C.POINTER(ps_profile_result), C.c_uint32, C.c_uint32, C.c_char_p, C.POINTER(C.c_double),
                                         C.c_char_p, C.c_size_t]),
    "ps_liftover_hit": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.POINTER(C.c_int32), C.c_char_p,
                                  C.c_size_t, C.POINTER(C.c_uint32)]),
    "ps_comb_bam": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(ps_comb_stats), C.c_char_p, C.c_size_t]),
    "ps_error_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_profile_opts), C.POINTER(C.c_int32), C.POINTER(ps_fault)]),
    "ps_multi_error_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_profile_opts), C.POINTER(C.c_int32), C.POINTER(ps_fault)]),
    "ps_create_multi": (C.c_int, [C.POINTER(VP), C.POINTER(C.c_int), C.c_int]),
    "ps_destroy_multi": (None, [VP]),
    "ps_multi_device_count": (C.c_int, [VP]),
    "ps_multi_context": (VP, [VP, C.c_int]),
    "ps_multi_last_error": (C.c_char_p, [VP]),
    "ps_multi_load_fasta": (C.c_int, [VP, C.c_char_p]),
    "ps_multi_profile_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_profile_opts), C.POINTER(ps_profile_result)]),
    "ps_multi_pileup_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_pileup_opts), C.POINTER(VP)]),
    "ps_multi_clust_bam": (C.c_int, [VP, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.POINTER(ps_pileup_counters),
                                     C.POINTER(ps_fault)]),
    "ps_clust_writer_open": (C.c_int, [C.POINTER(VP), VP, C.c_char_p, C.c_char_p, C.c_char_p]),
    "ps_clust_writer_feed": (C.c_int, [VP, C.POINTER(ps_read_batch), C.c_uint64, VP, C.c_uint64, VP, C.c_int, C.c_uint64]),
    "ps_clust_writer_finish": (C.c_int, [VP, C.POINTER(ps_pileup_counters)]),
    "ps_clust_writer_fault": (C.c_int, [VP, C.POINTER(ps_fault)]),
    "ps_clust_writer_stats": (None, [VP, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ps_clust_writer_error": (C.c_char_p, [VP]),
    "ps_clust_writer_close": (None, [VP]),
    "ps_profile_begin": (C.c_int, [VP, C.POINTER(ps_profile_opts)]),
    "ps_profile_masks_device": (C.c_int, [VP, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "ps_profile_batch": (C.c_int, [VP, C.POINTER(ps_read_batch)]),
    "ps_profile_batch_device": (C.c_int, [VP, C.POINTER(ps_read_batch), VP]),
    "ps_profile_acc_device": (C.c_int, [VP, C.POINTER(VP), C.POINTER(C.c_size_t)]),
    "ps_profile_set_stream": (C.c_int, [VP, VP]),
    "ps_profile_end": (C.c_int, [VP, C.POINTER(ps_profile_result)]),
    "ps_profile_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_profile_opts), C.POINTER(ps_profile_result)]),
    "ps_pileup_batch": (C.c_int, [VP, C.POINTER(ps_read_batch), C.POINTER(ps_pileup_opts), C.POINTER(VP)]),
    "ps_pileup_batch_device": (C.c_int, [VP, C.POINTER(ps_read_batch), C.POINTER(ps_pileup_opts), VP,
                                         C.POINTER(VP)]),
    "ps_pileup_submit_device": (C.c_int, [VP, C.POINTER(ps_read_batch), C.POINTER(ps_pileup_opts), VP,
                                          C.POINTER(VP)]),
    "ps_pileup_wait": (C.c_int, [VP]),
    "ps_pileup_max_key": (C.c_int, [VP, C.POINTER(ps_read_batch), VP, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                C.POINTER(C.c_int32)]),
    "ps_pileup_max_key_device": (C.c_int, [VP, C.POINTER(ps_read_batch), VP, C.POINTER(VP)]),
    "ps_pileup_counters_get": (C.c_int, [VP, C.POINTER(ps_pileup_counters)]),
    "ps_pileup_next": (C.c_int64, [VP, C.c_uint64, VP, C.c_uint64, VP, C.c_uint64]),
    "ps_pileup_open_cluster": (C.c_int, [VP, VP, VP, C.c_uint64]),
    "ps_pileup_head_partial": (C.c_int, [VP, VP, VP, C.c_uint64]),
    "ps_pileup_boundary_coverage": (C.c_int64, [VP, C.c_int, C.POINTER(C.c_int32), VP, C.c_uint64]),
    "ps_pileup_fault": (C.c_int, [VP, C.POINTER(ps_fault)]),
    "ps_pileup_close": (None, [VP]),
    "ps_pileup_bam": (C.c_int, [VP, C.c_char_p, C.POINTER(ps_pileup_opts), C.POINTER(VP)]),
    "ps_fasta_pack": (C.c_int, [C.c_char_p, C.POINTER(VP)]),
    "ps_fasta_reference": (C.POINTER(ps_reference), [VP]),
    "ps_fasta_contig_name": (C.c_char_p, [VP, C.c_uint32]),
    "ps_fasta_error": (C.c_char_p, [VP]),
    "ps_fasta_free": (None, [VP]),
    "ps_bam_open": (C.c_int, [C.POINTER(VP), C.c_char_p, VP, C.c_uint64, C.c_int]),
    "ps_bam_open_ex": (C.c_int, [C.POINTER(VP), C.c_char_p, VP, C.c_uint64, C.c_int, C.c_uint32]),
    "ps_bam_next": (C.c_int, [VP, C.POINTER(ps_read_batch)]),
    "ps_bam_error": (C.c_char_p, [VP]),
    "ps_bam_contig_order": (C.c_int64, [VP, VP, C.c_uint64]),
    "ps_bam_close": (None, [VP]),
    "ps_flush_create": (C.c_int, [C.POINTER(VP), C.c_uint32, C.c_uint32, C.POINTER(C.c_char_p)]),
    "ps_flush_add_snp": (C.c_int, [VP, C.c_char_p, C.c_int32, C.c_char_p, C.c_char_p]),
    "ps_flush_load_vcf": (C.c_int, [VP, C.c_char_p]),
    "ps_flush_clusters": (C.c_int, [VP, VP, C.c_uint64, VP, VP]),
    "ps_flush_totals_get": (C.c_int, [VP, C.POINTER(ps_flush_totals), VP, C.c_uint64]),
    "ps_flush_error": (C.c_char_p, [VP]),
    "ps_flush_destroy": (None, [VP]),
    "ps_track_batch": (C.c_int, [VP, C.POINTER(ps_read_batch), C.POINTER(VP)]),
    "ps_track_batch_device": (C.c_int, [VP, C.POINTER(ps_read_batch), VP, C.POINTER(VP)]),
    "ps_track_counters_get": (C.c_int, [VP, C.POINTER(ps_track_counters)]),
    "ps_track_runs": (C.c_int64, [VP, C.c_int, C.c_uint64, VP, C.c_uint64]),
    "ps_track_sites": (C.c_int64, [VP, C.c_uint64, VP, C.c_uint64]),
    "ps_track_fault": (C.c_int, [VP, C.POINTER(ps_fault)]),
    "ps_track_close": (None, [VP]),
    "ps_track_bam": (C.c_int, [VP, C.c_char_p, C.c_char_p, C.POINTER(ps_track_counters), C.POINTER(ps_fault)]),
    "ps_multi_track_bam": (C.c_int, [VP, C.c_char_p, C.c_char_p, C.POINTER(ps_track_counters), C.POINTER(ps_fault)]),
    "ps_kernel_launches": (C.c_uint64, [VP]),
    "ps_last_kernel_ms": (C.c_float, [VP]),
    "ps_kernel_times": (C.c_int, [VP, VP, C.c_int]),
    "ps_kernel_times_reset": (None, [VP, C.c_int]),
    "ps_pileup_stage_times": (C.c_int, [VP, VP]),
    "ps_pileup_flag_mode": (C.c_int, [VP]),
}

LIB_NAME = "libparasuite_b200.so"
_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def lib_path() -> str:
    # PARASUITE_B200_LIB: development override (kernel variants built side by side under lib/)
    return os.environ.get("PARASUITE_B200_LIB") or os.path.join(LIB_DIR, LIB_NAME)


def load_library() -> C.CDLL:
    """Load libparasuite_b200.so (built in-tree by __graft_entry__.build()).  Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise NativeLibraryMissing(
            f"{p} not built: run `python __graft_entry__.py build`. parasuite_b200 has no CPU fallback.")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)           # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.ps_abi_version() != PS_ABI_VERSION:
        raise RuntimeError("ABI version mismatch")
    _lib = lib
    return lib


class PsError(RuntimeError):
    def __init__(self, status: int, msg: str, fault=None):
        super().__init__(f"parasuite_b200 status {status}: {msg}")
        self.status = status
        self.fault = fault


class ReferenceWouldThrow(PsError):
    """The Java tool would have died with an uncaught exception on this input."""
