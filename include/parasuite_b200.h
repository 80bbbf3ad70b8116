/*
 * parasuite_b200.h -- C ABI of libparasuite_b200.so
 *
 * B200-native replacement of the two counting loops of PARA-suite (reference: akloetgen/PARA-suite):
 *
 *   error profile : src/src/utils/errorprofile/ErrorProfiling.java:146-409   (tool `error`, `map --refine`)
 *   T>C pileup    : src/src/utils/pileupclusters/PileupClusters.java:137-500 (tool `clust`)
 *
 * and adds one tool the Java toolkit does not have: the per-position T>C conversion and coverage track (tool `track`).
 *
 * The reference has no FFI of its own (pure Java).  This header is the boundary a thin JNI shim
 * binds (jni/parasuite_jni.c, INTEGRATION.md): plain C types, caller-owned output arrays, negative
 * PS_ERR_* status codes, no exception or CUDA error ever crosses it.  There is NO CPU fallback:
 * without a usable sm_100 GPU every compute entry point returns PS_ERR_NO_DEVICE.
 *
 * Each entry point cites the reference lines it stands in for.
 */
#ifndef PARASUITE_B200_H
#define PARASUITE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PS_ABI_VERSION 6

/* ---- status codes ------------------------------------------------------------------------ */
#define PS_OK 0
#define PS_ERR_INVALID_ARG (-1)
#define PS_ERR_NO_DEVICE (-2)          /* no CUDA device / not sm_100: there is no CPU fallback */
#define PS_ERR_CUDA (-3)
#define PS_ERR_OOM (-4)
#define PS_ERR_IO (-5)
#define PS_ERR_FORMAT (-6)             /* malformed BAM / FASTA / .fai */
#define PS_ERR_UNSORTED (-7)           /* header SO != coordinate (ErrorProfiling.java:124-132), or records whose contigs go
                                          backwards against the contig order (ps_reference_set_contig_order) */
#define PS_ERR_REFERENCE_WOULD_THROW (-8) /* input on which the JVM dies with an uncaught exception */
#define PS_ERR_STATE (-9)              /* call order violated (e.g. batch before begin) */
#define PS_ERR_UNSUPPORTED (-10)

/* reason codes reported with PS_ERR_REFERENCE_WOULD_THROW (ps_fault.code) */
#define PS_THROW_NONE 0
#define PS_THROW_REF_RANGE 1       /* FASTA fetch past contig end / unknown contig (htsjdk SAMException) */
#define PS_THROW_EMPTY_REF 2       /* refSequenceForRead[0] on an empty array (ErrorProfiling.java:180) */
#define PS_THROW_INDEL_FILL 3      /* I/D fill beyond mappingLength (ErrorProfiling.java:257,277) */
#define PS_THROW_INDEL_POS 4       /* insertions/deletionsPerPos index >= maxReadLength (:266,:287) */
#define PS_THROW_POS_MAXLEN 5      /* positionConversions[i], i >= maxReadLength (:377) */
#define PS_THROW_QUAL_RANGE 6      /* readQualities[i] out of range (:388, :405) */
#define PS_THROW_MASK51 7          /* mutationMapInRead[i], i >= 51 (PileupClusters.java:654) */
#define PS_THROW_BLOCK_RANGE 8     /* alignment block beyond the read bases (PileupClusters.java:594) */
/* not a reference exception: ps_fault.code of a record this SoA cannot hold (more than 255 CIGAR operations; htsjdk
 * takes any number, ErrorProfiling.java:206-207).  Reported with PS_ERR_UNSUPPORTED, never as a "would throw". */
#define PS_FAULT_CIGAR_OPS 9
/* not a reference exception: ps_fault.code of a mapped record that consumes no reference and whose POS lies past its
 * contig's end (ps_read_batch.past_end).  Its POS has no offset on its contig, and a batch carries no contig per record,
 * so the pileup, clust and track refuse it (PS_ERR_UNSUPPORTED) rather than place it on a contig.
 * The profile keeps the JVM's own fault for it (PS_THROW_EMPTY_REF at POS = length + 1, PS_THROW_REF_RANGE beyond). */
#define PS_FAULT_PAST_END 10

/* ---- packed reference ---------------------------------------------------------------------
 * All contigs concatenated into one coordinate space ("global offset", 0-based, < 2^32).
 *   seq2 : 2 bits/base, 16 bases per uint32, base p at bits [2*(p%16), 2*(p%16)+1] of word p/16;
 *          A=0 C=1 G=2 T=3 (case folded: ErrorProfiling.java:633-664 counts acgt like ACGT)
 *   inv  : 1 bit/base, bit p%32 of word p/32; set for every byte that is not one of ACGTacgt
 *          (such positions are never counted; seq2 holds 0 there)
 * Both arrays must be padded with >= 16 readable bytes past the last used word.
 */
typedef struct ps_reference {
  uint64_t n_bases;            /* total concatenated length */
  const uint32_t* seq2;        /* ceil(n_bases/16) words (+ padding) */
  const uint32_t* inv;         /* ceil(n_bases/32) words (+ padding) */
  uint32_t n_contigs;
  const uint64_t* contig_off;  /* [n_contigs+1] global offset of each contig's first base */
} ps_reference;

/* ---- SoA read batch -----------------------------------------------------------------------
 * What the host batcher makes of the records htsjdk would hand the Java loops, in file order.
 * Reads are grouped in tiles of PS_TILE_READS; variable-length streams are addressed by one
 * offset per tile plus an in-tile prefix sum over `meta`, so the per-read algorithmic bytes are
 *   ceil(L/4) + L + 4*n_cigar + 4 (ref_start) + 4 (meta)        (SURVEY.md 8(d)).
 */
#define PS_TILE_READS 256u

/* meta word: bits 0..15 L (read length), bits 16..23 n_cigar, bits 24..31 flags below */
#define PS_META_LEN(m) ((m) & 0xFFFFu)
#define PS_META_NCIGAR(m) (((m) >> 16) & 0xFFu)
#define PS_META_FLAGS(m) ((m) >> 24)
#define PS_MAKE_META(len, ncig, fl) (((uint32_t)(len) & 0xFFFFu) | (((uint32_t)(ncig) & 0xFFu) << 16) | ((uint32_t)(fl) << 24))
#define PS_RF_UNMAPPED 0x01u     /* BAM flag 0x4   */
#define PS_RF_REVERSE 0x02u      /* BAM flag 0x10  */
#define PS_RF_DUPLICATE 0x04u    /* BAM flag 0x400 */
#define PS_RF_POS_ZERO 0x08u     /* getAlignmentStart()==0 */
#define PS_RF_QUAL_MISSING 0x10u /* first quality byte 0xFF -> getBaseQualities() is empty */
#define PS_RF_HAS_INVALID 0x20u  /* read holds non-ACGT bases, listed in `exc` */
#define PS_RF_REF_RANGE 0x40u    /* FASTA fetch [start,end] would raise SAMException */
#define PS_RF_CIGAR_OVERFLOW 0x80u /* record had > 255 cigar ops; cigar stream holds none: every tool answers
                                      PS_ERR_UNSUPPORTED (fault code PS_FAULT_CIGAR_OPS) for a batch that holds one */

typedef struct ps_read_batch {
  uint64_t n_reads;
  const uint32_t* meta;           /* [n_reads] */
  const uint32_t* ref_start;      /* [n_reads] global 0-based offset of POS; undefined if unmapped/POS==0 */
  const uint8_t* bases2;          /* 2-bit codes, read r: ceil(L/4) bytes, base p at bits 2*(p%4) of byte p/4 */
  const uint8_t* qual;            /* raw phred bytes, L per read (kept even when missing) */
  const uint32_t* cigar;          /* BAM encoding len<<4|op, op 0..8 = MIDNSHP=X */
  const uint64_t* tile_base_off;  /* [n_tiles+1] byte offset of each tile in bases2 */
  const uint64_t* tile_qual_off;  /* [n_tiles+1] byte offset of each tile in qual */
  const uint64_t* tile_cigar_off; /* [n_tiles+1] element offset of each tile in cigar */
  const uint32_t* tile_exc_off;   /* [n_tiles+1] element offset of each tile in exc */
  const uint32_t* exc;            /* invalid read bases: (read_in_tile << 16) | position, sorted.  Every tool reads a
                                     listed base as N and ignores the code bases2 holds there (any value may be stored) */
  uint32_t uniform_len;           /* != 0: every read has this L (offsets are closed-form) */
  uint32_t uniform_ncigar;        /* != 0: every read has this many cigar ops */
  uint64_t bases_bytes;           /* total sizes of the streams (for copies) */
  uint64_t qual_bytes;
  uint64_t cigar_count;
  uint64_t exc_count;
  uint32_t max_len;               /* longest read of the batch when the producer knows it, else 0 (a hint: ragged batches of
                                     short reads are re-laid in rows of 16*ceil(min(max_len, max_read_length)/16) positions) */
  /* Compact form of a HOST batch of the PAR-CLIP shape, for the calls that upload it (ps_profile_batch, ps_pileup_batch,
   * ps_batch_upload): fewer bytes over the host link, expanded on the device by the upload.
   *   uniform_cigar != 0 (with uniform_ncigar == 1): every read's one cigar op is this word; `cigar` may be NULL
   *   flags8 != NULL (with uniform_len and uniform_ncigar): the PS_RF_* flags, one byte per read; `meta` may be NULL
   *   qual6 != NULL (with uniform_len): the qualities packed 6 bits each -- four per three bytes, little endian,
   *     ceil(L/4)*3 bytes per read, every quality <= 63 (no read with PS_RF_QUAL_MISSING); `qual` may be NULL,
   *     qual_bytes still counts the unpacked bytes
   *   start16 != NULL (with tile_start): ref_start[r] = tile_start[r / PS_TILE_READS] + start16[r] -- a sorted batch
   *     whose tiles of 256 reads each span less than 65536 bases; `ref_start` may be NULL
   * The view ps_batch_upload returns always holds the expanded `meta`, `cigar`, `qual` and `ref_start`. */
  uint32_t uniform_cigar;
  const uint8_t* flags8;
  const uint8_t* qual6;
  const uint16_t* start16;
  const uint32_t* tile_start;
  /* 1 + the ordinal of the first mapped record (POS != 0, at most 255 CIGAR operations) that consumes no reference and
   * whose POS is past its contig's end; 0: the batch holds none.  Set by the producers, which know each record's contig
   * (ps_bam_next, ReadBatch.from_records); the tools answer PS_FAULT_PAST_END for that record unless a record before it
   * faults first.  The producers give every such record the offset of its contig's last base, so that a slice that
   * leaves the first one out (and sets past_end relative to itself, 0 when the record lies outside it) keeps the rest
   * on their own contigs. */
  uint64_t past_end;
} ps_read_batch;

/* ---- error profile ------------------------------------------------------------------------ */
typedef struct ps_profile_opts {
  uint32_t max_read_length;  /* ErrorProfiling ctor arg (ErrorProfiling.java:58-64) */
  uint32_t infer_qualities;  /* `-q` (ErrorProfiling.java:402-407): also fill the quality histogram */
  uint32_t emit_t2c_masks;   /* device-resident batches of the PAR-CLIP shape: leave one T>C mask word per read in HBM
                                (ps_profile_masks_device) for a pileup call on the SAME batch (ps_pileup_opts) */
  uint32_t reserved;
} ps_profile_opts;

/* counters[] order (ErrorProfiling.java:134-141, :54) */
enum {
  PS_PC_NUM_READS_PROCESSED = 0,
  PS_PC_UNMAPPED,
  PS_PC_DUPLICATES,
  PS_PC_START_ZERO,
  PS_PC_INDEL_READ,
  PS_PC_SKIPPED_READS,
  PS_PC_LONGER_INDELS,
  PS_PC_TOTAL_BASES_CHECKED,
  PS_PC_COUNT
};

typedef struct ps_fault {
  int32_t code;          /* PS_THROW_* */
  uint64_t read_ordinal; /* 0-based ordinal (over all batches since begin) of the first such record */
} ps_fault;

/* Caller-allocated outputs, bit-identical to the Java fields after the loop :146-409.
 * int32 arrays carry Java's two's-complement wrap-around; the *_wide arrays (optional, may be NULL)
 * receive the un-wrapped 64-bit sums. */
typedef struct ps_profile_result {
  int32_t* position_conversions;      /* [max_read_length*16]  ([i][ref][read]) */
  int32_t* quality_per_mismatch;      /* [16] */
  int32_t* quality_per_mismatch_counts; /* [16] */
  double* insertions_per_pos;         /* [max_read_length] */
  double* deletions_per_pos;          /* [max_read_length] */
  int32_t* counters;                  /* [PS_PC_COUNT] */
  int64_t* quality_hist;              /* [max_read_length*256] or NULL (only with infer_qualities) */
  int64_t* wide;                      /* [ps_profile_acc_len()] raw accumulator vector or NULL */
  ps_fault fault;
} ps_profile_result;

/* accumulator vector layout (int64), the unit of the multi-GPU all-reduce (SURVEY 8(e)):
 *   [0, 16*maxLen) positionConversions | +16 qualityPerMismatch | +16 qualityPerMismatchCounts
 *   | +maxLen insertionsPerPos | +maxLen deletionsPerPos | +PS_PC_COUNT counters
 *   | (+256*maxLen quality histogram with infer_qualities) */
size_t ps_profile_acc_len(uint32_t max_read_length, uint32_t infer_qualities);

/* The six output files of the `error` tool after the loop (ErrorProfiling.java:410-591): <bam>.errorprofile,
 * .errorprofile.vcf, .qualityPerMismatch, .indels, .indelprofile, .qualities (empty without infer_qualities), from a
 * filled result.  Host only.  *averaged_t2c_epr (may be NULL) receives the value of the "Averaged T2C" log line. */
int ps_profile_write_files(const ps_profile_result* res, uint32_t max_read_length, uint32_t infer_qualities,
                           const char* bam_path, double* averaged_t2c_epr, char* err, size_t err_cap);

/* ---- T>C pileup ---------------------------------------------------------------------------- */
typedef struct ps_cluster {      /* one closed cluster, state at PileupClusters.java:178 (before the SNP filter) */
  uint64_t first_read;           /* ordinal of the read that opened it */
  uint32_t running_id;           /* "cl_<running_id>_<chr>"; first cluster is 2 (PileupClusters.java:355) */
  uint32_t contig;               /* index into the reference contig table */
  int32_t start;                 /* tempClusterStart, 1-based */
  int32_t end;                   /* tempClusterEnd */
  uint32_t num_reads;            /* numReadsPerCluster */
  uint32_t num_t2c;              /* numT2CMutationPerCluster */
  uint32_t minus_after_first;    /* minus-strand members after the first read (P6) */
  uint8_t first_reverse;         /* tempIsReverse */
  uint8_t combined_strand;       /* 0 "+", 1 "-", 2 "+/-"  (StrandOrientation.java:48-56) */
  uint16_t reserved;
  uint64_t mask51;               /* alleleFrequencyPositionsTemp as bits */
  uint64_t site_begin;           /* [site_begin, site_end) in the site array */
  uint64_t site_end;
} ps_cluster;

typedef struct ps_site {         /* one key of mutationMap with its baseCoveredMap value */
  int32_t pos;                   /* checkPosition, 1-based */
  uint32_t t2c;                  /* mutationMap value */
  uint32_t cov;                  /* baseCoveredMap value */
  uint32_t reserved;
  uint64_t order_key;            /* (ordinal of the read that first put this key << 6) | i  -- sorting a
                                    cluster's sites by it gives the HashMap.put order (SURVEY P8) */
} ps_site;

typedef struct ps_pileup_counters {
  uint64_t num_reads_processed;  /* PileupClusters.java:138 */
  uint64_t skipped_due_indel;    /* :156 */
  uint64_t double_stranded;      /* :496 (incl. the never-flushed last cluster) */
  uint64_t n_clusters;           /* closed clusters returned */
  uint64_t n_sites;
  uint8_t has_open_cluster;      /* the reference never flushes the last cluster (:528-529) */
} ps_pileup_counters;

typedef struct ps_ctx ps_ctx;
typedef struct ps_pileup ps_pileup;   /* opaque result handle */

/* ---- lifecycle ----------------------------------------------------------------------------- */
int ps_abi_version(void);
/* One context per GPU (one process per GPU under torch.distributed; a JVM holds several through ps_create_multi). */
int ps_create(ps_ctx** out, int device);
void ps_destroy(ps_ctx* ctx);
const char* ps_last_error(const ps_ctx* ctx);
const char* ps_strerror(int status);

/* ---- reference ------------------------------------------------------------------------------
 * Replaces `new IndexedFastaSequenceFile(fasta)` + one getSubsequenceAt per read
 * (ErrorProfiling.java:109-110,169-172; PileupClusters.java:66,598-601): the whole reference is
 * packed once and stays resident in HBM. */
int ps_reference_upload(ps_ctx* ctx, const ps_reference* host_ref);
int ps_reference_load_fasta(ps_ctx* ctx, const char* fasta_path); /* needs <fasta>.fai */
/* adopt device-resident arrays (no copy; caller keeps them alive) */
int ps_reference_adopt_device(ps_ctx* ctx, const ps_reference* dev_ref, const uint64_t* host_contig_off);
/* The order the input's records take through the contigs (a coordinate-sorted file follows the @SQ order of its own
 * header, which need not be the FASTA's).  The Java tools fetch bases by contig NAME (getSubsequenceAt(chr, ..),
 * ErrorProfiling.java:169-172, PileupClusters.java:598-601) and close a cluster whenever the contig CHANGES
 * (PileupClusters.java:175-176), so they follow any order; the pileup keeps a running maximum over the records and needs
 * to know it.  order[k] = FASTA index of the k-th contig; contigs not listed come after the listed ones, in FASTA order.
 * order == NULL or n == 0: FASTA order, which is also the state after every reference upload, load or adopt.
 *   - A kept record on a contig that comes earlier in this order than the record before it: PS_ERR_UNSORTED.
 *   - ps_pileup_opts.carry_contig and the `contig` of ps_pileup_max_key stay FASTA indices; the device keys
 *     (ps_pileup_max_key_device, carry_keys_device) are (position in this order + 1) << 32 | end, so keys of two contexts
 *     compare only when both have the same order.
 *   - The profile does not depend on the order.  The file tools (ps_pileup_bam, ps_clust_bam and their ps_multi_* forms)
 *     take the order of the file's header for the call, on every context they drive, and leave the caller's order in
 *     force afterwards.
 * Waits for all work already queued on the context's device before it changes the table.  PS_ERR_INVALID_ARG: an
 * index twice, an index >= n_contigs, n > n_contigs; PS_ERR_STATE: no reference yet, or a ps_pileup_submit_device call
 * not waited for. */
int ps_reference_set_contig_order(ps_ctx* ctx, const uint32_t* order, uint32_t n);

/* ---- batches -----------------------------------------------------------------------------------
 * Copy a host batch (pinned or pageable) into device memory owned by the context, asynchronously on the context's
 * stream, and return a device-resident view of it for the *_batch_device calls (pass stream = NULL so they run on
 * the same stream, after the copy).  The view stays valid until the second-next ps_batch_upload / ps_*_batch call on
 * this context (two staging slots).  Lets the two tools share one upload of the same records. */
int ps_batch_upload(ps_ctx* ctx, const ps_read_batch* host_batch, ps_read_batch* dev_view);
/* (A *_batch_device / ps_pileup_max_key_device call that is handed such a view together with a stream of the caller's
 * waits, on that stream, for the part of the upload it reads: everything for the profile, everything but the quality
 * bytes -- which travel last -- for the pileup and the key kernel.) */

/* ---- error profile: replaces the loop ErrorProfiling.java:146-409 ---------------------------- */
int ps_profile_begin(ps_ctx* ctx, const ps_profile_opts* opts);
/* host-resident batch: staged through pinned memory, H2D, kernels; asynchronous, returns when queued */
int ps_profile_batch(ps_ctx* ctx, const ps_read_batch* host_batch);
/* device-resident batch (all pointers are device pointers) on `stream` (a cudaStream_t, may be NULL) */
int ps_profile_batch_device(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream);
/* With ps_profile_opts.emit_t2c_masks: device address of the mask words of the LAST ps_profile_batch_device call of the
 * open run (*n_words = its n_reads), written on that call's stream; *dev_masks = NULL when that batch did not have the
 * PAR-CLIP shape (uniform length <= 62, one cigar op).  Valid until the next profile batch on this context. */
int ps_profile_masks_device(ps_ctx* ctx, const uint64_t** dev_masks, uint64_t* n_words);
/* device address of the int64 accumulator vector (for an NCCL all-reduce by the caller) */
int ps_profile_acc_device(ps_ctx* ctx, void** dev_ptr, size_t* n_int64);
/* The accumulator vector of the open run is next touched on `stream` (e.g. an all-reduce queued there, ordered behind
 * the batch kernels by the caller): ps_profile_end reads it back on that stream and waits for that stream only -- not
 * for other work queued behind the batch kernels on their own stream (a submitted pileup call, say). */
int ps_profile_set_stream(ps_ctx* ctx, void* stream);
/* synchronise, wrap to Java int semantics, fill the caller's arrays */
int ps_profile_end(ps_ctx* ctx, ps_profile_result* out);
/* whole tool loop from files (BAM must be coordinate sorted) */
int ps_profile_bam(ps_ctx* ctx, const char* bam_path, const ps_profile_opts* opts, ps_profile_result* out);

/* ---- T>C pileup: replaces the loop PileupClusters.java:137-500 (+ :585-673) ------------------- */
typedef struct ps_pileup_opts {
  uint32_t first_running_id;  /* runningID before the first cluster; reference: 1 (PileupClusters.java:133) */
  /* carry-in from a preceding shard (halo merge, SURVEY 8(e)); all zero for a whole file */
  uint32_t carry_valid;
  uint32_t carry_contig;
  int32_t carry_cluster_end;
  /* the same carry-in left on the DEVICE: carry_keys_n keys as ps_pileup_max_key_device writes them, one per preceding
   * shard (e.g. the first `rank` entries of an NCCL all-gather); their maximum is the carry-in, no host round trip.
   * Ignored when carry_keys_n == 0; combined (max) with the host triple above when both are given. */
  uint32_t carry_keys_n;
  const uint64_t* carry_keys_device;
  /* Optional: the T>C mask words ps_profile_batch_device left for THIS batch (ps_profile_masks_device), one per read:
   * bit 63 = word valid, bit 62 = minus strand, bits 0..61 = T>C by index of the strand-oriented read
   * (mutationMapInRead, PileupClusters.java:651-661).  The pileup then reads 12 bytes per record instead of decoding
   * bases and reference again; records without a valid word are decoded as usual.  The caller vouches that the words
   * belong to the same records and reference.  NULL: decode every record. */
  const uint64_t* t2c_masks_device;
} ps_pileup_opts;

int ps_pileup_batch(ps_ctx* ctx, const ps_read_batch* host_batch, const ps_pileup_opts* opts, ps_pileup** out);
int ps_pileup_batch_device(ps_ctx* ctx, const ps_read_batch* dev_batch, const ps_pileup_opts* opts, void* stream,
                           ps_pileup** out);
/* The same call in two halves: ps_pileup_submit_device queues the kernels on `stream` and returns without waiting for
 * the device; ps_pileup_wait completes the call (it may have to repeat a pass with larger arrays) and returns what
 * ps_pileup_batch_device would have returned.  In between the host is free (e.g. to take back the profile of the same
 * batch); every other ps_pileup_* call on the handle except ps_pileup_close answers PS_ERR_STATE until the wait, and a
 * context takes one submitted call at a time.  ps_pileup_close on a submitted handle waits first. */
int ps_pileup_submit_device(ps_ctx* ctx, const ps_read_batch* dev_batch, const ps_pileup_opts* opts, void* stream,
                            ps_pileup** out);
int ps_pileup_wait(ps_pileup* h);
/* Region sharding: max over the batch's kept records of (contig, alignment end), contigs compared by their position in
 * the context's contig order (ps_reference_set_contig_order); *contig is the FASTA index.  The exclusive prefix-max of
 * these over the shards (one pair per shard: an all-gather of 8 scalars) is shard s's carry-in, so all shards run at
 * once. */
int ps_pileup_max_key(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream, uint32_t* valid, uint32_t* contig,
                      int32_t* end);
/* The same maximum left on the device, asynchronously on `stream`: *dev_key points to one uint64 owned by the context,
 * (position of the contig in the context's contig order + 1) << 32 | end, 0 if the batch holds no kept record; valid
 * until the next call of this function. */
int ps_pileup_max_key_device(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream, uint64_t** dev_key);
int ps_pileup_counters_get(const ps_pileup* h, ps_pileup_counters* out);
/* copy up to `max_clusters` closed clusters starting at `first` (and their sites) into caller arrays;
 * returns the number copied (>= 0) or a negative status */
int64_t ps_pileup_next(ps_pileup* h, uint64_t first, ps_cluster* clusters, uint64_t max_clusters, ps_site* sites,
                       uint64_t max_sites);
/* the still-open last cluster (never flushed by the reference); needed for the halo merge */
int ps_pileup_open_cluster(ps_pileup* h, ps_cluster* cluster, ps_site* sites, uint64_t max_sites);
/* with opts->carry_valid: the leading reads that continue the preceding shard's open cluster (returns 1 and the
 * partial sums to merge into it, or 0).  first_read/start/first_reverse describe the first such read only. */
int ps_pileup_head_partial(ps_pileup* h, ps_cluster* cluster, ps_site* sites, uint64_t max_sites);
/* baseCoveredMap of a boundary cluster as a dense array: cov[k] = coverage at position *first_pos + k.
 * which = 0: head partial, 1: open cluster.  cov == NULL just returns the length.  A T>C site seen on one side
 * of a shard cut is also covered by reads on the other side; the merge adds this in. */
int64_t ps_pileup_boundary_coverage(ps_pileup* h, int which, int32_t* first_pos, uint32_t* cov, uint64_t max);
int ps_pileup_fault(const ps_pileup* h, ps_fault* out);
void ps_pileup_close(ps_pileup* h);
/* The file is taken in windows of records (PARASUITE_B200_WINDOW_READS, default 2^23), in the contig order of the file's
 * header (ps_reference_set_contig_order): every window's carry-in is the maximum (contig, end) over the windows before it, the reads at its head that continue the cluster left open by the
 * window before are folded into that cluster on the host (halo merge).  The handle holds the merged records of the whole
 * file on the host; no limit on the number of records. */
int ps_pileup_bam(ps_ctx* ctx, const char* bam_path, const ps_pileup_opts* opts, ps_pileup** out);
/* The whole `clust` tool from files (PileupClusters.calculateReadPileups, :62-584): record loop on the GPU in windows,
 * flush arithmetic and the six output files natively (ps_flush_*, ps_clust_writer_*).  snp_vcf may be NULL.  The
 * reference must have been loaded with ps_reference_load_fasta (the raw-case FASTA is read for the sequence columns). */
int ps_clust_bam(ps_ctx* ctx, const char* bam_path, const char* out_path, const char* snp_vcf, uint32_t min_read_coverage,
                 ps_pileup_counters* counters_out, ps_fault* fault_out);
/* The whole `error` tool from files (ErrorProfiling.inferErrorProfile without the plot): ps_profile_bam + the six
 * output files next to the BAM (ps_profile_write_files).  counters_out: [PS_PC_COUNT] or NULL. */
int ps_error_bam(ps_ctx* ctx, const char* bam_path, const ps_profile_opts* opts, int32_t* counters_out, ps_fault* fault_out);

/* ---- T>C conversion and coverage track (tool `track`; no Java counterpart) ----------------------------------------
 * Per position and strand: the coverage and the T>C events of the records the pileup keeps (ps_pileup_batch: unmapped
 * records and those whose CIGAR holds (I or D) and N are skipped, duplicates counted; the same faults with the same
 * ordinals, except that there is no 51-position limit -- PS_THROW_MASK51 is never raised).  Positions follow the CIGAR on
 * the genome: M, =, X consume read and reference, D and N the reference only (no coverage), I and S the read only, H and
 * P nothing.  BAM flag 0x10 puts a read on the minus track.  Every aligned base adds 1 to its strand's coverage, whatever
 * the bases; a T>C event is ref T / read C on the plus strand and ref A / read G on the minus strand (T>C on the read's
 * own strand), counted where the reference base is ACGTacgt and the read base is not listed in `exc`.
 * A kept record whose start is smaller than the previous kept record's (contig order included:
 * ps_reference_set_contig_order) gives PS_ERR_UNSORTED. */
typedef struct ps_track_counters {
  uint64_t num_reads_processed;
  uint64_t unmapped;
  uint64_t skipped_due_indel;
  uint64_t reads_counted;        /* records on the track */
  uint64_t aligned_bases[2];     /* [strand]: 0 plus, 1 minus; = sum over runs of (end0 - start0) * cov */
  uint64_t t2c_events[2];        /* = sum of t2c over the strand's sites */
  uint64_t n_runs[2];
  uint64_t n_sites;
  uint64_t fast_path_reads;      /* reads whose T>C bits were found bit-parallel (uniform length <= 64, one M/=/X op) */
} ps_track_counters;
typedef struct ps_track_run {    /* one bedGraph row: maximal run of equal non-zero coverage */
  uint32_t contig;               /* FASTA index */
  uint32_t start0;               /* 0-based, half-open */
  uint32_t end0;
  uint32_t cov;
} ps_track_run;
typedef struct ps_track_site {   /* one (position, strand) with at least one T>C event */
  uint32_t contig;               /* FASTA index */
  int32_t pos;                   /* 1-based */
  uint32_t strand;               /* 0 plus, 1 minus */
  uint32_t t2c;
  uint32_t cov;                  /* coverage of that strand at pos */
} ps_track_site;
typedef struct ps_track ps_track;  /* opaque result handle (host memory) */
/* One batch is the whole input.  Runs come by strand, contigs in the order the records visit them, then by position;
 * sites likewise, plus before minus at one position.  The handle is returned with PS_OK and with a fault
 * (PS_ERR_REFERENCE_WOULD_THROW, PS_ERR_UNSUPPORTED: ps_track_fault). */
int ps_track_batch(ps_ctx* ctx, const ps_read_batch* host_batch, ps_track** out);
int ps_track_batch_device(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream, ps_track** out);
int ps_track_counters_get(const ps_track* h, ps_track_counters* out);
/* copy up to `max` runs of `strand` (0 plus, 1 minus) / sites starting at `first`; returns the number copied */
int64_t ps_track_runs(const ps_track* h, int strand, uint64_t first, ps_track_run* runs, uint64_t max);
int64_t ps_track_sites(const ps_track* h, uint64_t first, ps_track_site* sites, uint64_t max);
int ps_track_fault(const ps_track* h, ps_fault* out);
void ps_track_close(ps_track* h);
/* Per-position base counts (opts->base_counts != 0), beside the runs and sites, which stay as they are:
 * - Scope: the records, faults, ordinals, positions and strand rule of the track.  Every aligned base at a position whose
 *   reference is ACGTacgt is counted by read base A, C, G, T or N; N is a base listed in `exc`, whatever bases2 holds.
 *   Positions whose reference is not ACGT give no row and count toward no total (their coverage is in the runs as ever).
 * - Orientation: bases on the read's strand.  On the minus strand reference and read base are complemented, so ref T /
 *   column C is T>C on both strands: for a row with ref T, n[1] is the t2c of the site at (pos, strand), 0 without one.
 * - A position gets a row on a strand when that strand's coverage is >= min_coverage and the selected substitutions
 *   there number >= min_events.  substitutions: bit 4 * ref + read (A0 C1 G2 T3, strand orientation); diagonal bits are
 *   ignored; 0 selects all twelve; bits above 15 give PS_ERR_INVALID_ARG.  N calls are never events; a threshold of 0
 *   counts as 1.
 * - Rows come in the sites' order: contigs in the order the records visit them, then by position, plus before minus.
 * - totals.bases[strand][ref][read] counts every counted base, with or without a row: its cells sum to the aligned bases
 *   at ACGT reference positions, and bases[s][3][1] == t2c_events[s].  ps_track_counters is the same with or without. */
typedef struct ps_track_opts {
  uint32_t base_counts;          /* 0: the plain track */
  uint32_t min_coverage;
  uint32_t min_events;
  uint32_t substitutions;        /* 16-bit mask, 0 = all twelve */
} ps_track_opts;
typedef struct ps_track_base_row { /* 36 B */
  uint32_t contig;               /* FASTA index */
  int32_t pos;                   /* 1-based */
  uint8_t strand;                /* 0 plus, 1 minus */
  uint8_t ref;                   /* reference base in strand orientation, A0 C1 G2 T3 */
  uint16_t reserved;
  uint32_t cov;                  /* coverage of that strand at pos = n[0] + ... + n[4] */
  uint32_t n[5];                 /* read bases A, C, G, T, N in strand orientation */
} ps_track_base_row;
typedef struct ps_track_base_totals {
  uint64_t bases[2][4][5];       /* [strand][ref][read A C G T N] */
  uint64_t n_rows;
} ps_track_base_totals;
/* opts == NULL: ps_track_batch / ps_track_batch_device */
int ps_track_batch_ex(ps_ctx* ctx, const ps_read_batch* host_batch, const ps_track_opts* opts, ps_track** out);
int ps_track_batch_device_ex(ps_ctx* ctx, const ps_read_batch* dev_batch, const ps_track_opts* opts, void* stream,
                             ps_track** out);
/* PS_ERR_STATE on a handle made without base counts; rows: copy up to `max` from `first`, returns the number copied */
int64_t ps_track_base_rows(const ps_track* h, uint64_t first, ps_track_base_row* rows, uint64_t max);
int ps_track_base_totals_get(const ps_track* h, ps_track_base_totals* out);
/* The tool from files: <out_prefix>.plus.bedGraph and <out_prefix>.minus.bedGraph (chrom, start0, end0, coverage; no
 * header; one row per maximal run of equal non-zero coverage) and <out_prefix>.t2c.tsv (header
 * chrom/pos/strand/t2c/coverage, one row per (position, strand) with t2c >= 1, pos 1-based).  Contigs come in the order the
 * records visit them (the header's), rows by position.  The file is taken in windows of PARASUITE_B200_WINDOW_READS
 * records; the files do not depend on the window size nor on the number of devices.  The reference must have been loaded
 * with ps_reference_load_fasta / ps_multi_load_fasta (contig names).  counters_out / fault_out may be NULL. */
int ps_track_bam(ps_ctx* ctx, const char* bam_path, const char* out_prefix, ps_track_counters* counters_out,
                 ps_fault* fault_out);
/* With opts->base_counts also <out_prefix>.bases.tsv (header chrom/pos/strand/ref/coverage/A/C/G/T/N, the rows of
 * ps_track_base_rows, pos 1-based), independent of the window size and the number of devices; the other three files are
 * byte-identical to ps_track_bam's.  opts == NULL: ps_track_bam.  totals_out may be NULL. */
int ps_track_bam_ex(ps_ctx* ctx, const char* bam_path, const char* out_prefix, const ps_track_opts* opts,
                    ps_track_counters* counters_out, ps_track_base_totals* totals_out, ps_fault* fault_out);

/* ---- `comb` tool (host only): transcript hits lifted to genomic coordinates, merged with the genomic hits ---------------
 * Replaces CombineGenomeTranscript.combine / printReadsToBamFile (utils/postprocessing/CombineGenomeTranscript.java:36-666;
 * Main.java:438-486 `comb -g <genomic.bam> -t <transcript.bam> -o <combined.bam>`): the step that writes the `aMbNcM`
 * cigars both kernels must tolerate.  The transcript BAM must be queryname-sorted and its reference names must be
 * gene|transcript|chr|exonStarts;..|exonEnds;..|strand (PS_ERR_UNSORTED / PS_ERR_REFERENCE_WOULD_THROW otherwise). */
typedef struct ps_comb_stats {
  uint64_t genomic_records;                /* copied through from the genomic BAM */
  uint64_t transcript_records;             /* read from the transcript BAM */
  uint64_t lifted_records;                 /* written with genomic coordinates */
  uint64_t mapped_reads;                   /* mappedReads (:59, :662) */
  uint64_t spliced_reads;                  /* splicedReads (:479) */
  uint64_t missed_transcript_alignments;   /* indel + splice junction (:294, :431, :447) */
} ps_comb_stats;
/* One hit (:146-474).  *new_start = -1: the hit does not lift.  On PS_ERR_REFERENCE_WOULD_THROW new_cigar holds the message. */
int ps_liftover_hit(const char* transcript_name, int32_t aln_start, int32_t aln_end, int32_t read_len, const char* cigar,
                    int32_t* new_start, char* new_cigar, size_t new_cigar_cap, uint32_t* missed);
int ps_comb_bam(const char* genomic_bam, const char* transcript_bam, const char* out_bam, ps_comb_stats* stats, char* err,
                size_t err_cap);

/* ---- several GPUs behind one handle (one process, e.g. a JVM; Main.java:595-597, :634-636 enter here) -----------------
 * devices == NULL or n == 0: the list in PARASUITE_B200_DEVICES ("0,1,2"), else device 0.  The handle owns one context
 * per device.  The reference is packed once and made resident on every device; the profile sends batches round-robin and
 * sums the (< 10 KB) accumulator vectors on the host, the pileup sends windows round-robin and merges the boundary
 * clusters on the host (SURVEY 8(e)).  Results are bit-identical to the single-context calls. */
typedef struct ps_multi ps_multi;
int ps_create_multi(ps_multi** out, const int* devices, int n);
void ps_destroy_multi(ps_multi* m);
int ps_multi_device_count(const ps_multi* m);
ps_ctx* ps_multi_context(ps_multi* m, int i);            /* borrowed: for batch-level calls on one of the devices */
const char* ps_multi_last_error(const ps_multi* m);
int ps_multi_load_fasta(ps_multi* m, const char* fasta_path);
int ps_multi_profile_bam(ps_multi* m, const char* bam_path, const ps_profile_opts* opts, ps_profile_result* out);
int ps_multi_pileup_bam(ps_multi* m, const char* bam_path, const ps_pileup_opts* opts, ps_pileup** out);
int ps_multi_error_bam(ps_multi* m, const char* bam_path, const ps_profile_opts* opts, int32_t* counters_out, ps_fault* fault_out);
int ps_multi_clust_bam(ps_multi* m, const char* bam_path, const char* out_path, const char* snp_vcf,
                       uint32_t min_read_coverage, ps_pileup_counters* counters_out, ps_fault* fault_out);
/* windows round-robin over the devices; the files are byte-identical to ps_track_bam's */
int ps_multi_track_bam(ps_multi* m, const char* bam_path, const char* out_prefix, ps_track_counters* counters_out,
                       ps_fault* fault_out);
int ps_multi_track_bam_ex(ps_multi* m, const char* bam_path, const char* out_prefix, const ps_track_opts* opts,
                          ps_track_counters* counters_out, ps_track_base_totals* totals_out, ps_fault* fault_out);

/* ---- host batcher (usable without a GPU) --------------------------------------------------------
 * What htsjdk does for the two loops, as a library: FASTA(+.fai) -> packed reference; BGZF/BAM -> SoA batches in
 * page-locked host memory (pageable when no CUDA device is present), records in file order, presented exactly as
 * SAMRecord presents them to ErrorProfiling.java:146-409 / PileupClusters.java:137-500. */
typedef struct ps_packed_fasta ps_packed_fasta;
typedef struct ps_bam ps_bam;
/* *out is set even on failure (read ps_fasta_error / ps_bam_error, then free / close it) */
int ps_fasta_pack(const char* fasta_path, ps_packed_fasta** out);           /* needs <fasta>.fai */
const ps_reference* ps_fasta_reference(const ps_packed_fasta* f);            /* host arrays owned by f */
const char* ps_fasta_contig_name(const ps_packed_fasta* f, uint32_t i);
const char* ps_fasta_error(const ps_packed_fasta* f);
void ps_fasta_free(ps_packed_fasta* f);
/* Opens a coordinate-sorted BAM (PS_ERR_UNSORTED otherwise: ErrorProfiling.java:124-132).  Contigs are matched to the
 * FASTA by name, as getSubsequenceAt(chr, ..) does (ErrorProfiling.java:169-172); records on a contig the FASTA lacks
 * carry PS_RF_REF_RANGE.  max_batch_reads = 0 picks a default; threads <= 0 uses the host cores.
 * ps_bam_open answers PS_ERR_UNSUPPORTED when the header lists the FASTA's contigs in another order than the FASTA index:
 * its records would not follow the FASTA order a context keys the pileup in by default.  ps_bam_open_ex with
 * PS_BAM_ANY_CONTIG_ORDER takes any header order, as the Java tools do; the caller then keys the pileup in the header's
 * order (ps_bam_contig_order -> ps_reference_set_contig_order).  The file tools (ps_profile_bam, ps_pileup_bam,
 * ps_clust_bam, ps_error_bam and the ps_multi_* forms) open their input this way and do that themselves. */
#define PS_BAM_ANY_CONTIG_ORDER 1u
int ps_bam_open(ps_bam** out, const char* bam_path, const ps_packed_fasta* ref, uint64_t max_batch_reads, int threads);
int ps_bam_open_ex(ps_bam** out, const char* bam_path, const ps_packed_fasta* ref, uint64_t max_batch_reads, int threads,
                   uint32_t flags);
/* The file's contig order for ps_reference_set_contig_order: FASTA indices of the @SQ lines in header order, contigs the
 * FASTA lacks left out.  Returns its length; order == NULL asks for the length only (PS_ERR_INVALID_ARG if it exceeds
 * max). */
int64_t ps_bam_contig_order(const ps_bam* b, uint32_t* order, uint64_t max);
/* 1: *batch filled (host pointers, valid until the third-next call); 0: end of file; < 0: status */
int ps_bam_next(ps_bam* b, ps_read_batch* batch);
const char* ps_bam_error(const ps_bam* b);
void ps_bam_close(ps_bam* b);

/* ---- cluster flush (host code, usable without a GPU) ----------------------------------------------
 * What PileupClusters.java does with every closed cluster before it writes its rows (:178-260: SNP filter,
 * anchor site, sorted T>C fractions, allele statistics) and the run totals (:502-545), on the records ps_pileup_next
 * returns.  The anchor tie-break follows java.util.HashMap (JDK 8+) iteration order; SNPs as SNPCalling.java:49-69. */
typedef struct ps_flush ps_flush;
typedef struct ps_flush_row {
  uint8_t emitted;           /* numReadsPerCluster >= minReadCoverage: the cluster row is written (:180, :317-343) */
  uint8_t has_ccr;           /* tempBestMutationPos > 0: CCR FASTA + row are written (:262-315) */
  uint16_t reserved;
  uint32_t num_t2c_sites;    /* numT2CSitesPerCluster = mutationMap.size() before the SNP filter (:181) */
  int32_t best_pos;          /* tempBestMutationPos, -1 if none */
  uint32_t best_count;       /* mutationMap.get(tempBestMutationPos) */
  double best_value;         /* tempBestMutationValue */
  double fraction;           /* fractionT2CMutationPerCluster */
} ps_flush_row;
typedef struct ps_flush_totals {
  uint64_t snp_hit;                    /* :193 */
  uint64_t high_frequent_error;        /* :196 */
  uint64_t num_crosslinked_clusters;   /* :250 */
  uint64_t num_allele_positions;       /* :254 */
  uint64_t allele_positions[51];       /* :253 */
  uint64_t n_allele_frequency;         /* alleleFrequencyInformation.size() */
} ps_flush_totals;
int ps_flush_create(ps_flush** out, uint32_t min_read_coverage, uint32_t n_contigs, const char* const* contig_names);
int ps_flush_add_snp(ps_flush* f, const char* chrom, int32_t pos, const char* ref, const char* alt0);
int ps_flush_load_vcf(ps_flush* f, const char* vcf_path);     /* plain, gzip or bgzip */
int ps_flush_clusters(ps_flush* f, const ps_cluster* clusters, uint64_t n, const ps_site* sites, ps_flush_row* rows);
int ps_flush_totals_get(const ps_flush* f, ps_flush_totals* out, double* allele_frequency_information, uint64_t max);
const char* ps_flush_error(const ps_flush* f);
void ps_flush_destroy(ps_flush* f);

/* ---- output files of the clust tool (host code, usable without a GPU) --------------------------------------
 * What PileupClusters.java writes: <out> (cluster rows with the cluster sequence assembled read by read, :317-343 and
 * :367-487), <out>.ccr.fasta / <out>.ccr.tsv (:262-315), <out>.report (:502-514), <bam>.sitefrequency.tsv and
 * <bam>.sitepositions.tsv (:529-545) -- byte for byte, doubles printed as Double.toString prints them.
 * The writer is fed, batch by batch and in file order, with the host SoA of the records (it walks their CIGARs for the
 * cluster sequence) and with the clusters that closed with that batch (ps_pileup_next; after the halo merge when the
 * file is taken in windows); it flushes them through `flush` (ps_flush_clusters must not be called for them again).
 * A read opens a cluster iff its ordinal is the first_read of the next record: boundaries are never re-derived here.
 * fasta_path needs <fasta>.fai; contigs must be those of the packed reference, in the same order. */
typedef struct ps_clust_writer ps_clust_writer;
int ps_clust_writer_open(ps_clust_writer** out, ps_flush* flush, const char* fasta_path, const char* out_path,
                         const char* bam_path);
int ps_clust_writer_feed(ps_clust_writer* w, const ps_read_batch* host_batch, uint64_t first_ordinal,
                         const ps_cluster* closed, uint64_t n_closed, const ps_site* sites, int has_open,
                         uint64_t open_first_read);
/* end of the run: the last cluster is never flushed (:528-529); writes .report / sitefrequency / sitepositions and
 * closes every file.  totals: skipped_due_indel and double_stranded of the whole run are used. */
int ps_clust_writer_finish(ps_clust_writer* w, const ps_pileup_counters* totals);
/* PS_ERR_REFERENCE_WOULD_THROW from ps_clust_writer_feed: the record on whose FASTA fetch the JVM would have died */
int ps_clust_writer_fault(const ps_clust_writer* w, ps_fault* out);
/* rows written so far; CCR windows that begin in front of their contig (anchor within 20 bases of its start: htsjdk
 * then reads file bytes in front of the contig -- not emulated, the window is written empty) */
void ps_clust_writer_stats(const ps_clust_writer* w, uint64_t* rows, uint64_t* ccr_rows, uint64_t* ccr_start_before_contig);
const char* ps_clust_writer_error(const ps_clust_writer* w);
void ps_clust_writer_close(ps_clust_writer* w);

/* ---- instrumentation ------------------------------------------------------------------------ */
/* number of kernels this context has launched since creation (bench.py "gpu_launches") */
uint64_t ps_kernel_launches(const ps_ctx* ctx);
/* device time (ms, CUDA events on the launching stream) of the last ps_*_batch_device call's dominant kernel */
float ps_last_kernel_ms(const ps_ctx* ctx);
/* device times (ms) of the dominant kernel of every ps_*_batch[_device] call since the last reset (a track call records
 * five stages: key pass and scans, segment placement, accumulation, coverage scans, selection), in call
 * order (at most 512 are kept); returns how many were written.  reset(enabled=0) switches the event pairs off. */
int ps_kernel_times(ps_ctx* ctx, float* ms, int max);
void ps_kernel_times_reset(ps_ctx* ctx, int enabled);
/* device times (ms) of the three kernels of the last pileup call: flag scan, cluster kernel, site compaction */
int ps_pileup_stage_times(ps_ctx* ctx, float* ms3);
/* 0: pileup calls on this context use the speculative boundary-flag pass (carry-in of a 2048-read tile = maximum over
 * the 128 reads in front of it, every assumption checked afterwards); 1: a check failed once (a record reaching over
 * more than 128 of its successors) and the context keeps to the exact look-back pass.  Results are identical either
 * way. */
int ps_pileup_flag_mode(const ps_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* PARASUITE_B200_H */
