// Internal declarations shared by the translation units of libparasuite_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include "parasuite_b200.h"
#include "record.h"

#define PS_BLOCK_THREADS 256   // == PS_TILE_READS: one read per thread, one tile per block iteration

// fault word kept on the device: min over (ordinal << 8 | code); ~0 = none
#define PS_FAULT_NONE 0xFFFFFFFFFFFFFFFFull

struct DeviceRef {
  const uint32_t* seq2 = nullptr;
  const uint32_t* inv = nullptr;
  const uint64_t* contig_off = nullptr;  // device copy
  const uint32_t* contig_rank = nullptr; // [n_contigs] position of each contig in the input's sort order (pileup keys)
  uint64_t n_bases = 0;
  uint32_t n_contigs = 0;
};

// device-side view of a batch (plain pointers, passed by value to kernels)
struct DeviceBatch {
  uint64_t n_reads;
  const uint32_t* meta;
  const uint32_t* ref_start;
  const uint8_t* bases2;
  const uint8_t* qual;
  const uint32_t* cigar;
  const uint64_t* tile_base_off;
  const uint64_t* tile_qual_off;
  const uint64_t* tile_cigar_off;
  const uint32_t* tile_exc_off;
  const uint32_t* exc;
  uint32_t uniform_len;
  uint32_t uniform_ncigar;
  uint64_t cigar_count;    // total cigar elements (0: not known)
  uint32_t max_len;        // longest read (0: not known)
  uint64_t past_end;       // ps_read_batch.past_end: the kernels never see it, the tools run on the reads before it
};

inline DeviceBatch view_of(const ps_read_batch* b) {
  DeviceBatch v;
  v.n_reads = b->n_reads; v.meta = b->meta; v.ref_start = b->ref_start; v.bases2 = b->bases2; v.qual = b->qual;
  v.cigar = b->cigar; v.tile_base_off = b->tile_base_off; v.tile_qual_off = b->tile_qual_off;
  v.tile_cigar_off = b->tile_cigar_off; v.tile_exc_off = b->tile_exc_off; v.exc = b->exc;
  v.uniform_len = b->uniform_len; v.uniform_ncigar = b->uniform_ncigar; v.cigar_count = b->cigar_count; v.max_len = b->max_len;
  v.past_end = b->past_end;
  return v;
}

struct ProfileLayout {   // offsets (in int64 elements) inside the accumulator vector
  uint32_t max_len;
  uint32_t infer_q;
  uint32_t conv, qsum, qcnt, ins, del, ctr, qhist, total;
};
inline ProfileLayout make_layout(uint32_t max_len, uint32_t infer_q) {
  ProfileLayout l;
  l.max_len = max_len;
  l.infer_q = infer_q;
  l.conv = 0;
  l.qsum = 16 * max_len;
  l.qcnt = l.qsum + 16;
  l.ins = l.qcnt + 16;
  l.del = l.ins + max_len;
  l.ctr = l.del + max_len;
  l.qhist = l.ctr + PS_PC_COUNT;
  l.total = l.qhist + (infer_q ? 256 * max_len : 0);
  return l;
}

// buffer that grows on demand
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct StagedBatch {   // device copy of a host batch
  DevBuf meta, ref_start, bases2, qual, cigar, tbo, tqo, tco, teo, exc, flags8, qual6, start16, tile_start;
  DevBuf sam_flags, mapq;   // the track's read filters (track_stage_aux)
  DeviceBatch view{};
};

#define PS_TIMER_RING 512

struct ps_packed_fasta;

struct ps_ctx {
  int device = 0;
  int sm_count = 148;
  std::string err;
  // reference
  DeviceRef ref;
  DevBuf ref_seq2, ref_inv, ref_contig, ref_rank;
  std::vector<uint64_t> contig_off;  // host copy
  // sort order of the input's contigs (ps_reference_set_contig_order): rank[c] = position of FASTA contig c in it,
  // by_rank = the inverse; identity after every reference upload.  ref.contig_rank is the device copy of `rank`.
  std::vector<uint32_t> contig_rank, contig_by_rank;
  bool ref_loaded = false;
  ps_packed_fasta* fasta = nullptr;   // set by ps_reference_load_fasta: contig names for BAM headers
  bool fasta_shared = false;          // the packed FASTA belongs to a ps_multi (several contexts share one)
  std::string fasta_path;             // raw-case FASTA for the clust output files (cluster sequence, CCR windows)
  // profile state
  bool profile_open = false;
  ProfileLayout layout{};
  DevBuf acc;        // int64[layout.total]
  DevBuf fault;      // uint64 fault word + debug / deferred-count words (64 bytes)
  DevBuf deferred;   // uint32 read indices the fast profile kernel hands to the generic routine
  DevBuf rg_okmap;                            // -q on the fast path: which reads the fast kernel counted
  DevBuf rg_off, rg_bases, rg_qual, rg_op0;   // ragged batches re-laid for the fast profile kernel (profile.cu: repack)
  uint64_t reads_seen = 0;
  uint32_t profile_batches = 0;   // fast-path batches of the open run (selects the deferred-read counter)
  cudaStream_t profile_stream = nullptr;   // stream of the last profile batch
  bool emit_masks = false;        // ps_profile_opts.emit_t2c_masks of the open run
  DevBuf t2c_mask;                // uint64 per read of the last device-resident fast-path batch
  uint64_t t2c_mask_n = 0;        // != 0: the words of that many reads are valid (or in flight on profile_stream)
  // streams / staging
  cudaStream_t stream = nullptr;
  StagedBatch staged[2];
  cudaEvent_t staged_done[2] = {nullptr, nullptr};
  cudaEvent_t staged_core[2] = {nullptr, nullptr};   // everything but the qualities of the slot's batch has arrived
  cudaStream_t stream2 = nullptr;                      // auxiliary stream: pileup of a batch whose qualities are still in flight
  cudaStream_t stream_rb = nullptr;                    // read-back of the profile accumulators behind the last batch's kernel
  cudaEvent_t prof_done_ev = nullptr;                  // that kernel's end, for stream_rb
  int staged_next = 0;
  uint64_t stage_serial = 0;   // uploads so far (a staged batch stays valid until the second-next one)
  // instrumentation
  uint64_t launches = 0;
  cudaEvent_t ev_start[PS_TIMER_RING];
  cudaEvent_t ev_stop[PS_TIMER_RING];
  uint32_t ev_count = 0;   // pairs recorded since reset
  bool timers_on = true;
  cudaEvent_t pl_ev[4] = {nullptr, nullptr, nullptr, nullptr};   // around the three pileup kernels of the last call
  // chained launches (launch_chained): the kernels of the resident step carry programmatic stream serialization unless
  // PARASUITE_B200_PDL=0 at ps_create.  No event may sit between chained kernels, so their timers are %globaltimer
  // stamps: ts_ring holds one stamp pair per timer slot (device_common.cuh: stamp_start / stamp_end), ev_stamped tells
  // which slots took stamps instead of events, cur_ts is the pair of the open slot (null: events or timers off)
  bool pdl = true;
  DevBuf ts_ring;
  bool ev_stamped[PS_TIMER_RING] = {};
  unsigned long long* cur_ts = nullptr;
  unsigned long long pl_ts[4] = {0, 0, 0, 0};   // stage stamps of the last pileup call (PlState::ts)
  bool pl_ts_valid = false;
  // occupancy, once per (kernel, dynamic shared memory) on this context's device (fn_blocks_per_sm)
  struct FnAttr { const void* fn; size_t smem; int per_sm; };
  std::vector<FnAttr> fn_attr;
  cudaEvent_t reset_ev = nullptr;   // accumulators of the current profile run have been cleared
  bool pl_ev_valid = false;
  void* h_pinned = nullptr;   // 4 KB of page-locked host memory for small read-backs
  void* h_acc = nullptr;      // page-locked landing buffer of the profile accumulator (ps_profile_end), grown on demand
  size_t h_acc_bytes = 0;
  // early read-back: every profile batch queues the copy of the (small) accumulator behind its kernel, so that
  // ps_profile_end usually finds it done; void once the caller took the device pointer (ps_profile_acc_device)
  cudaEvent_t early_ev = nullptr;
  uint64_t early_reads = 0;
  cudaStream_t early_stream = nullptr;
  bool early_valid = false;
  // ps_profile_end clears the accumulators for the next run behind its read-back: ps_profile_begin finds them clean
  const void* clean_ptr = nullptr;
  size_t clean_bytes = 0;
  // pileup scratch (pileup.cu): run state, look-back descriptors
  DevBuf pl_scratch[12];
  unsigned int pl_epoch = 0;    // look-back epoch (descriptors are never reset)
  uint64_t pl_cap_cl = 0, pl_cap_ev = 0;   // cluster-slot / site capacities learnt from earlier batches
  struct ps_pileup* pl_pending = nullptr;   // handle of a submitted pileup call that has not been waited for
  bool pl_flag_scan_kernel = false;   // PARASUITE_B200_FLAG_SCAN_KERNEL=1 at ps_create: always prefix the tile table with the one-block scan (tests)
  bool pl_compact_lookback = false;   // PARASUITE_B200_COMPACT_LOOKBACK=1 at ps_create: always order the site runs with the look-back (tests)
  bool pl_exact_flags = false;   // a speculative flag pass failed on this context: keep to the exact look-back kernel
  // track scratch (track.cu): run state, keys, scans, segments, position arrays, selections, records, dense head / tail,
  // base rows, indel rows
  DevBuf tr_scratch[14];
};

// ---- pileup handles over host-resident records (pileup.cu; used by the windowed file loops in tool_loops.cpp) --------
ps_pileup* pileup_host_handle(ps_ctx* ctx, std::vector<ps_cluster>&& clusters, std::vector<ps_site>&& sites, bool has_open,
                              const ps_cluster& open, std::vector<ps_site>&& open_sites, int32_t open_cov_pos0,
                              std::vector<uint32_t>&& open_cov, const ps_pileup_counters& counters);
void pileup_set_fault(ps_pileup* h, const ps_fault& f);
// wrap the int64 accumulator vector of a profile run into the caller's arrays (ctx.cu; Java int wrap-around, Q8)
void profile_fill_result(const ProfileLayout& l, const int64_t* acc, ps_profile_result* out);

// sets the pileup key order of a context with a reference (ctx.cu; ps_reference_set_contig_order without the state checks)
int set_contig_order(ps_ctx* ctx, const uint32_t* order, uint32_t n);

// ---- pileup keys: (rank of the contig + 1) << 32 | alignment end, 0 = no kept record ------------------------------
// The running maximum of these keys is Java's (tempClusterChr, tempClusterEnd): a contig change is a larger key only when
// contigs come in the order `rank` describes (ps_reference_set_contig_order).  rank: ps_ctx::contig_rank.
inline uint64_t pileup_key(const std::vector<uint32_t>& rank, uint32_t contig, int32_t end) {
  return ((uint64_t)(rank[contig] + 1) << 32) | (uint32_t)end;
}
// inverse of pileup_key (key != 0); by_rank: ps_ctx::contig_by_rank
inline void pileup_key_decode(const std::vector<uint32_t>& by_rank, uint64_t key, uint32_t* contig, int32_t* end) {
  *contig = by_rank[(uint32_t)(key >> 32) - 1];
  *end = (int32_t)(uint32_t)key;
}

// ---- kernel launchers (defined in the .cu files) ----------------------------------------------------
// t2c_mask (optional): n_reads words; *mask_written tells whether the batch took the fast kernel, which fills them
cudaError_t launch_profile(ps_ctx* ctx, const DeviceBatch& b, uint64_t ordinal0, cudaStream_t stream,
                           unsigned long long* t2c_mask = nullptr, bool* mask_written = nullptr);

// Blocks of `threads` threads of kernel `fn` with `smem` bytes of dynamic shared memory that fit one SM, cached per
// context; the kernel's dynamic shared memory attribute is raised to at least `smem` on the context's device (one
// process-wide record per device and kernel: it is never lowered), so the launch path makes no such call again.
cudaError_t fn_blocks_per_sm(ps_ctx* ctx, const void* fn, int threads, size_t smem, int* per_sm);

// Launch of a kernel of the resident step (profile kernels, pileup kernels): with ctx->pdl it carries programmatic
// stream serialization, so the grid becomes resident while its predecessor drains (device_common.cuh: pdl_wait).
template <typename... KArgs, typename... Args>
cudaError_t launch_chained(const ps_ctx* ctx, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                           Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = ctx->pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// timed sections (ctx.cu): a pair of events, or for chained kernels the stamp pair ctx->cur_ts
void timer_begin(ps_ctx* ctx, cudaStream_t st);
void timer_begin_chained(ps_ctx* ctx, cudaStream_t st);
void timer_end(ps_ctx* ctx, cudaStream_t st);

int set_error(ps_ctx* ctx, int status, const std::string& msg);
int cuda_fail(ps_ctx* ctx, cudaError_t e, const char* what);
#define PS_CUDA(ctx, expr)                                   \
  do {                                                       \
    cudaError_t _e = (expr);                                 \
    if (_e != cudaSuccess) return cuda_fail(ctx, _e, #expr); \
  } while (0)
