// C ABI of libparasuite_b200.so: context, reference residency, error-profile entry points.
// (include/parasuite_b200.h documents which reference lines each call replaces.)
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "internal.h"

int set_error(ps_ctx* ctx, int status, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return status;
}
int cuda_fail(ps_ctx* ctx, cudaError_t e, const char* what) {
  std::string m = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  cudaGetLastError();
  return set_error(ctx, e == cudaErrorMemoryAllocation ? PS_ERR_OOM : PS_ERR_CUDA, m);
}

static DeviceBatch view_of(const ps_read_batch* b) {
  DeviceBatch v;
  v.n_reads = b->n_reads;
  v.meta = b->meta;
  v.ref_start = b->ref_start;
  v.bases2 = b->bases2;
  v.qual = b->qual;
  v.cigar = b->cigar;
  v.tile_base_off = b->tile_base_off;
  v.tile_qual_off = b->tile_qual_off;
  v.tile_cigar_off = b->tile_cigar_off;
  v.tile_exc_off = b->tile_exc_off;
  v.exc = b->exc;
  v.uniform_len = b->uniform_len;
  v.uniform_ncigar = b->uniform_ncigar;
  v.cigar_count = b->cigar_count;
  v.max_len = b->max_len;
  return v;
}

static int check_batch(ps_ctx* ctx, const ps_read_batch* b, bool allow_compact = false) {
  if (!b) return set_error(ctx, PS_ERR_INVALID_ARG, "batch is NULL");
  if (b->n_reads == 0) return PS_OK;
  const bool meta_ok = b->meta || (allow_compact && b->flags8 && b->uniform_len && b->uniform_ncigar);
  const bool cigar_ok = b->cigar || (allow_compact && b->uniform_cigar && b->uniform_ncigar == 1);
  const bool qual_ok = b->qual || (allow_compact && b->qual6 && b->uniform_len);
  const bool start_ok = b->ref_start || (allow_compact && b->start16 && b->tile_start);
  if (!meta_ok || !start_ok || !b->bases2 || !qual_ok || !cigar_ok || !b->tile_exc_off || !b->exc)
    return set_error(ctx, PS_ERR_INVALID_ARG, "batch has NULL streams");
  if ((!b->uniform_len && (!b->tile_base_off || !b->tile_qual_off)) || (!b->uniform_ncigar && !b->tile_cigar_off))
    return set_error(ctx, PS_ERR_INVALID_ARG, "variable-length batch without tile offsets");
  if (b->n_reads / PS_TILE_READS >= 0xFFFFFFFFull)
    return set_error(ctx, PS_ERR_INVALID_ARG, "batch too large (tile index is 32-bit)");
  return PS_OK;
}

// expansion of the compact host form (ps_read_batch: flags8, uniform_cigar) behind its upload
__global__ void expand_meta_kernel(const uint8_t* __restrict__ flags8, uint32_t len_ncig, uint32_t* __restrict__ meta, uint64_t n) {
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x)
    meta[r] = len_ncig | ((uint32_t)flags8[r] << 24);
}
// qualities packed 6 bits each (four per three bytes) -> one byte each, rows of L bytes
__global__ void unpack_qual6_kernel(const uint8_t* __restrict__ q6, uint8_t* __restrict__ qual, uint64_t n, uint32_t L) {
  const uint32_t gpr = (L + 3) / 4;
  const uint64_t total = n * gpr;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = g / gpr;
    const uint32_t j = (uint32_t)(g - r * gpr);
    const uint8_t* p = q6 + g * 3;
    const uint32_t w = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
    uint8_t* o = qual + r * L + 4u * j;
    const uint32_t v = (w & 63u) | (((w >> 6) & 63u) << 8) | (((w >> 12) & 63u) << 16) | (((w >> 18) & 63u) << 24);
    const uint32_t left = L - 4u * j;
    if (left >= 4u && (reinterpret_cast<uintptr_t>(o) & 3u) == 0) *reinterpret_cast<uint32_t*>(o) = v;
    else
      for (uint32_t k = 0; k < left && k < 4u; ++k) o[k] = (uint8_t)(v >> (8u * k));
  }
}
__global__ void expand_start_kernel(const uint16_t* __restrict__ start16, const uint32_t* __restrict__ tile_start,
                                    uint32_t* __restrict__ ref_start, uint64_t n) {
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x)
    ref_start[r] = tile_start[r / PS_TILE_READS] + start16[r];
}
__global__ void fill_u32_kernel(uint32_t* __restrict__ out, uint32_t v, uint64_t n) {
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) out[r] = v;
}

// H2D copy of a host batch into one of the two staging slots (async on ctx->stream)
int stage_batch(ps_ctx* ctx, const ps_read_batch* hb, bool with_qual, StagedBatch** out) {
  const int slot = ctx->staged_next;
  ctx->staged_next ^= 1;
  ctx->stage_serial++;
  StagedBatch& s = ctx->staged[slot];
  // the slot may still be read by a kernel queued two batches ago: same stream, so ordering is implicit
  const uint64_t n = hb->n_reads;
  const uint64_t nt = (n + PS_TILE_READS - 1) / PS_TILE_READS;
  struct Item { DevBuf* d; const void* h; size_t bytes; };
  // qualities last: they are more than half of the bytes and only the profile kernel reads them
  const bool compact_meta = hb->meta == nullptr, compact_cigar = hb->cigar == nullptr;
  const bool packed_qual = with_qual && hb->qual == nullptr;
  const bool compact_start = hb->ref_start == nullptr;
  if (compact_start && !(hb->start16 && hb->tile_start))
    return set_error(ctx, PS_ERR_INVALID_ARG, "batch has a NULL ref_start stream without start16 / tile_start");
  if ((compact_meta && !(hb->flags8 && hb->uniform_len && hb->uniform_ncigar)) ||
      (compact_cigar && !(hb->uniform_cigar && hb->uniform_ncigar == 1)) || (packed_qual && !(hb->qual6 && hb->uniform_len)))
    return set_error(ctx, PS_ERR_INVALID_ARG, "batch has NULL meta / cigar / qual streams without the compact form that replaces them");
  const size_t q6_bytes = packed_qual ? (size_t)n * ((hb->uniform_len + 3) / 4) * 3 : 0;
  Item items[] = {
      {&s.meta, hb->meta, n * 4},
      {&s.flags8, compact_meta ? hb->flags8 : nullptr, compact_meta ? (size_t)n : 0},
      {&s.ref_start, hb->ref_start, n * 4},
      {&s.start16, compact_start ? hb->start16 : nullptr, compact_start ? (size_t)n * 2 : 0},
      {&s.tile_start, compact_start ? hb->tile_start : nullptr, compact_start ? (size_t)nt * 4 : 0},
      {&s.cigar, hb->cigar, (size_t)(compact_cigar ? n : hb->cigar_count) * 4},
      {&s.bases2, hb->bases2, (size_t)hb->bases_bytes},
      {&s.tbo, hb->tile_base_off, hb->tile_base_off ? (nt + 1) * 8 : 0},
      {&s.tqo, hb->tile_qual_off, hb->tile_qual_off ? (nt + 1) * 8 : 0},
      {&s.tco, hb->tile_cigar_off, hb->tile_cigar_off ? (nt + 1) * 8 : 0},
      {&s.teo, hb->tile_exc_off, (nt + 1) * 4},
      {&s.exc, hb->exc, (size_t)hb->exc_count * 4},
      {&s.qual, hb->qual, with_qual ? (size_t)hb->qual_bytes : 0},   // the pileup never reads qualities
      {&s.qual6, packed_qual ? hb->qual6 : nullptr, q6_bytes},
  };
  if (!ctx->staged_core[slot]) cudaEventCreateWithFlags(&ctx->staged_core[slot], cudaEventDisableTiming);
  for (auto& it : items) {
    PS_CUDA(ctx, it.d->reserve(it.bytes + 64));   // +64: kernels may read a few bytes past the last read
    if (it.d == &s.qual) {
      // everything the pileup reads is on its way: expand the compact streams, then mark the point
      const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 8);
      if (compact_meta) {
        expand_meta_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<const uint8_t*>(s.flags8.p),
                                                           PS_MAKE_META(hb->uniform_len, hb->uniform_ncigar, 0),
                                                           static_cast<uint32_t*>(s.meta.p), n);
        ctx->launches++;
      }
      if (compact_cigar) {
        fill_u32_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<uint32_t*>(s.cigar.p), hb->uniform_cigar, n);
        ctx->launches++;
      }
      if (compact_start) {
        expand_start_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<const uint16_t*>(s.start16.p),
                                                            static_cast<const uint32_t*>(s.tile_start.p),
                                                            static_cast<uint32_t*>(s.ref_start.p), n);
        ctx->launches++;
      }
      if (compact_meta || compact_cigar || compact_start) PS_CUDA(ctx, cudaGetLastError());
      cudaEventRecord(ctx->staged_core[slot], ctx->stream);
    }
    if (it.bytes && it.h) PS_CUDA(ctx, cudaMemcpyAsync(it.d->p, it.h, it.bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (packed_qual) {
    const unsigned grid = (unsigned)std::min<uint64_t>((n * ((hb->uniform_len + 3) / 4) + 255) / 256, (uint64_t)ctx->sm_count * 16);
    unpack_qual6_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<const uint8_t*>(s.qual6.p), static_cast<uint8_t*>(s.qual.p), n,
                                                        hb->uniform_len);
    ctx->launches++;
    PS_CUDA(ctx, cudaGetLastError());
  }
  if (!ctx->staged_done[slot]) cudaEventCreateWithFlags(&ctx->staged_done[slot], cudaEventDisableTiming);
  cudaEventRecord(ctx->staged_done[slot], ctx->stream);   // host buffers of this batch may be reused once it has fired
  DeviceBatch& v = s.view;
  v.n_reads = n;
  v.meta = (const uint32_t*)s.meta.p;
  v.ref_start = (const uint32_t*)s.ref_start.p;
  v.bases2 = (const uint8_t*)s.bases2.p;
  v.qual = (const uint8_t*)s.qual.p;
  v.cigar = (const uint32_t*)s.cigar.p;
  v.tile_base_off = hb->tile_base_off ? (const uint64_t*)s.tbo.p : nullptr;
  v.tile_qual_off = hb->tile_qual_off ? (const uint64_t*)s.tqo.p : nullptr;
  v.tile_cigar_off = hb->tile_cigar_off ? (const uint64_t*)s.tco.p : nullptr;
  v.tile_exc_off = (const uint32_t*)s.teo.p;
  v.exc = (const uint32_t*)s.exc.p;
  v.uniform_len = hb->uniform_len;
  v.uniform_ncigar = hb->uniform_ncigar;
  v.cigar_count = compact_cigar ? n : hb->cigar_count;
  v.max_len = hb->max_len;
  *out = &s;
  return PS_OK;
}

void timer_begin(ps_ctx* ctx, cudaStream_t st) {
  if (!ctx->timers_on || ctx->ev_count >= PS_TIMER_RING) return;
  cudaEventRecord(ctx->ev_start[ctx->ev_count], st);
}
void timer_end(ps_ctx* ctx, cudaStream_t st) {
  if (!ctx->timers_on || ctx->ev_count >= PS_TIMER_RING) return;
  cudaEventRecord(ctx->ev_stop[ctx->ev_count], st);
  ctx->ev_count++;
}

// ---- reference: contig table and contig order -----------------------------------------------------
// Contig order of the pileup keys: by_rank[k] = FASTA index of the k-th contig (a permutation of 0 .. n_contigs-1).
// The table is read by kernels queued on any stream of the device: everything queued before is waited for, so none of
// them sees a half-written table.
static int upload_contig_order(ps_ctx* ctx, std::vector<uint32_t>&& by_rank) {
  const uint32_t n = (uint32_t)by_rank.size();
  std::vector<uint32_t> rank(n);
  for (uint32_t k = 0; k < n; ++k) rank[by_rank[k]] = k;
  PS_CUDA(ctx, cudaDeviceSynchronize());
  PS_CUDA(ctx, ctx->ref_rank.reserve((size_t)n * 4));
  PS_CUDA(ctx, cudaMemcpy(ctx->ref_rank.p, rank.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
  ctx->ref.contig_rank = (const uint32_t*)ctx->ref_rank.p;
  ctx->contig_rank.swap(rank);
  ctx->contig_by_rank.swap(by_rank);
  return PS_OK;
}

static int set_contigs(ps_ctx* ctx, const uint64_t* host_contig_off, uint32_t n_contigs, uint64_t n_bases) {
  if (!host_contig_off || n_contigs == 0) return set_error(ctx, PS_ERR_INVALID_ARG, "reference without contigs");
  if (n_bases >= (1ull << 32)) return set_error(ctx, PS_ERR_UNSUPPORTED, "reference >= 2^32 bases");
  ctx->contig_off.assign(host_contig_off, host_contig_off + n_contigs + 1);
  if (ctx->contig_off.back() != n_bases) return set_error(ctx, PS_ERR_INVALID_ARG, "contig table does not sum to n_bases");
  PS_CUDA(ctx, ctx->ref_contig.reserve((n_contigs + 1) * 8));
  PS_CUDA(ctx, cudaMemcpy(ctx->ref_contig.p, host_contig_off, (n_contigs + 1) * 8, cudaMemcpyHostToDevice));
  ctx->ref.contig_off = (const uint64_t*)ctx->ref_contig.p;
  ctx->ref.n_contigs = n_contigs;
  ctx->ref.n_bases = n_bases;
  std::vector<uint32_t> fasta_order(n_contigs);
  for (uint32_t c = 0; c < n_contigs; ++c) fasta_order[c] = c;
  return upload_contig_order(ctx, std::move(fasta_order));
}

int set_contig_order(ps_ctx* ctx, const uint32_t* order, uint32_t n) {
  cudaSetDevice(ctx->device);
  const uint32_t nc = ctx->ref.n_contigs;
  if (n > nc) return set_error(ctx, PS_ERR_INVALID_ARG, "contig order lists more contigs than the reference has");
  if (n && !order) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL contig order");
  std::vector<uint32_t> by_rank;
  by_rank.reserve(nc);
  std::vector<char> listed(nc, 0);
  for (uint32_t k = 0; k < n; ++k) {
    if (order[k] >= nc) return set_error(ctx, PS_ERR_INVALID_ARG, "contig order names a contig the reference lacks");
    if (listed[order[k]]) return set_error(ctx, PS_ERR_INVALID_ARG, "contig order lists a contig twice");
    listed[order[k]] = 1;
    by_rank.push_back(order[k]);
  }
  for (uint32_t c = 0; c < nc; ++c)      // contigs not listed follow, in FASTA order
    if (!listed[c]) by_rank.push_back(c);
  return upload_contig_order(ctx, std::move(by_rank));
}

extern "C" {

int ps_abi_version(void) { return PS_ABI_VERSION; }

const char* ps_strerror(int status) {
  switch (status) {
    case PS_OK: return "ok";
    case PS_ERR_INVALID_ARG: return "invalid argument";
    case PS_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
    case PS_ERR_CUDA: return "CUDA error";
    case PS_ERR_OOM: return "out of device memory";
    case PS_ERR_IO: return "I/O error";
    case PS_ERR_FORMAT: return "malformed input file";
    case PS_ERR_UNSORTED: return "BAM file is not sorted. Please provide a sorted BAM-file as input alignment file.";
    case PS_ERR_REFERENCE_WOULD_THROW: return "the reference implementation would die with an uncaught exception on this input";
    case PS_ERR_STATE: return "call order violated";
    case PS_ERR_UNSUPPORTED: return "unsupported";
  }
  return "unknown status";
}

int ps_create(ps_ctx** out, int device) {
  if (!out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device < 0 || device >= n) {
    cudaGetLastError();
    return PS_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PS_ERR_NO_DEVICE;
  if (prop.major != 10) return PS_ERR_NO_DEVICE;   // kernels are built for sm_100a only
  if (cudaSetDevice(device) != cudaSuccess) return PS_ERR_NO_DEVICE;
  ps_ctx* ctx = new ps_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("PARASUITE_B200_COMPACT_LOOKBACK")) ctx->pl_compact_lookback = e[0] == '1';
  if (const char* e = getenv("PARASUITE_B200_FLAG_SCAN_KERNEL")) ctx->pl_flag_scan_kernel = e[0] == '1';
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return PS_ERR_CUDA; }
  if (cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); ctx->stream2 = nullptr; }
  if (cudaStreamCreateWithFlags(&ctx->stream_rb, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); ctx->stream_rb = nullptr; }
  if (cudaEventCreateWithFlags(&ctx->prof_done_ev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); ctx->prof_done_ev = nullptr; }
  for (int i = 0; i < PS_TIMER_RING; ++i) {
    cudaEventCreate(&ctx->ev_start[i]);
    cudaEventCreate(&ctx->ev_stop[i]);
  }
  for (auto& e : ctx->pl_ev) cudaEventCreate(&e);
  cudaEventCreateWithFlags(&ctx->reset_ev, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->early_ev, cudaEventDisableTiming);
  if (cudaHostAlloc(&ctx->h_pinned, 4096, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); ctx->h_pinned = nullptr; }
  {   // result buffers are stream-ordered allocations: keep freed blocks in the pool instead of returning them to the OS
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  *out = ctx;
  return PS_OK;
}

void ps_destroy(ps_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < PS_TIMER_RING; ++i) {
    cudaEventDestroy(ctx->ev_start[i]);
    cudaEventDestroy(ctx->ev_stop[i]);
  }
  for (auto& e : ctx->pl_ev) cudaEventDestroy(e);
  cudaEventDestroy(ctx->reset_ev);
  if (ctx->early_ev) cudaEventDestroy(ctx->early_ev);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  if (ctx->h_acc) cudaFreeHost(ctx->h_acc);
  if (ctx->fasta && !ctx->fasta_shared) ps_fasta_free(ctx->fasta);
  for (auto& e : ctx->staged_done) if (e) cudaEventDestroy(e);
  for (auto& e : ctx->staged_core) if (e) cudaEventDestroy(e);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->stream_rb) cudaStreamDestroy(ctx->stream_rb);
  if (ctx->prof_done_ev) cudaEventDestroy(ctx->prof_done_ev);
  ctx->ref_seq2.release(); ctx->ref_inv.release(); ctx->ref_contig.release(); ctx->ref_rank.release();
  ctx->acc.release(); ctx->fault.release(); ctx->deferred.release(); ctx->t2c_mask.release();
  ctx->rg_okmap.release(); ctx->rg_off.release(); ctx->rg_bases.release(); ctx->rg_qual.release(); ctx->rg_op0.release();
  for (auto& s : ctx->staged) {
    s.meta.release(); s.ref_start.release(); s.bases2.release(); s.qual.release(); s.cigar.release();
    s.tbo.release(); s.tqo.release(); s.tco.release(); s.teo.release(); s.exc.release(); s.flags8.release(); s.qual6.release(); s.start16.release(); s.tile_start.release();
  }
  for (auto& b : ctx->pl_scratch) b.release();
  for (auto& b : ctx->tr_scratch) b.release();
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* ps_last_error(const ps_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

// ---- reference ---------------------------------------------------------------------------------------
int ps_reference_upload(ps_ctx* ctx, const ps_reference* r) {
  if (!ctx || !r || !r->seq2 || !r->inv) return set_error(ctx, PS_ERR_INVALID_ARG, "bad reference");
  cudaSetDevice(ctx->device);
  int st = set_contigs(ctx, r->contig_off, r->n_contigs, r->n_bases);
  if (st) return st;
  size_t b2 = ((r->n_bases + 15) / 16 + 4) * 4, b1 = ((r->n_bases + 31) / 32 + 4) * 4;
  PS_CUDA(ctx, ctx->ref_seq2.reserve(b2));
  PS_CUDA(ctx, ctx->ref_inv.reserve(b1));
  PS_CUDA(ctx, cudaMemcpy(ctx->ref_seq2.p, r->seq2, b2, cudaMemcpyHostToDevice));
  PS_CUDA(ctx, cudaMemcpy(ctx->ref_inv.p, r->inv, b1, cudaMemcpyHostToDevice));
  ctx->ref.seq2 = (const uint32_t*)ctx->ref_seq2.p;
  ctx->ref.inv = (const uint32_t*)ctx->ref_inv.p;
  ctx->ref_loaded = true;
  return PS_OK;
}

int ps_reference_set_contig_order(ps_ctx* ctx, const uint32_t* order, uint32_t n) {
  if (!ctx) return PS_ERR_INVALID_ARG;
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  if (ctx->pl_pending) return set_error(ctx, PS_ERR_STATE, "a submitted pileup call of this context has not been waited for");
  cudaSetDevice(ctx->device);
  return set_contig_order(ctx, order, n);
}

int ps_reference_adopt_device(ps_ctx* ctx, const ps_reference* r, const uint64_t* host_contig_off) {
  if (!ctx || !r || !r->seq2 || !r->inv) return set_error(ctx, PS_ERR_INVALID_ARG, "bad reference");
  cudaSetDevice(ctx->device);
  int st = set_contigs(ctx, host_contig_off, r->n_contigs, r->n_bases);
  if (st) return st;
  ctx->ref.seq2 = r->seq2;
  ctx->ref.inv = r->inv;
  ctx->ref_loaded = true;
  return PS_OK;
}

// ---- error profile -----------------------------------------------------------------------------------
size_t ps_profile_acc_len(uint32_t max_read_length, uint32_t infer_qualities) {
  return make_layout(max_read_length, infer_qualities).total;
}

// zero the accumulator vector, arm the fault word; kernels of the run may be queued on another stream: reset_ev orders
// them after the clearing
static cudaError_t clear_accumulators(ps_ctx* ctx, size_t acc_bytes, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(ctx->acc.p, 0, acc_bytes, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(ctx->fault.p, 0xFF, 8, s);
  if (e == cudaSuccess) e = cudaMemsetAsync((char*)ctx->fault.p + 8, 0, 56, s);
  if (e == cudaSuccess) e = cudaEventRecord(ctx->reset_ev, s);
  return e;
}

// accumulator + fault word -> page-locked host memory, queued on s
static cudaError_t queue_readback(ps_ctx* ctx, cudaStream_t s) {
  const size_t acc_bytes = (size_t)ctx->layout.total * 8;
  cudaError_t e = cudaMemcpyAsync(ctx->h_acc, ctx->acc.p, acc_bytes, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(static_cast<char*>(ctx->h_acc) + acc_bytes, ctx->fault.p, 8, cudaMemcpyDeviceToHost, s);
  return e;
}
constexpr size_t kEarlyReadbackMax = 64 << 10;   // with -q the vector holds a 256 x maxLen histogram: read back once, at the end

static void early_readback(ps_ctx* ctx, cudaStream_t s) {
  ctx->early_valid = false;
  if ((size_t)ctx->layout.total * 8 > kEarlyReadbackMax) return;
  // the copy goes to a stream of its own behind an event: on the kernels' stream it would sit between this tool's last
  // kernel and whatever the caller queues next (the pileup kernels), two stream-op boundaries on the critical path
  cudaStream_t rb = s;
  if (ctx->stream_rb && ctx->prof_done_ev && cudaEventRecord(ctx->prof_done_ev, s) == cudaSuccess &&
      cudaStreamWaitEvent(ctx->stream_rb, ctx->prof_done_ev, 0) == cudaSuccess)
    rb = ctx->stream_rb;
  if (queue_readback(ctx, rb) != cudaSuccess || cudaEventRecord(ctx->early_ev, rb) != cudaSuccess) { cudaGetLastError(); return; }
  ctx->early_valid = true;
  ctx->early_reads = ctx->reads_seen;
  ctx->early_stream = s;
}

int ps_profile_begin(ps_ctx* ctx, const ps_profile_opts* opts) {
  if (!ctx || !opts) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  if (opts->max_read_length == 0 || opts->max_read_length > 3000)
    return set_error(ctx, PS_ERR_INVALID_ARG, "max_read_length must be in [1, 3000]");
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  ctx->layout = make_layout(opts->max_read_length, opts->infer_qualities ? 1 : 0);
  const size_t acc_bytes = (size_t)ctx->layout.total * 8;
  PS_CUDA(ctx, ctx->acc.reserve(acc_bytes));
  PS_CUDA(ctx, ctx->fault.reserve(64));
  if (!(ctx->clean_ptr == ctx->acc.p && ctx->clean_bytes >= acc_bytes)) {   // else: cleared behind the last read-back
    PS_CUDA(ctx, clear_accumulators(ctx, acc_bytes, ctx->stream));
  }
  ctx->clean_ptr = nullptr;
  ctx->clean_bytes = 0;
  if (ctx->h_acc_bytes < acc_bytes + 8) {     // page-locked landing buffer: accumulator followed by the fault word
    if (ctx->h_acc) cudaFreeHost(ctx->h_acc);
    ctx->h_acc = nullptr; ctx->h_acc_bytes = 0;
    PS_CUDA(ctx, cudaHostAlloc(&ctx->h_acc, acc_bytes + 8, cudaHostAllocDefault));
    ctx->h_acc_bytes = acc_bytes + 8;
  }
  ctx->early_valid = false;
  ctx->emit_masks = opts->emit_t2c_masks != 0;
  ctx->t2c_mask_n = 0;
  ctx->profile_stream = nullptr;
  ctx->reads_seen = 0;
  ctx->profile_batches = 0;
  ctx->profile_open = true;
  return PS_OK;
}

int ps_profile_batch_device(ps_ctx* ctx, const ps_read_batch* b, void* stream) {
  if (!ctx) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  int st = check_batch(ctx, b);
  if (st) return st;
  cudaSetDevice(ctx->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
  PS_CUDA(ctx, cudaStreamWaitEvent(s, ctx->reset_ev, 0));     // the clearing may have been queued on another stream
  // a batch in a staging slot of this context (ps_batch_upload) run on a caller's stream: wait for its upload
  for (int slot = 0; slot < 2; ++slot)
    if (s != ctx->stream && b->n_reads && b->meta == ctx->staged[slot].view.meta && ctx->staged_done[slot])
      PS_CUDA(ctx, cudaStreamWaitEvent(s, ctx->staged_done[slot], 0));
  ctx->profile_stream = s;
  unsigned long long* masks = nullptr;
  ctx->t2c_mask_n = 0;
  if (ctx->emit_masks && b->n_reads) {
    PS_CUDA(ctx, ctx->t2c_mask.reserve((size_t)b->n_reads * 8));
    masks = static_cast<unsigned long long*>(ctx->t2c_mask.p);
  }
  bool written = false;
  timer_begin(ctx, s);
  PS_CUDA(ctx, launch_profile(ctx, view_of(b), ctx->reads_seen, s, masks, &written));
  timer_end(ctx, s);
  if (written) ctx->t2c_mask_n = b->n_reads;
  ctx->reads_seen += b->n_reads;
  early_readback(ctx, s);
  return PS_OK;
}

int ps_profile_batch(ps_ctx* ctx, const ps_read_batch* hb) {
  if (!ctx) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  int st = check_batch(ctx, hb, true);
  if (st) return st;
  if (hb->n_reads == 0) return PS_OK;
  cudaSetDevice(ctx->device);
  StagedBatch* sb = nullptr;
  st = stage_batch(ctx, hb, true, &sb);
  if (st) return st;
  PS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->reset_ev, 0));
  ctx->profile_stream = ctx->stream;
  timer_begin(ctx, ctx->stream);
  PS_CUDA(ctx, launch_profile(ctx, sb->view, ctx->reads_seen, ctx->stream));
  timer_end(ctx, ctx->stream);
  ctx->reads_seen += hb->n_reads;
  early_readback(ctx, ctx->stream);
  return PS_OK;
}

int ps_batch_upload(ps_ctx* ctx, const ps_read_batch* hb, ps_read_batch* dev_view) {
  if (!ctx || !dev_view) return PS_ERR_INVALID_ARG;
  int st = check_batch(ctx, hb, true);
  if (st) return st;
  cudaSetDevice(ctx->device);
  StagedBatch* sb = nullptr;
  st = stage_batch(ctx, hb, true, &sb);
  if (st) return st;
  *dev_view = *hb;
  const DeviceBatch& v = sb->view;
  dev_view->meta = v.meta; dev_view->ref_start = v.ref_start; dev_view->bases2 = v.bases2; dev_view->qual = v.qual;
  dev_view->cigar = v.cigar; dev_view->tile_base_off = v.tile_base_off; dev_view->tile_qual_off = v.tile_qual_off;
  dev_view->tile_cigar_off = v.tile_cigar_off; dev_view->tile_exc_off = v.tile_exc_off; dev_view->exc = v.exc;
  dev_view->cigar_count = v.cigar_count;
  dev_view->flags8 = nullptr;          // the view is always in the expanded form
  dev_view->qual6 = nullptr;
  dev_view->start16 = nullptr;
  dev_view->tile_start = nullptr;
  return PS_OK;
}

int ps_profile_masks_device(ps_ctx* ctx, const uint64_t** dev_masks, uint64_t* n_words) {
  if (!ctx || !dev_masks || !n_words) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  *dev_masks = ctx->t2c_mask_n ? static_cast<const uint64_t*>(ctx->t2c_mask.p) : nullptr;
  *n_words = ctx->t2c_mask_n;
  return PS_OK;
}

int ps_profile_acc_device(ps_ctx* ctx, void** dev_ptr, size_t* n_int64) {
  if (!ctx || !dev_ptr || !n_int64) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  *dev_ptr = ctx->acc.p;
  *n_int64 = ctx->layout.total;
  ctx->early_valid = false;      // the caller may change the vector (all-reduce): ps_profile_end reads it again
  return PS_OK;
}

int ps_profile_set_stream(ps_ctx* ctx, void* stream) {
  if (!ctx) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  ctx->profile_stream = stream ? (cudaStream_t)stream : ctx->stream;
  ctx->early_valid = false;
  return PS_OK;
}

}  // extern "C"

void profile_fill_result(const ProfileLayout& l, const int64_t* acc, ps_profile_result* out) {
  auto wrap = [](int64_t v) { return (int32_t)(uint32_t)(uint64_t)v; };   // Java int two's-complement wrap (Q8)
  const uint32_t m = l.max_len;
  if (out->position_conversions) for (uint32_t k = 0; k < 16 * m; ++k) out->position_conversions[k] = wrap(acc[l.conv + k]);
  if (out->quality_per_mismatch) for (int k = 0; k < 16; ++k) out->quality_per_mismatch[k] = wrap(acc[l.qsum + k]);
  if (out->quality_per_mismatch_counts) for (int k = 0; k < 16; ++k) out->quality_per_mismatch_counts[k] = wrap(acc[l.qcnt + k]);
  if (out->insertions_per_pos) for (uint32_t k = 0; k < m; ++k) out->insertions_per_pos[k] = (double)acc[l.ins + k];
  if (out->deletions_per_pos) for (uint32_t k = 0; k < m; ++k) out->deletions_per_pos[k] = (double)acc[l.del + k];
  if (out->counters) for (int k = 0; k < PS_PC_COUNT; ++k) out->counters[k] = wrap(acc[l.ctr + k]);
  if (out->quality_hist && l.infer_q) memcpy(out->quality_hist, &acc[l.qhist], (size_t)256 * m * 8);
  if (out->wide) memcpy(out->wide, acc, (size_t)l.total * 8);
}

extern "C" {

int ps_profile_end(ps_ctx* ctx, ps_profile_result* out) {
  if (!ctx || !out) return PS_ERR_INVALID_ARG;
  if (!ctx->profile_open) return set_error(ctx, PS_ERR_STATE, "ps_profile_begin not called");
  cudaSetDevice(ctx->device);
  const ProfileLayout& l = ctx->layout;
  const size_t acc_bytes = (size_t)l.total * 8;
  const int64_t* acc = static_cast<const int64_t*>(ctx->h_acc);
  // the last batch's stream (the context's or the caller's); earlier batches on other streams are the caller's to order
  cudaStream_t ps = ctx->profile_stream ? ctx->profile_stream : ctx->stream;
  if (ctx->early_valid && ctx->early_reads == ctx->reads_seen && ctx->early_stream == ps) {
    PS_CUDA(ctx, cudaEventSynchronize(ctx->early_ev));     // queued right behind the last batch's kernel
  } else {
    PS_CUDA(ctx, queue_readback(ctx, ps));
    PS_CUDA(ctx, cudaStreamSynchronize(ps));
  }
  ctx->early_valid = false;
  // clear for the next run now instead of in front of its first kernel.  Every producer of the vector has completed (the
  // host has just waited for the read-back that followed them), so the memsets need no place in the kernels' stream,
  // where they would sit between whatever the caller has queued there (the pileup kernels) and the next run
  if (clear_accumulators(ctx, acc_bytes, ctx->stream_rb ? ctx->stream_rb : ps) == cudaSuccess) { ctx->clean_ptr = ctx->acc.p; ctx->clean_bytes = acc_bytes; }
  else cudaGetLastError();
  unsigned long long fw;
  memcpy(&fw, static_cast<const char*>(ctx->h_acc) + acc_bytes, 8);
  ctx->profile_open = false;
  out->fault.code = 0;
  out->fault.read_ordinal = 0;
  if (fw != PS_FAULT_NONE) {
    out->fault.code = (int32_t)(fw & 0xFF);
    out->fault.read_ordinal = fw >> 8;
    char msg[160];
    if ((fw & 0xFF) == PS_FAULT_CIGAR_OPS) {
      snprintf(msg, sizeof msg, "record %llu has more than 255 CIGAR operations", (unsigned long long)(fw >> 8));
      return set_error(ctx, PS_ERR_UNSUPPORTED, msg);
    }
    snprintf(msg, sizeof msg, "record %llu: the JVM would die here (PS_THROW code %d)", (unsigned long long)(fw >> 8),
             (int)(fw & 0xFF));
    return set_error(ctx, PS_ERR_REFERENCE_WOULD_THROW, msg);
  }
  profile_fill_result(l, acc, out);
  return PS_OK;
}

// debug: words after the fault word ([1] = reads that took the fast path in the current run)
unsigned long long ps_debug_word(ps_ctx* ctx, int idx) {
  unsigned long long v = 0;
  if (!ctx || !ctx->fault.p || idx < 0 || idx > 7) return 0;
  cudaDeviceSynchronize();
  cudaMemcpy(&v, (char*)ctx->fault.p + 8 * idx, 8, cudaMemcpyDeviceToHost);
  return v;
}

// ---- instrumentation ---------------------------------------------------------------------------------
uint64_t ps_kernel_launches(const ps_ctx* ctx) { return ctx ? ctx->launches : 0; }

float ps_last_kernel_ms(const ps_ctx* ctx) {
  if (!ctx || ctx->ev_count == 0) return -1.f;
  float ms = -1.f;
  cudaEventSynchronize(ctx->ev_stop[ctx->ev_count - 1]);
  cudaEventElapsedTime(&ms, ctx->ev_start[ctx->ev_count - 1], ctx->ev_stop[ctx->ev_count - 1]);
  return ms;
}

int ps_kernel_times(ps_ctx* ctx, float* ms, int max) {
  if (!ctx || !ms) return PS_ERR_INVALID_ARG;
  int n = (int)ctx->ev_count < max ? (int)ctx->ev_count : max;
  for (int i = 0; i < n; ++i) {
    cudaEventSynchronize(ctx->ev_stop[i]);
    cudaEventElapsedTime(&ms[i], ctx->ev_start[i], ctx->ev_stop[i]);
  }
  return n;
}

int ps_pileup_stage_times(ps_ctx* ctx, float* ms3) {
  if (!ctx || !ms3) return PS_ERR_INVALID_ARG;
  if (!ctx->pl_ev_valid) return PS_ERR_STATE;
  cudaEventSynchronize(ctx->pl_ev[3]);
  for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&ms3[i], ctx->pl_ev[i], ctx->pl_ev[i + 1]);
  return PS_OK;
}

int ps_pileup_flag_mode(const ps_ctx* ctx) { return ctx && ctx->pl_exact_flags ? 1 : 0; }

void ps_kernel_times_reset(ps_ctx* ctx, int enabled) {
  if (!ctx) return;
  ctx->ev_count = 0;
  ctx->timers_on = enabled != 0;
}

}  // extern "C"
