// K4: per-position T>C conversion and coverage track, split by strand (tool `track`).  Not a port of a Java tool: the
// PAR-CLIP toolkit reports clusters only; this is the per-locus signal genome browsers, crosslink-site callers and
// conversion-rate models start from.
//
// Records: those the pileup's record loop keeps (pl_decode_generic, SURVEY P1) with the pileup's faults and ordinals,
// except that there is no 51-position limit (PS_THROW_MASK51 is never raised).  Positions follow a genomic walk of the
// CIGAR (M/=/X: read and reference, D/N: reference, I/S: read, H/P: nothing); BAM flag 0x10 puts a read on the minus
// track.  Every aligned base adds 1 to its strand's coverage; T>C events are counted in genome orientation (plus: ref T
// and read C, minus: ref A and read G) where the reference base is ACGTacgt and the read base is not in `exc`.
//
// Device layout -- nothing scales with the contig or genome length:
//   tr_read_kernel       per read: filters, faults, counters, key pair {(rank+1)<<32 | end, (rank+1)<<32 | start}
//   (CUB) max scan       of the key pairs: running maximum of the end (segments) and of the start (sortedness)
//   tr_segment_kernel    a kept read opens a SEGMENT when its contig changes or it starts more than one base past the
//                        running maximum end: every segment is followed by a position no read covers
//   (CUB) sum scan       of the segment flags = segment index of every read
//   tr_seg_bounds_kernel first read and maximum end of every segment
//   tr_seg_len_kernel    segment length + 1 slot for the -1 one past its end; (CUB) exclusive sum = compact base
//   tr_seg_place_kernel  compact index range that is reported (windowed file tool: head and tail stay dense)
//   tr_accum_kernel<NW, BC>  per read: +1/-1 per alignment block into one int32 difference array per strand, +1 per
//                        T>C event.  NW > 0: uniform length <= 64, one M/=/X op -- T>C bits found bit-parallel on the
//                        2-bit words of read and reference.  BC (base counts): also +1 per event -- a read base other
//                        than the reference base, or an N call -- into five uint32 counters (A C G T N, strand
//                        orientation) per position and strand, and the genome-wide matrix in block-shared counters
//   (CUB) sum scan       of each difference array = coverage (every segment's differences sum to zero)
//   (CUB) select         run starts / ends per strand, T>C sites; tr_emit_*_kernel turn them into records.  BC: a select
//                        of the (position, strand) items with >= min_events non-N events, then tr_base_rows_kernel
//                        (reference base, mask, min_coverage) and a select of the rows it kept
// Compact space: M = sum over segments of (span + 1) <= sum over kept reads of (reference span + 1).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "device_common.cuh"
#include "track.h"

void timer_begin(ps_ctx* ctx, cudaStream_t st);
void timer_end(ps_ctx* ctx, cudaStream_t st);
int stage_batch(ps_ctx* ctx, const ps_read_batch* hb, bool with_qual, StagedBatch** out);

namespace {

constexpr int TR_THREADS = 256;

struct TrState {
  unsigned long long fault;          // min over (ordinal << 8 | code)
  unsigned long long unmapped, skipped, counted, fast;
  unsigned long long aligned[2], t2c[2];
  unsigned long long blocks[2];      // alignment blocks: every run starts or ends at one of their 2 * blocks edges
  unsigned long long first_key;      // min start key over the kept reads (~0: none)
  unsigned long long lo, hi;         // reported compact range [lo, hi)
  unsigned int unsorted;
  unsigned long long bases[2][4][5]; // base counts: [strand][ref][read A C G T N], strand orientation
};

struct TrParams {
  DeviceBatch b;
  DeviceRef ref;
  TrState* st;
  ulonglong2* keys;                  // [n] {end key, start key}, 0 = not kept
  ulonglong2* scan;                  // [n] inclusive running maximum of keys
  uint32_t* flag;                    // [n] segment flag, then (scan) segment index + 1
  uint32_t* seg_g;                   // [segs] global offset of the segment's first base
  uint32_t* seg_end;                 // [segs] last base covered (1-based contig position), then the segment length
  uint32_t* seg_contig;              // [segs] FASTA index
  unsigned long long* seg_key;       // [segs] start key
  unsigned long long* seg_base;      // [segs] compact index of the first base
  int32_t* diff;                     // [2][M + 1]
  uint32_t* t2c;                     // [2][M]
  uint64_t M;
  unsigned long long prev_end;       // windowed: max end key over the earlier windows (0: none)
  int windowed;
  uint32_t* bc;                      // base counts: [2][5][M] events by read base A C G T N (strand orientation)
};

struct MaxPair {
  __device__ __forceinline__ ulonglong2 operator()(const ulonglong2& a, const ulonglong2& b) const {
    return make_ulonglong2(a.x > b.x ? a.x : b.x, a.y > b.y ? a.y : b.y);
  }
};

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
  return v;
}

// Filters and faults exactly as pl_decode_generic (and pl_key for skipped_due_indel), without the 51-position limit.
__global__ void __launch_bounds__(TR_THREADS) tr_read_kernel(const __grid_constant__ TrParams P) {
  ContigCache cc;
  unsigned long long n_unm = 0, n_skip = 0, n_cnt = 0, al[2] = {0, 0}, nb[2] = {0, 0}, first = ~0ull;
  const uint64_t n = P.b.n_reads;
  for (uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); q < n; q += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = q + (threadIdx.x & 31u);
    const bool in = r < n;
    const uint32_t meta = in ? __ldg(P.b.meta + r) : PS_MAKE_META(0, 0, PS_RF_UNMAPPED);
    const ReadOffsets off = warp_read_offsets(P.b, q, r, in, meta);    // warp-collective
    if (!in) continue;
    ulonglong2 key = make_ulonglong2(0ull, 0ull);
    const uint32_t flags = PS_META_FLAGS(meta), L = PS_META_LEN(meta), ncig = PS_META_NCIGAR(meta);
    const uint32_t* cig = P.b.cigar + off.cigar;
    do {
      if (flags & PS_RF_UNMAPPED) { ++n_unm; break; }
      if (flags & PS_RF_CIGAR_OVERFLOW) { raise_fault(&P.st->fault, r, PS_FAULT_CIGAR_OPS); break; }
      uint32_t R = 0, alen = 0, blk = 0;
      bool hasI = false, hasD = false, hasN = false;
      for (uint32_t e = 0; e < ncig; ++e) {
        const uint32_t c = __ldg(cig + e), op = c & 15u;
        hasI |= op == 1u; hasD |= op == 2u; hasN |= op == 3u;
        if (op_consumes_ref(op)) R += c >> 4;
        if (op_is_match(op)) { alen += c >> 4; ++blk; }
      }
      if ((hasI || hasD) && hasN) { ++n_skip; break; }
      if (flags & PS_RF_POS_ZERO) { raise_fault(&P.st->fault, r, PS_THROW_REF_RANGE); break; }
      const uint64_t g0 = __ldg(P.b.ref_start + r);
      if (!contig_lookup(P.ref, g0, cc)) { raise_fault(&P.st->fault, r, PS_THROW_REF_RANGE); break; }
      bool bad = false;
      int64_t rdp = 0, rfp = 0;
      for (uint32_t e = 0; e < ncig && !bad; ++e) {
        const uint32_t c = __ldg(cig + e), op = c & 15u;
        const int64_t len = c >> 4;
        if (op == 4u || op == 1u) rdp += len;
        else if (op == 2u || op == 3u) rfp += len;
        else if (op_is_match(op)) {
          if (rdp + len > (int64_t)L) { raise_fault(&P.st->fault, r, PS_THROW_BLOCK_RANGE); bad = true; }
          else if ((flags & PS_RF_REF_RANGE) || g0 + (uint64_t)(rfp + len) > cc.hi) {
            raise_fault(&P.st->fault, r, PS_THROW_REF_RANGE); bad = true;
          }
          rdp += len; rfp += len;
        }
      }
      if (bad) break;
      const int32_t start = (int32_t)(g0 - cc.lo) + 1, end = start + (int32_t)R - 1;
      const unsigned long long hi = (unsigned long long)(cc.rank + 1) << 32;
      key = make_ulonglong2(hi | (uint32_t)end, hi | (uint32_t)start);
      ++n_cnt;
      al[(flags & PS_RF_REVERSE) ? 1 : 0] += alen;
      nb[(flags & PS_RF_REVERSE) ? 1 : 0] += blk;
      first = key.y < first ? key.y : first;
    } while (false);
    P.keys[r] = key;
  }
  n_unm = warp_sum(n_unm); n_skip = warp_sum(n_skip); n_cnt = warp_sum(n_cnt);
  al[0] = warp_sum(al[0]); al[1] = warp_sum(al[1]); nb[0] = warp_sum(nb[0]); nb[1] = warp_sum(nb[1]);
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, first, d); first = o < first ? o : first; }
  if ((threadIdx.x & 31u) == 0) {
    if (n_unm) atomicAdd(&P.st->unmapped, n_unm);
    if (n_skip) atomicAdd(&P.st->skipped, n_skip);
    if (n_cnt) atomicAdd(&P.st->counted, n_cnt);
    if (al[0]) atomicAdd(&P.st->aligned[0], al[0]);
    if (al[1]) atomicAdd(&P.st->aligned[1], al[1]);
    if (nb[0]) atomicAdd(&P.st->blocks[0], nb[0]);
    if (nb[1]) atomicAdd(&P.st->blocks[1], nb[1]);
    if (first != ~0ull) atomicMin(&P.st->first_key, first);
  }
}

// segment flags; a start smaller than the running maximum start is unsorted input (contig backwards included)
__global__ void __launch_bounds__(TR_THREADS) tr_segment_kernel(const __grid_constant__ TrParams P) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.b.n_reads) return;
  const ulonglong2 k = P.keys[r];
  uint32_t f = 0;
  if (k.x) {
    const ulonglong2 p = r ? P.scan[r - 1] : make_ulonglong2(0ull, 0ull);
    if (p.y > k.y) P.st->unsorted = 1u;
    const int64_t start = (int64_t)(uint32_t)k.y, pend = (int64_t)(uint32_t)p.x;
    f = (p.x == 0 || (p.x >> 32) != (k.x >> 32) || pend + 1 < start) ? 1u : 0u;
  }
  P.flag[r] = f;
}

// P.flag now holds the inclusive count of segment flags: first read and maximum end of every segment
__global__ void __launch_bounds__(TR_THREADS) tr_seg_bounds_kernel(const __grid_constant__ TrParams P) {
  ContigCache cc;
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.b.n_reads) return;
  const ulonglong2 k = P.keys[r];
  if (!k.x) return;
  const uint32_t s = P.flag[r] - 1;
  const bool opens = r == 0 || P.flag[r - 1] != P.flag[r];
  if (opens) {
    const uint32_t g0 = __ldg(P.b.ref_start + r);
    contig_lookup(P.ref, (uint64_t)g0, cc);
    P.seg_g[s] = g0;
    P.seg_contig[s] = cc.idx;
    P.seg_key[s] = k.y;
  }
  atomicMax(P.seg_end + s, (uint32_t)k.x);
}

__global__ void tr_seg_len_kernel(const __grid_constant__ TrParams P, uint32_t n_segs) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segs) return;
  // slots: the bases [start, end] and one more for the -1 one past the end
  const uint32_t start = (uint32_t)P.seg_key[s];
  P.seg_end[s] = P.seg_end[s] + 2u - start;
  P.seg_base[s] = P.seg_end[s];
}

// reported compact range: positions after prev_end (windowed) and before the last kept start (windowed); first index of
// a segment whose keys are > bound (lo) or >= split (hi)
__global__ void tr_seg_place_kernel(const __grid_constant__ TrParams P, uint32_t n_segs, unsigned long long split) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segs) return;
  const unsigned long long k0 = P.seg_key[s], base = P.seg_base[s];
  const unsigned long long len = P.seg_end[s];      // the length by now
  auto first_at_least = [&](unsigned long long bound) -> unsigned long long {   // first slot with key >= bound
    if (bound <= k0) return base;
    if ((bound >> 32) != (k0 >> 32) || bound - k0 >= len) return ~0ull;
    return base + (bound - k0);
  };
  const unsigned long long lo = P.prev_end ? first_at_least(P.prev_end + 1) : base;
  const unsigned long long hi = first_at_least(split);
  if (lo != ~0ull) atomicMin(&P.st->lo, lo);
  if (hi != ~0ull) atomicMin(&P.st->hi, hi);
}

__device__ __forceinline__ uint32_t tr_even_bits(uint32_t c) {   // even bits of c -> low 16 bits
  c &= 0x55555555u;
  c = (c | (c >> 1)) & 0x33333333u;
  c = (c | (c >> 2)) & 0x0F0F0F0Fu;
  c = (c | (c >> 4)) & 0x00FF00FFu;
  c = (c | (c >> 8)) & 0x0000FFFFu;
  return c;
}

// general path: one read, any CIGAR
__device__ __noinline__ void tr_accum_generic(const TrParams& P, uint64_t r, uint32_t meta, uint64_t off_base,
                                              uint64_t off_cigar, int64_t to_compact, unsigned long long* ev) {
  const uint32_t flags = PS_META_FLAGS(meta), ncig = PS_META_NCIGAR(meta);
  const uint32_t* cig = P.b.cigar + off_cigar;
  const bool rev = flags & PS_RF_REVERSE, has_inv = flags & PS_RF_HAS_INVALID;
  const int s = rev ? 1 : 0;
  int32_t* diff = P.diff + (size_t)s * (P.M + 1);
  uint32_t* t2c = P.t2c + (size_t)s * P.M;
  const uint8_t* rb = P.b.bases2 + off_base;
  const uint64_t g0 = __ldg(P.b.ref_start + r);
  ExcRange ex{0, 0};
  if (has_inv) ex = read_exc_range(P.b, r / PS_TILE_READS, (uint32_t)(r % PS_TILE_READS));
  int64_t rdp = 0, rfp = 0;
  for (uint32_t e = 0; e < ncig; ++e) {
    const uint32_t c = __ldg(cig + e), op = c & 15u;
    const int64_t n = c >> 4;
    if (op == 4u || op == 1u) rdp += n;
    else if (op == 2u || op == 3u) rfp += n;
    else if (op_is_match(op)) {
      if (n) {
        const int64_t i0 = (int64_t)(g0 + (uint64_t)rfp) + to_compact;
        atomicAdd(diff + i0, 1);
        atomicAdd(diff + i0 + n, -1);
      }
      for (int64_t z = 0; z < n; ++z) {
        const uint64_t g = g0 + (uint64_t)(rfp + z);
        const uint32_t p = (uint32_t)(rdp + z);
        if (ref_invalid_at(P.ref, g)) continue;
        const uint32_t a = ref_code_at(P.ref, g), bb = read_code_at(rb, p);
        if (!(rev ? (a == 0u && bb == 2u) : (a == 3u && bb == 1u))) continue;
        if (has_inv && read_pos_invalid(P.b, ex, p)) continue;
        atomicAdd(t2c + ((int64_t)g + to_compact), 1u);
        ++ev[s];
      }
      rdp += n; rfp += n;
    }
  }
}

// base counts of one read, any CIGAR: an event per read base other than the reference base and per N call into P.bc,
// every counted base into the block's matrix `tb` ([2][4][5], shared)
__device__ __noinline__ void tr_bases_generic(const TrParams& P, uint64_t r, uint32_t meta, uint64_t off_base,
                                              uint64_t off_cigar, int64_t to_compact, unsigned long long* tb) {
  const uint32_t flags = PS_META_FLAGS(meta), ncig = PS_META_NCIGAR(meta);
  const uint32_t* cig = P.b.cigar + off_cigar;
  const bool rev = flags & PS_RF_REVERSE, has_inv = flags & PS_RF_HAS_INVALID;
  const int s = rev ? 1 : 0;
  const uint32_t flip = rev ? 3u : 0u;             // minus strand: complement (A0 <-> T3, C1 <-> G2)
  uint32_t* bc = P.bc + (size_t)s * 5 * P.M;
  tb += s * 20;
  const uint8_t* rb = P.b.bases2 + off_base;
  const uint64_t g0 = __ldg(P.b.ref_start + r);
  ExcRange ex{0, 0};
  if (has_inv) ex = read_exc_range(P.b, r / PS_TILE_READS, (uint32_t)(r % PS_TILE_READS));
  int64_t rdp = 0, rfp = 0;
  for (uint32_t e = 0; e < ncig; ++e) {
    const uint32_t c = __ldg(cig + e), op = c & 15u;
    const int64_t n = c >> 4;
    if (op == 4u || op == 1u) rdp += n;
    else if (op == 2u || op == 3u) rfp += n;
    else if (op_is_match(op)) {
      for (int64_t z = 0; z < n; ++z) {
        const uint64_t g = g0 + (uint64_t)(rfp + z);
        const uint32_t p = (uint32_t)(rdp + z);
        if (ref_invalid_at(P.ref, g)) continue;
        const uint32_t a = ref_code_at(P.ref, g) ^ flip;
        const uint32_t bb = (has_inv && read_pos_invalid(P.b, ex, p)) ? 4u : (read_code_at(rb, p) ^ flip);
        if (bb != a) atomicAdd(bc + (size_t)bb * P.M + (uint64_t)((int64_t)g + to_compact), 1u);
        atomicAdd(tb + a * 5 + bb, 1ull);
      }
      rdp += n; rfp += n;
    }
  }
}

// base counts of one read on the bit-parallel path: mismatches are (ref ^ read) folded to one bit per base, N calls the
// positions listed in `exc`; the matrix diagonal is one popcount per reference base minus its events and N calls
template <int NW>
__device__ __forceinline__ void tr_bases_fast(const TrParams& P, const uint32_t (&w)[NW + 1], const uint32_t (&bw)[NW + 1],
                                              uint32_t sh, uint32_t bsh, unsigned long long inv, uint32_t L, uint32_t meta,
                                              uint64_t r, int st, int64_t c0, unsigned long long* tb) {
  const unsigned long long valid = ~inv & (L >= 64 ? ~0ull : ((1ull << L) - 1ull));
  const unsigned long long nm = (PS_META_FLAGS(meta) & PS_RF_HAS_INVALID) ? (read_exc_mask64(P.b, r) & valid) : 0ull;
  const uint32_t flip = st ? 3u : 0u;
  uint32_t* bc = P.bc + (size_t)st * 5 * P.M + c0;
  tb += st * 20;
  unsigned long long lo = 0, hi = 0, mm = 0;
#pragma unroll
  for (int j = 0; j < NW; ++j) {
    const uint32_t rf = __funnelshift_r(w[j], w[j + 1], sh), rd = __funnelshift_r(bw[j], bw[j + 1], bsh), x = rf ^ rd;
    lo |= (unsigned long long)tr_even_bits(rf) << (16 * j);
    hi |= (unsigned long long)tr_even_bits(rf >> 1) << (16 * j);
    mm |= (unsigned long long)tr_even_bits(x | (x >> 1)) << (16 * j);
  }
  mm &= valid & ~nm;
#pragma unroll
  for (uint32_t c = 0; c < 4; ++c) {
    const unsigned long long rc = ((c & 2u) ? hi : ~hi) & ((c & 1u) ? lo : ~lo) & valid;
    const uint32_t all = (uint32_t)__popcll(rc), nn = (uint32_t)__popcll(rc & nm), ne = (uint32_t)__popcll(rc & mm);
    const uint32_t a = c ^ flip;
    if (all != nn + ne) atomicAdd(tb + a * 6, (unsigned long long)(all - nn - ne));      // [a][a]
    if (nn) atomicAdd(tb + a * 5 + 4, (unsigned long long)nn);
  }
#pragma unroll
  for (int j = 0; j < NW; ++j) {
    uint32_t me = (uint32_t)(mm >> (16 * j)) & 0xFFFFu;
    if (!me) continue;
    const uint32_t rf = __funnelshift_r(w[j], w[j + 1], sh), rd = __funnelshift_r(bw[j], bw[j + 1], bsh);
    while (me) {
      const int k = __ffs((int)me) - 1;
      me &= me - 1;
      const uint32_t a = ((rf >> (2 * k)) & 3u) ^ flip, b = ((rd >> (2 * k)) & 3u) ^ flip;
      atomicAdd(bc + (size_t)b * P.M + 16 * j + k, 1u);
      atomicAdd(tb + a * 5 + b, 1ull);
    }
  }
  for (unsigned long long q = nm; q;) {
    const int k = __ffsll((long long)q) - 1;
    q &= q - 1;
    atomicAdd(bc + 4 * P.M + k, 1u);
  }
}

// NW > 0: the batch has uniform length L <= 64 and one cigar op per read; reads whose op is M/=/X of length L take the
// bit-parallel path (the positions listed in `exc` are cleared from its event mask: the code stored there is arbitrary)
template <int NW, bool BC>
__global__ void __launch_bounds__(TR_THREADS) tr_accum_kernel(const __grid_constant__ TrParams P) {
  unsigned long long ev[2] = {0, 0}, fast = 0;
  unsigned long long* tb = nullptr;
  if constexpr (BC) {
    __shared__ unsigned long long sh_bases[40];
    for (int k = threadIdx.x; k < 40; k += blockDim.x) sh_bases[k] = 0;
    __syncthreads();
    tb = sh_bases;
  }
  const uint64_t n = P.b.n_reads;
  for (uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); q < n; q += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = q + (threadIdx.x & 31u);
    const bool in = r < n;
    const uint32_t meta = in ? __ldg(P.b.meta + r) : 0u;
    uint64_t obase = 0, ocig = 0;
    if constexpr (NW == 0) {
      const ReadOffsets off = warp_read_offsets(P.b, q, r, in, meta);   // warp-collective
      obase = off.base; ocig = off.cigar;
    } else {
      obase = r * (uint64_t)((P.b.uniform_len + 3) >> 2);
      ocig = r;
    }
    if (!in) continue;
    const ulonglong2 k = P.keys[r];
    if (!k.x) continue;
    const uint32_t s = P.flag[r] - 1;
    const int64_t to_compact = (int64_t)P.seg_base[s] - (int64_t)P.seg_g[s];
    if constexpr (NW > 0) {
      const uint32_t L = P.b.uniform_len, cg = __ldg(P.b.cigar + r);
      if (op_is_match(cg & 15u) && (cg >> 4) == L && PS_META_LEN(meta) == L) {
        const bool rev = PS_META_FLAGS(meta) & PS_RF_REVERSE;
        const int st = rev ? 1 : 0;
        const uint32_t g0 = __ldg(P.b.ref_start + r);
        const uint32_t* src = reinterpret_cast<const uint32_t*>(P.b.bases2 + (obase & ~3ull));
        const uint32_t bsh = (uint32_t)(obase & 3u) * 8u;
        uint32_t bw[NW + 1], w[NW + 1];
#pragma unroll
        for (int j = 0; j <= NW; ++j) { bw[j] = __ldg(src + j); w[j] = __ldg(P.ref.seq2 + (g0 >> 4) + j); }
        const uint32_t sh = (g0 & 15u) * 2u, ii = g0 >> 5, s1 = g0 & 31u;
        const uint32_t i0 = __ldg(P.ref.inv + ii), i1 = __ldg(P.ref.inv + ii + 1), i2 = NW > 2 ? __ldg(P.ref.inv + ii + 2) : 0u;
        unsigned long long m = 0;
#pragma unroll
        for (int j = 0; j < NW; ++j) {
          const uint32_t rf = __funnelshift_r(w[j], w[j + 1], sh);
          const uint32_t rd = __funnelshift_r(bw[j], bw[j + 1], bsh);
          // plus: ref T (11) and read C (01); minus: ref A (00) and read G (10)
          const uint32_t h = rev ? (~(rf | (rf >> 1)) & (rd >> 1) & ~rd) : (rf & (rf >> 1) & rd & ~(rd >> 1));
          m |= (unsigned long long)tr_even_bits(h) << (16 * j);
        }
        const unsigned long long inv = (unsigned long long)__funnelshift_r(i0, i1, s1) |
                                       ((unsigned long long)(NW > 2 ? __funnelshift_r(i1, i2, s1) : 0u) << 32);
        m &= ~inv;
        m &= L >= 64 ? ~0ull : ((1ull << L) - 1ull);
        if ((PS_META_FLAGS(meta) & PS_RF_HAS_INVALID) && m) m &= ~read_exc_mask64(P.b, r);   // only with a candidate event
        const int64_t c0 = (int64_t)g0 + to_compact;
        atomicAdd(P.diff + (size_t)st * (P.M + 1) + c0, 1);
        atomicAdd(P.diff + (size_t)st * (P.M + 1) + c0 + L, -1);
        uint32_t* t2c = P.t2c + (size_t)st * P.M + c0;
        ev[st] += (unsigned long long)__popcll(m);
        while (m) {
          const int j = __ffsll((long long)m) - 1;
          m &= m - 1;
          atomicAdd(t2c + j, 1u);
        }
        if constexpr (BC) tr_bases_fast<NW>(P, w, bw, sh, bsh, inv, L, meta, r, st, c0, tb);
        ++fast;
        continue;
      }
    }
    tr_accum_generic(P, r, meta, obase, ocig, to_compact, ev);
    if constexpr (BC) tr_bases_generic(P, r, meta, obase, ocig, to_compact, tb);
  }
  ev[0] = warp_sum(ev[0]); ev[1] = warp_sum(ev[1]); fast = warp_sum(fast);
  if ((threadIdx.x & 31u) == 0) {
    if (ev[0]) atomicAdd(&P.st->t2c[0], ev[0]);
    if (ev[1]) atomicAdd(&P.st->t2c[1], ev[1]);
    if (fast) atomicAdd(&P.st->fast, fast);
  }
  if constexpr (BC) {
    __syncthreads();
    for (int k = threadIdx.x; k < 40; k += blockDim.x)
      if (tb[k]) atomicAdd(&P.st->bases[0][0][0] + k, tb[k]);
  }
}

// ---- selection predicates over compact indices -------------------------------------------------------------------
struct RunStart {
  const int32_t* cov; unsigned long long lo;
  __device__ __forceinline__ bool operator()(const unsigned long long& i) const {
    const int32_t c = cov[i];
    return c != 0 && (i == lo || cov[i - 1] != c);
  }
};
struct RunEnd {
  const int32_t* cov; unsigned long long hi;
  __device__ __forceinline__ bool operator()(const unsigned long long& i) const {
    const int32_t c = cov[i];
    return c != 0 && (i + 1 == hi || cov[i + 1] != c);
  }
};
struct SiteAt {          // item 2*i + strand
  const uint32_t* t2c; uint64_t M;
  __device__ __forceinline__ bool operator()(const unsigned long long& k) const {
    return t2c[(k & 1ull) * M + (k >> 1)] != 0u;
  }
};

struct BaseCandidate {   // item 2*i + strand: at least min_ev events other than N calls, whatever their type
  const uint32_t* bc; uint64_t M; uint32_t min_ev;
  __device__ __forceinline__ bool operator()(const unsigned long long& k) const {
    const uint32_t* p = bc + (k & 1ull) * 5 * M + (k >> 1);
    return p[0] + p[M] + p[2 * M] + p[3 * M] >= min_ev;
  }
};
struct RowKept {
  __device__ __forceinline__ bool operator()(const ps_track_base_row& x) const { return x.cov != 0u; }
};

// segment of compact index i (seg_base ascending)
__device__ __forceinline__ uint32_t seg_of(const TrParams& P, uint32_t n_segs, unsigned long long i) {
  uint32_t lo = 0, hi = n_segs;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (P.seg_base[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ uint32_t pos0_of(const TrParams& P, uint32_t s, unsigned long long i) {
  return (uint32_t)P.seg_key[s] - 1u + (uint32_t)(i - P.seg_base[s]);
}

__global__ void tr_emit_runs_kernel(const __grid_constant__ TrParams P, uint32_t n_segs, const int32_t* cov,
                                    const unsigned long long* starts, const unsigned long long* ends, uint64_t n,
                                    ps_track_run* out) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const unsigned long long a = starts[k], b = ends[k];
  const uint32_t s = seg_of(P, n_segs, a);
  ps_track_run x;
  x.contig = P.seg_contig[s];
  x.start0 = pos0_of(P, s, a);
  x.end0 = pos0_of(P, s, b) + 1u;
  x.cov = (uint32_t)cov[a];
  out[k] = x;
}

__global__ void tr_emit_sites_kernel(const __grid_constant__ TrParams P, uint32_t n_segs, const unsigned long long* sel,
                                     uint64_t n, ps_track_site* out) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const unsigned long long it = sel[k], i = it >> 1;
  const uint32_t strand = (uint32_t)(it & 1ull);
  const uint32_t s = seg_of(P, n_segs, i);
  ps_track_site x;
  x.contig = P.seg_contig[s];
  x.pos = (int32_t)pos0_of(P, s, i) + 1;
  x.strand = strand;
  x.t2c = P.t2c[(size_t)strand * P.M + i];
  x.cov = (uint32_t)P.diff[(size_t)strand * (P.M + 1) + i];
  out[k] = x;
}

// one base row per candidate (the reference base, the mask and min_coverage decide); cov = 0: no row
__global__ void tr_base_rows_kernel(const __grid_constant__ TrParams P, uint32_t n_segs, const unsigned long long* cand,
                                    uint64_t n, TrackBases sel, ps_track_base_row* out) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const unsigned long long it = cand[k], i = it >> 1;
  const uint32_t strand = (uint32_t)(it & 1ull);
  const uint32_t s = seg_of(P, n_segs, i);
  const uint64_t g = (uint64_t)P.seg_g[s] + (i - P.seg_base[s]);
  ps_track_base_row x{};
  if (!ref_invalid_at(P.ref, g)) {
    const uint32_t a = ref_code_at(P.ref, g) ^ (strand ? 3u : 0u);
    const uint32_t cov = (uint32_t)P.diff[(size_t)strand * (P.M + 1) + i];
    uint32_t ev[5];
#pragma unroll
    for (int b = 0; b < 5; ++b) ev[b] = P.bc[((size_t)strand * 5 + b) * P.M + i];
    if (track_base_row(sel, a, cov, ev, x.n)) {
      x.contig = P.seg_contig[s];
      x.pos = (int32_t)pos0_of(P, s, i) + 1;
      x.strand = (uint8_t)strand;
      x.ref = (uint8_t)a;
      x.cov = cov;
    }
  }
  out[k] = x;
}

// dense copy of the positions [key0, key0 + len) (one contig) from the compact arrays: cov+, cov-, t2c+, t2c-, and with
// base counts (BC) the ten event counters
template <bool BC>
__global__ void tr_dense_kernel(const __grid_constant__ TrParams P, uint32_t n_segs, unsigned long long key0, uint32_t len,
                                uint32_t* out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= len) return;
  const unsigned long long key = key0 + k;
  uint32_t lo = 0, hi = n_segs;                    // last segment whose start key <= key
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (P.seg_key[mid] <= key) lo = mid; else hi = mid;
  }
  constexpr int NV = BC ? 14 : 4;
  uint32_t v[NV] = {};
  const unsigned long long k0 = P.seg_key[lo];
  if (key >= k0 && (key >> 32) == (k0 >> 32) && key - k0 < P.seg_end[lo]) {
    const unsigned long long i = P.seg_base[lo] + (key - k0);
    v[0] = (uint32_t)P.diff[i];
    v[1] = (uint32_t)P.diff[(P.M + 1) + i];
    v[2] = P.t2c[i];
    v[3] = P.t2c[P.M + i];
    if constexpr (BC) {
#pragma unroll
      for (int j = 4; j < NV; ++j) v[j] = P.bc[(size_t)(j - 4) * P.M + i];
    }
  }
#pragma unroll
  for (int j = 0; j < NV; ++j) out[(size_t)j * len + k] = v[j];
}

__global__ void tr_init_state(TrState* st) {
  st->fault = PS_FAULT_NONE; st->unmapped = 0; st->skipped = 0; st->counted = 0; st->fast = 0;
  st->aligned[0] = st->aligned[1] = 0; st->t2c[0] = st->t2c[1] = 0; st->blocks[0] = st->blocks[1] = 0;
  st->first_key = ~0ull; st->lo = ~0ull; st->hi = ~0ull; st->unsorted = 0;
}

// scratch of the track calls, kept by the context (ps_ctx::tr_scratch) and grown on demand: a call waits for the
// device before it returns, so the next call may reuse it
template <typename T>
T* slot(ps_ctx* ctx, int k, size_t count, cudaError_t& err) {
  if (err != cudaSuccess) return nullptr;
  err = ctx->tr_scratch[k].reserve(count * sizeof(T) + 64);
  return static_cast<T*>(ctx->tr_scratch[k].p);
}
constexpr int kTrCubSlot = 9;

template <typename F>
cudaError_t cub_call(ps_ctx* ctx, F&& f) {         // size query, temporary storage (one slot), run
  size_t bytes = 0;
  cudaError_t e = f(nullptr, bytes);
  if (e != cudaSuccess) return e;
  void* tmp = slot<uint8_t>(ctx, kTrCubSlot, bytes, e);
  if (e != cudaSuccess) return e;
  return f(tmp, bytes);
}

uint32_t grid_for(uint64_t n, int threads = TR_THREADS) { return (uint32_t)std::max<uint64_t>(1, (n + threads - 1) / threads); }

}  // namespace

#define TR_CUDA(expr)                                       \
  do {                                                      \
    cudaError_t _e = (expr);                                \
    if (_e != cudaSuccess) return cuda_fail(ctx, _e, #expr); \
  } while (0)

int track_bases_of(const ps_track_opts* o, TrackBases* out) {
  *out = TrackBases();
  if (!o) return PS_OK;
  if (o->substitutions >> 16) return PS_ERR_INVALID_ARG;
  out->on = o->base_counts != 0;
  out->min_cov = std::max<uint32_t>(1u, o->min_coverage);
  out->min_ev = std::max<uint32_t>(1u, o->min_events);
  out->mask = (o->substitutions ? o->substitutions : 0xFFFFu) & ~0x8421u;     // diagonal bits 4 * c + c cleared
  return PS_OK;
}

int track_run(ps_ctx* ctx, const DeviceBatch& b, cudaStream_t st, bool windowed, uint64_t prev_end, TrackOut* out,
              const TrackBases& bases) {
  if (b.past_end && b.past_end <= b.n_reads) {
    // a record past its contig's end: the reads before it decide whether an earlier record faults first
    DeviceBatch head = b;
    head.n_reads = b.past_end - 1;
    head.past_end = 0;
    const int rc = track_run(ctx, head, st, windowed, prev_end, out, bases);
    if (rc != PS_OK && rc != PS_ERR_UNSORTED) return rc;
    out->base_rows.clear();                // a faulting call reports no base rows
    out->totals = ps_track_base_totals{};
    out->ctr.num_reads_processed = b.n_reads;
    out->fault.code = PS_FAULT_PAST_END;
    out->fault.read_ordinal = b.past_end - 1;
    return set_error(ctx, PS_ERR_UNSUPPORTED, "track: a record with no reference span starts past its contig's end");
  }
  *out = TrackOut();
  out->bases_on = bases.on;
  const uint64_t n = b.n_reads;
  out->ctr.num_reads_processed = n;
  if (n == 0) return PS_OK;
  if (n >= 0xFFFFFFFFull) return set_error(ctx, PS_ERR_UNSUPPORTED, "track batch of >= 2^32 reads");
  cudaError_t err = cudaSuccess;
  TrState* d_st = slot<TrState>(ctx, 0, 1, err);
  TrParams P{};
  P.b = b; P.ref = ctx->ref; P.st = d_st; P.prev_end = windowed ? prev_end : 0; P.windowed = windowed;
  P.keys = slot<ulonglong2>(ctx, 1, n, err);
  P.scan = slot<ulonglong2>(ctx, 2, n, err);
  P.flag = slot<uint32_t>(ctx, 3, n, err);
  TR_CUDA(err);
  const uint32_t grid_g = (uint32_t)std::min<uint64_t>(grid_for(n), (uint64_t)ctx->sm_count * 8);
  timer_begin(ctx, st);
  tr_init_state<<<1, 1, 0, st>>>(d_st);
  if (bases.on) TR_CUDA(cudaMemsetAsync(d_st->bases, 0, sizeof d_st->bases, st));
  tr_read_kernel<<<grid_g, TR_THREADS, 0, st>>>(P);
  TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceScan::InclusiveScan(t, sz, P.keys, P.scan, MaxPair(), (int64_t)n, st); }));
  tr_segment_kernel<<<grid_for(n), TR_THREADS, 0, st>>>(P);
  TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceScan::InclusiveSum(t, sz, P.flag, P.flag, (int64_t)n, st); }));
  timer_end(ctx, st);
  ctx->launches += 5;
  // run state: faults decide before anything is allocated for the positions
  struct Head { TrState s; uint32_t n_segs; uint32_t pad; ulonglong2 total; } hh{};
  TR_CUDA(cudaMemcpyAsync(&hh.s, d_st, sizeof(TrState), cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaMemcpyAsync(&hh.n_segs, P.flag + n - 1, 4, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaMemcpyAsync(&hh.total, P.scan + n - 1, sizeof(ulonglong2), cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaStreamSynchronize(st));
  out->ctr.unmapped = hh.s.unmapped;
  out->ctr.skipped_due_indel = hh.s.skipped;
  out->ctr.reads_counted = hh.s.counted;
  out->ctr.aligned_bases[0] = hh.s.aligned[0];
  out->ctr.aligned_bases[1] = hh.s.aligned[1];
  if (hh.s.fault != PS_FAULT_NONE) {
    out->fault.code = (int32_t)(hh.s.fault & 0xFF);
    out->fault.read_ordinal = hh.s.fault >> 8;
    if (out->fault.code == PS_FAULT_CIGAR_OPS)
      return set_error(ctx, PS_ERR_UNSUPPORTED, "track: a record of this batch has more than 255 CIGAR operations");
    return set_error(ctx, PS_ERR_REFERENCE_WOULD_THROW, "track: the pileup would die on a record of this batch");
  }
  if (hh.s.unsorted) return set_error(ctx, PS_ERR_UNSORTED, ps_strerror(PS_ERR_UNSORTED));
  const uint32_t n_segs = hh.n_segs;
  // PARASUITE_B200_DEBUG: the shape of the call -- segments, compact size M, reported range [lo, hi), head and tail
  const bool dbg = getenv("PARASUITE_B200_DEBUG") != nullptr;
  auto print_shape = [&](uint64_t M, uint64_t reported) {
    if (dbg)
      fprintf(stderr, "[ps_track] segments %u, compact %llu, reported %llu, head %u, tail %u\n", n_segs,
              (unsigned long long)M, (unsigned long long)reported, out->head.len, out->tail.len);
  };
  if (n_segs == 0) { print_shape(0, 0); return PS_OK; }
  out->first_key = hh.s.first_key;
  out->last_key = hh.total.y;
  out->max_end_key = hh.total.x;

  P.seg_key = slot<unsigned long long>(ctx, 4, 4ull * n_segs, err);     // key, base, then three uint32 arrays
  TR_CUDA(err);
  P.seg_base = P.seg_key + n_segs;
  P.seg_g = reinterpret_cast<uint32_t*>(P.seg_base + n_segs);
  P.seg_end = P.seg_g + n_segs;
  P.seg_contig = P.seg_end + n_segs;
  timer_begin(ctx, st);
  TR_CUDA(cudaMemsetAsync(P.seg_end, 0, n_segs * 4ull, st));
  tr_seg_bounds_kernel<<<grid_for(n), TR_THREADS, 0, st>>>(P);
  tr_seg_len_kernel<<<grid_for(n_segs), TR_THREADS, 0, st>>>(P, n_segs);
  TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceScan::ExclusiveSum(t, sz, P.seg_base, P.seg_base, (int64_t)n_segs, st); }));
  const unsigned long long split = windowed ? hh.total.y : ~0ull;
  tr_seg_place_kernel<<<grid_for(n_segs), TR_THREADS, 0, st>>>(P, n_segs, split);
  timer_end(ctx, st);
  ctx->launches += 4;
  struct Place { unsigned long long base; uint32_t len; uint32_t pad; unsigned long long lo, hi; } hp{};
  TR_CUDA(cudaMemcpyAsync(&hp.base, P.seg_base + n_segs - 1, 8, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaMemcpyAsync(&hp.len, P.seg_end + n_segs - 1, 4, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaMemcpyAsync(&hp.lo, &d_st->lo, 16, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaStreamSynchronize(st));
  const uint64_t M = hp.base + hp.len;
  if (M >= (1ull << 31)) return set_error(ctx, PS_ERR_UNSUPPORTED, "track: the reads of one batch span more than 2^31 positions");
  const uint64_t lo = std::min<uint64_t>(hp.lo, M), hi = std::max<uint64_t>(lo, std::min<uint64_t>(hp.hi, M));
  P.M = M;
  // difference arrays / coverage, the T>C counts, then (base counts) the event counters
  P.diff = slot<int32_t>(ctx, 5, 4 * (M + 1) + (bases.on ? 10 * M : 0), err);
  TR_CUDA(err);
  P.t2c = reinterpret_cast<uint32_t*>(P.diff + 2 * (M + 1));
  P.bc = bases.on ? P.t2c + 2 * M : nullptr;
  timer_begin(ctx, st);
  TR_CUDA(cudaMemsetAsync(P.diff, 0, 2 * (M + 1) * 4, st));
  TR_CUDA(cudaMemsetAsync(P.t2c, 0, (bases.on ? 12 : 2) * M * 4, st));
  const uint32_t L = b.uniform_len;
  const int nw = (L >= 1 && L <= 64 && b.uniform_ncigar == 1 && (reinterpret_cast<uintptr_t>(b.bases2) & 3u) == 0) ? (int)((L + 15) / 16) : 0;
  if (!bases.on) {
    switch (nw) {
      case 1: tr_accum_kernel<1, false><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 2: tr_accum_kernel<2, false><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 3: tr_accum_kernel<3, false><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 4: tr_accum_kernel<4, false><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      default: tr_accum_kernel<0, false><<<grid_g, TR_THREADS, 0, st>>>(P); break;
    }
  } else {
    switch (nw) {
      case 1: tr_accum_kernel<1, true><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 2: tr_accum_kernel<2, true><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 3: tr_accum_kernel<3, true><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      case 4: tr_accum_kernel<4, true><<<grid_g, TR_THREADS, 0, st>>>(P); break;
      default: tr_accum_kernel<0, true><<<grid_g, TR_THREADS, 0, st>>>(P); break;
    }
  }
  timer_end(ctx, st);
  timer_begin(ctx, st);
  for (int s = 0; s < 2; ++s) {
    int32_t* d = P.diff + (size_t)s * (M + 1);
    TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceScan::InclusiveSum(t, sz, d, d, (int64_t)M, st); }));
  }
  timer_end(ctx, st);
  ctx->launches += 3;

  // selection of the reported range [lo, hi): at most 2 * blocks + 1 runs a strand (edges), at most one site a T>C event
  unsigned long long tot[3];
  TR_CUDA(cudaMemcpyAsync(tot, &d_st->fast, 8, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaMemcpyAsync(tot + 1, &d_st->t2c[0], 16, cudaMemcpyDeviceToHost, st));
  if (bases.on) TR_CUDA(cudaMemcpyAsync(out->totals.bases, d_st->bases, sizeof out->totals.bases, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaStreamSynchronize(st));
  out->ctr.fast_path_reads = tot[0];
  out->ctr.t2c_events[0] = tot[1];
  out->ctr.t2c_events[1] = tot[2];
  const uint64_t nr = hi - lo;
  const uint64_t cap_r[2] = {std::min<uint64_t>(nr, 2 * hh.s.blocks[0] + 1), std::min<uint64_t>(nr, 2 * hh.s.blocks[1] + 1)};
  const uint64_t cap_s = std::min<uint64_t>(2 * nr, tot[1] + tot[2]);
  // base-count candidates: at most one per min_ev events other than N calls
  uint64_t events = 0;
  if (bases.on)
    for (int s = 0; s < 2; ++s)
      for (int a = 0; a < 4; ++a)
        for (int c = 0; c < 4; ++c) events += a == c ? 0 : out->totals.bases[s][a][c];
  const uint64_t cap_c = std::min<uint64_t>(2 * nr, events / bases.min_ev);
  const uint64_t off_r[4] = {0, cap_r[0], 2 * cap_r[0], 2 * cap_r[0] + cap_r[1]}, off_s = 2 * (cap_r[0] + cap_r[1]);
  unsigned long long* sel = slot<unsigned long long>(ctx, 6, off_s + cap_s + cap_c + 8, err);
  TR_CUDA(err);
  unsigned long long* d_cnt = sel + off_s + cap_s + cap_c;      // runs (4), sites, candidates, base rows
  timer_begin(ctx, st);
  TR_CUDA(cudaMemsetAsync(d_cnt, 0, 7 * 8, st));
  thrust::counting_iterator<unsigned long long> it_pos(lo), it_site(2 * lo);
  for (int s = 0; s < 2 && nr; ++s) {
    const int32_t* cov = P.diff + (size_t)s * (M + 1);
    TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceSelect::If(t, sz, it_pos, sel + off_r[2 * s], d_cnt + 2 * s, (int64_t)nr, RunStart{cov, lo}, st); }));
    TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceSelect::If(t, sz, it_pos, sel + off_r[2 * s + 1], d_cnt + 2 * s + 1, (int64_t)nr, RunEnd{cov, hi}, st); }));
  }
  unsigned long long* sites_sel = sel + off_s;
  if (nr && cap_s) TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceSelect::If(t, sz, it_site, sites_sel, d_cnt + 4, (int64_t)(2 * nr), SiteAt{P.t2c, M}, st); }));
  unsigned long long* cand = sel + off_s + cap_s;
  if (nr && cap_c) TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceSelect::If(t, sz, it_site, cand, d_cnt + 5, (int64_t)(2 * nr), BaseCandidate{P.bc, M, bases.min_ev}, st); }));
  unsigned long long cnt[6] = {0, 0, 0, 0, 0, 0};
  TR_CUDA(cudaMemcpyAsync(cnt, d_cnt, (bases.on ? 6 : 5) * 8, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaStreamSynchronize(st));
  if (cnt[0] != cnt[1] || cnt[2] != cnt[3] || cnt[0] > cap_r[0] || cnt[2] > cap_r[1] || cnt[4] > cap_s || cnt[5] > cap_c)
    return set_error(ctx, PS_ERR_CUDA, "track: run or site selection out of bounds");
  ps_track_run* d_runs = slot<ps_track_run>(ctx, 7, cnt[0] + cnt[2] + 1, err);
  ps_track_site* d_sites = slot<ps_track_site>(ctx, 8, cnt[4] + 1, err);
  TR_CUDA(err);
  for (int s = 0; s < 2; ++s) {
    const uint64_t k = cnt[2 * s];
    if (!k) continue;
    tr_emit_runs_kernel<<<grid_for(k), TR_THREADS, 0, st>>>(P, n_segs, P.diff + (size_t)s * (M + 1), sel + off_r[2 * s],
                                                            sel + off_r[2 * s + 1], k, d_runs + (s ? cnt[0] : 0));
    ctx->launches++;
  }
  if (cnt[4]) { tr_emit_sites_kernel<<<grid_for(cnt[4]), TR_THREADS, 0, st>>>(P, n_segs, sites_sel, cnt[4], d_sites); ctx->launches++; }
  ps_track_base_row* d_rows = nullptr;             // [cnt[5]] one per candidate, then the kept ones
  if (cnt[5]) {
    d_rows = slot<ps_track_base_row>(ctx, 12, 2 * cnt[5], err);
    TR_CUDA(err);
    tr_base_rows_kernel<<<grid_for(cnt[5]), TR_THREADS, 0, st>>>(P, n_segs, cand, cnt[5], bases, d_rows);
    ctx->launches++;
    TR_CUDA(cub_call(ctx, [&](void* t, size_t& sz) { return cub::DeviceSelect::If(t, sz, d_rows, d_rows + cnt[5], d_cnt + 6, (int64_t)cnt[5], RowKept{}, st); }));
  }
  timer_end(ctx, st);
  // windowed: positions up to prev_end (head) and from the split on (tail) stay dense for the host merge
  uint32_t* d_dense[2] = {nullptr, nullptr};
  const uint32_t nv = bases.on ? 14 : 4;           // dense arrays a position hands over
  if (windowed) {
    const unsigned long long f = hh.s.first_key, E = hh.total.x;
    if (prev_end && (f >> 32) == (prev_end >> 32) && f <= prev_end) {
      out->head.key0 = f;
      out->head.len = (uint32_t)(prev_end - f + 1);
    }
    const unsigned long long t0 = std::max<unsigned long long>(split, prev_end + 1);
    if ((t0 >> 32) == (E >> 32) && t0 <= E) {
      out->tail.key0 = t0;
      out->tail.len = (uint32_t)(E - t0 + 1);
    }
    d_dense[0] = slot<uint32_t>(ctx, 10, (uint64_t)nv * out->head.len, err);
    d_dense[1] = slot<uint32_t>(ctx, 11, (uint64_t)nv * out->tail.len, err);
    TR_CUDA(err);
    TrackDense* dn[2] = {&out->head, &out->tail};
    for (int j = 0; j < 2; ++j) {
      if (!dn[j]->len) continue;
      if (bases.on) tr_dense_kernel<true><<<grid_for(dn[j]->len), TR_THREADS, 0, st>>>(P, n_segs, dn[j]->key0, dn[j]->len, d_dense[j]);
      else tr_dense_kernel<false><<<grid_for(dn[j]->len), TR_THREADS, 0, st>>>(P, n_segs, dn[j]->key0, dn[j]->len, d_dense[j]);
      ctx->launches++;
    }
  }
  ctx->launches += 5;
  TR_CUDA(cudaGetLastError());
  out->runs[0].resize(cnt[0]);
  out->runs[1].resize(cnt[2]);
  out->sites.resize(cnt[4]);
  if (cnt[0]) TR_CUDA(cudaMemcpyAsync(out->runs[0].data(), d_runs, cnt[0] * sizeof(ps_track_run), cudaMemcpyDeviceToHost, st));
  if (cnt[2]) TR_CUDA(cudaMemcpyAsync(out->runs[1].data(), d_runs + cnt[0], cnt[2] * sizeof(ps_track_run), cudaMemcpyDeviceToHost, st));
  if (cnt[4]) TR_CUDA(cudaMemcpyAsync(out->sites.data(), d_sites, cnt[4] * sizeof(ps_track_site), cudaMemcpyDeviceToHost, st));
  TrackDense* dn[2] = {&out->head, &out->tail};
  for (int j = 0; j < 2; ++j) {
    if (!dn[j]->len) continue;
    dn[j]->v.resize((uint64_t)nv * dn[j]->len);
    TR_CUDA(cudaMemcpyAsync(dn[j]->v.data(), d_dense[j], 4ull * nv * dn[j]->len, cudaMemcpyDeviceToHost, st));
  }
  unsigned long long n_rows = 0;
  if (cnt[5]) TR_CUDA(cudaMemcpyAsync(&n_rows, d_cnt + 6, 8, cudaMemcpyDeviceToHost, st));
  TR_CUDA(cudaStreamSynchronize(st));
  if (n_rows > cnt[5]) return set_error(ctx, PS_ERR_CUDA, "track: base row selection out of bounds");
  out->base_rows.resize(n_rows);
  if (n_rows) {
    TR_CUDA(cudaMemcpyAsync(out->base_rows.data(), d_rows + cnt[5], n_rows * sizeof(ps_track_base_row), cudaMemcpyDeviceToHost, st));
    TR_CUDA(cudaStreamSynchronize(st));
  }
  out->totals.n_rows = n_rows;
  out->ctr.n_runs[0] = cnt[0];
  out->ctr.n_runs[1] = cnt[2];
  out->ctr.n_sites = cnt[4];
  print_shape(M, nr);
  return PS_OK;
}

struct ps_track {
  TrackOut out;
};

static DeviceBatch tr_view_of(const ps_read_batch* b) {
  DeviceBatch v;
  v.n_reads = b->n_reads; v.meta = b->meta; v.ref_start = b->ref_start; v.bases2 = b->bases2; v.qual = b->qual;
  v.cigar = b->cigar; v.tile_base_off = b->tile_base_off; v.tile_qual_off = b->tile_qual_off;
  v.tile_cigar_off = b->tile_cigar_off; v.tile_exc_off = b->tile_exc_off; v.exc = b->exc;
  v.uniform_len = b->uniform_len; v.uniform_ncigar = b->uniform_ncigar; v.cigar_count = b->cigar_count; v.max_len = b->max_len;
  v.past_end = b->past_end;
  return v;
}

// a handle is returned with PS_OK and with a fault (PS_ERR_REFERENCE_WOULD_THROW, PS_ERR_UNSUPPORTED): ps_track_fault
static int track_call(ps_ctx* ctx, const DeviceBatch& v, cudaStream_t st, const TrackBases& bases, ps_track** out) {
  ps_track* h = new ps_track();
  const int rc = track_run(ctx, v, st, false, 0, &h->out, bases);
  if (rc == PS_OK || h->out.fault.code != 0) *out = h;
  else delete h;
  return rc;
}

extern "C" {

int ps_track_batch_device_ex(ps_ctx* ctx, const ps_read_batch* b, const ps_track_opts* opts, void* stream, ps_track** out) {
  if (!ctx || !b || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  TrackBases bases;
  if (track_bases_of(opts, &bases) != PS_OK) return set_error(ctx, PS_ERR_INVALID_ARG, "track: substitutions has bits above 15");
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  // a batch in a staging slot of this context: the track reads no qualities, so the core of the upload suffices
  for (int slot = 0; slot < 2; ++slot)
    if (st != ctx->stream && b->n_reads && b->meta == ctx->staged[slot].view.meta && ctx->staged_core[slot])
      cudaStreamWaitEvent(st, ctx->staged_core[slot], 0);
  return track_call(ctx, tr_view_of(b), st, bases, out);
}

int ps_track_batch_device(ps_ctx* ctx, const ps_read_batch* b, void* stream, ps_track** out) {
  return ps_track_batch_device_ex(ctx, b, nullptr, stream, out);
}

int ps_track_batch_ex(ps_ctx* ctx, const ps_read_batch* hb, const ps_track_opts* opts, ps_track** out) {
  if (!ctx || !hb || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  TrackBases bases;
  if (track_bases_of(opts, &bases) != PS_OK) return set_error(ctx, PS_ERR_INVALID_ARG, "track: substitutions has bits above 15");
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  if (hb->n_reads == 0) {
    *out = new ps_track();
    (*out)->out.ctr.num_reads_processed = 0;
    (*out)->out.bases_on = bases.on;
    return PS_OK;
  }
  StagedBatch* sb = nullptr;
  const int rc = stage_batch(ctx, hb, /*with_qual=*/false, &sb);
  if (rc) return rc;
  return track_call(ctx, sb->view, ctx->stream, bases, out);
}

int ps_track_batch(ps_ctx* ctx, const ps_read_batch* hb, ps_track** out) { return ps_track_batch_ex(ctx, hb, nullptr, out); }

int ps_track_counters_get(const ps_track* h, ps_track_counters* out) {
  if (!h || !out) return PS_ERR_INVALID_ARG;
  *out = h->out.ctr;
  return PS_OK;
}

int64_t ps_track_runs(const ps_track* h, int strand, uint64_t first, ps_track_run* runs, uint64_t max) {
  if (!h || (strand != 0 && strand != 1) || (!runs && max)) return PS_ERR_INVALID_ARG;
  const std::vector<ps_track_run>& v = h->out.runs[strand];
  if (first >= v.size()) return 0;
  const uint64_t k = std::min<uint64_t>(max, v.size() - first);
  if (k) std::memcpy(runs, v.data() + first, k * sizeof(ps_track_run));
  return (int64_t)k;
}

int64_t ps_track_sites(const ps_track* h, uint64_t first, ps_track_site* sites, uint64_t max) {
  if (!h || (!sites && max)) return PS_ERR_INVALID_ARG;
  const std::vector<ps_track_site>& v = h->out.sites;
  if (first >= v.size()) return 0;
  const uint64_t k = std::min<uint64_t>(max, v.size() - first);
  if (k) std::memcpy(sites, v.data() + first, k * sizeof(ps_track_site));
  return (int64_t)k;
}

int64_t ps_track_base_rows(const ps_track* h, uint64_t first, ps_track_base_row* rows, uint64_t max) {
  if (!h || (!rows && max)) return PS_ERR_INVALID_ARG;
  if (!h->out.bases_on) return PS_ERR_STATE;
  const std::vector<ps_track_base_row>& v = h->out.base_rows;
  if (first >= v.size()) return 0;
  const uint64_t k = std::min<uint64_t>(max, v.size() - first);
  if (k) std::memcpy(rows, v.data() + first, k * sizeof(ps_track_base_row));
  return (int64_t)k;
}

int ps_track_base_totals_get(const ps_track* h, ps_track_base_totals* out) {
  if (!h || !out) return PS_ERR_INVALID_ARG;
  if (!h->out.bases_on) return PS_ERR_STATE;
  *out = h->out.totals;
  return PS_OK;
}

int ps_track_fault(const ps_track* h, ps_fault* out) {
  if (!h || !out) return PS_ERR_INVALID_ARG;
  *out = h->out.fault;
  return PS_OK;
}

void ps_track_close(ps_track* h) { delete h; }

}  // extern "C"
