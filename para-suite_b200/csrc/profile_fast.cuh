// Fast path of the error-profile kernel (included by profile.cu inside its anonymous namespace).
//
// Shape: uniform read length L <= 64, one M cigar op per read (L == R) -- the PAR-CLIP case.
//
// Work unit = a WARP-tile of 64 consecutive reads (2 per lane).  Every warp runs its own 2-stage ring of
// cp.async.bulk (TMA) copies with its own mbarriers, so there is no block-wide barrier in the main loop.  The two reads
// of a lane are taken through ONE straight-line body (arrays of two, every phase unrolled over both), so the two
// dependency chains interleave; everything rare (N / IUPAC in the window or in the read, reads outside the shape) sits
// behind warp-uniform branches.  All per-base work is bit-parallel on 2-bit packed words:
//   match counts   per-thread bit-sliced ("vertical") counters over one-hot (A|C, G|T) x position lanes, merged
//                  across the warp with a carry-save butterfly every 2^P-2 reads (no atomics on the hot path)
//   quality sums   dp4a of the quality bytes against 0/-1 byte masks.  The masks come straight from the packed read
//                  codes: a PRMT whose two source operands are the same table word only looks at the low two bits of
//                  a selector nibble, so the raw code word selects the masks of positions 0,2,4,6 of an 8-position
//                  chunk and the word shifted by 2 those of positions 1,3,5,7; the quality bytes are put in the same
//                  even / odd order with one PRMT each.  Sums are by read base over ALL positions and corrected by the
//                  mismatch / invalid sums at the block flush.
//   mismatches     rare path, one at a time: the strand-oriented code words of a read are parked in shared memory, the
//                  loop body looks the event's pair up there and issues two native 32-bit shared reductions (count by
//                  position and pair, quality by pair); ref T / read C events also set a bit of the read's T>C mask
//   T>C mask       (optional output) one 64-bit word per read: bit i = conversion at index i of the strand-oriented
//                  read, bit 62 = minus strand, bit 63 = the word is valid (the read had the fast shape).  The pileup
//                  consumes it instead of decoding the read again (ps_profile_pileup_batch_device).
// Reads outside the shape (flags, other cigars, contig edges) are appended to a dense list for
// profile_deferred_kernel instead of being walked inline (one slow lane would stall the other 31).
//
// RG (ragged) instantiation: batches whose reads differ in length or cigar (what an aligner leaves of adapter-trimmed
// PAR-CLIP reads) are first re-laid by profile_repack_kernel into rows of S = 16 * ceil(max_read_length / 16) <= 64
// positions (bases and qualities zero-padded, first cigar op per read).  The kernel then runs with L = S as the row
// geometry and takes every length-dependent mask (read extent, reference-window extent, reversal shift, cigar shape)
// from the read's own length in its meta word; zero-padded qualities add nothing to the sums.

#define FAST_STAGES 2
#define WT_READS 64            // reads per warp-tile
#define FAST_THREADS 128
#define FAST_WARPS (FAST_THREADS / 32)
#ifndef FAST_BLOCKS_PER_SM
#define FAST_BLOCKS_PER_SM 4
#endif
// (the per-read-length instantiation runs 4 CTAs per SM up to 48-position rows -- 128 registers, no spills, 5 % faster
//  than 3 -- and 3 CTAs per SM with 64-position rows, where 4 measured 6 % slower)
#define FAST_QCOPIES 8         // copies of the per-pair mismatch quality cells (spreads same-address reductions)
#ifndef FAST_REV_SPLIT
#define FAST_REV_SPLIT 1       // test "any minus-strand read" per half of the warp-tile instead of once per tile
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine), completion signalled on the mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ int dp4a_ss(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp4a.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// shared-memory accesses by 32-bit shared address (no generic-to-shared conversion in the loops)
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ int lds_s8(uint32_t a) { int v; asm volatile("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void red_s32(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// prmt.b32, default mode: bits 2..0 of selector nibble n pick the source byte, bit 3 replicates its sign
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) {
  uint32_t r; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(s)); return r;
}
// one lane of the (converged) warp: code under this predicate runs with exactly one active thread, so the bulk-copy
// operands go to the uniform datapath without a uniformisation loop
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t n) {   // PTX shl: amounts >= 32 give 0
  uint32_t r; asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n)); return r;
}

struct FastStage {      // byte offsets inside one warp-stage buffer
  uint32_t meta, start, cigar, bases, qual, total;
};
__host__ __device__ inline FastStage fast_stage_layout(uint32_t L) {
  FastStage s;
  const uint32_t bpr = (L + 3) / 4;
  s.meta = 0;
  s.start = WT_READS * 4;
  s.cigar = 2 * WT_READS * 4;
  s.bases = 3 * WT_READS * 4;
  s.qual = s.bases + ((WT_READS * bpr + 15) & ~15u) + 16;   // +16: word reads may run past a row end
  s.total = (s.qual + WT_READS * L + 16 + 127) & ~127u;
  return s;
}

struct FastLayout {     // byte offsets of the block's shared memory
  uint32_t misc, zero, tbl, mm_cnt, mm_q, fast, warp0, warp_stride, inv, park, bars, stage0, total;
};
__host__ __device__ inline FastLayout fast_layout(uint32_t max_len, uint32_t L, uint32_t nw) {
  FastLayout f;
  f.misc = 0;                                   // u64[16]
  f.zero = 128;                                 // 96 zero bytes: the quality row of a read outside the shape
  f.tbl = 224;                                  // u32[4] PRMT tables: byte b of word b is 0xFF
  f.mm_cnt = 256;                               // u32[max_len*16] mismatch counts by position and pair
  f.mm_q = f.mm_cnt + max_len * 64;             // u32[16*FAST_QCOPIES] mismatch quality sums by pair
  f.fast = f.mm_q + 16 * FAST_QCOPIES * 4;      // u32[max_len*4] match counts by (position, base)
  f.warp0 = (f.fast + max_len * 16 + 127) & ~127u;
  f.bars = 0;                                   // per warp: u64[FAST_STAGES] (+pad to 32)
  f.inv = 32;                                   // per warp: u32[WT_READS*nw] N calls of the tile's reads
  f.park = f.inv + WT_READS * nw * 4;           // per warp: u32[2 reads][rf|rd][nw][32 lanes]
  f.stage0 = (f.park + 2 * 2 * nw * 32 * 4 + 127) & ~127u;
  f.warp_stride = f.stage0 + FAST_STAGES * fast_stage_layout(L).total;
  f.total = f.warp0 + FAST_WARPS * f.warp_stride;
  return f;
}

// bit-sliced counter: planes[p] holds bit p of 32 independent counters
template <int NPL>
__device__ __forceinline__ void vc_add2(uint32_t (&pl)[NPL], uint32_t x, uint32_t y) {
  uint32_t s = pl[0] ^ x ^ y;
  uint32_t c = (pl[0] & x) | (pl[0] & y) | (x & y);
  pl[0] = s;
#pragma unroll
  for (int p = 1; p < NPL; ++p) {
    const uint32_t t = pl[p] & c;
    pl[p] ^= c;
    c = t;
  }
}

template <int NPL>
struct Planes { uint32_t p[NPL]; };

// sum the bit-sliced counters of the 32 lanes; lane l ends up with the integer total of bit-lane l
// (passed by value so the caller's planes stay in registers across the call)
template <int NPL>
__device__ __noinline__ uint32_t vc_warp_total(Planes<NPL> pl) {
  uint32_t a[NPL + 5];
#pragma unroll
  for (int p = 0; p < NPL; ++p) a[p] = pl.p[p];
#pragma unroll
  for (int p = NPL; p < NPL + 5; ++p) a[p] = 0;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int np = NPL + s;   // planes holding data before this step
    uint32_t c = 0;
#pragma unroll
    for (int p = 0; p < NPL + 5; ++p) {
      if (p <= np) {
        const uint32_t b = p < np ? __shfl_xor_sync(0xFFFFFFFFu, a[p], 1 << s) : 0u;
        const uint32_t av = a[p];
        a[p] = av ^ b ^ c;
        c = (av & b) | (av & c) | (b & c);
      }
    }
  }
  const uint32_t lane = threadIdx.x & 31;
  uint32_t tot = 0;
#pragma unroll
  for (int p = 0; p < NPL + 5; ++p) tot |= ((a[p] >> lane) & 1u) << p;
  return tot;
}

// match count of base a at one position from the four counted lanes E0..E3 (see the one-hot words below)
__device__ __forceinline__ uint32_t fast_base_count(const uint32_t* e, uint32_t a) {
  const uint32_t e0 = e[0], e1 = e[1], e2 = e[2], e3 = e[3];
  return a == 0 ? e0 - e1 - e2 + e3 : (a == 1 ? e1 - e3 : (a == 2 ? e2 - e3 : e3));
}

// number of bit-sliced counter words for NW 2-bit words: (A|C) and (G|T) per word; when the last word holds at
// most 8 positions its two one-hot words share one counter word (A|C in the low half, G|T in the high half)
__host__ __device__ constexpr int fast_nc(int NW, int LT) {
  return (LT > 0 && LT - 16 * (NW - 1) <= 8) ? 2 * NW - 1 : 2 * NW;
}

// even bits of a 16-bit invalid map -> even bits of 32
__device__ __forceinline__ uint32_t fast_spread16(uint32_t h) {
  h &= 0xFFFFu;
  h = (h | (h << 8)) & 0x00FF00FFu;
  h = (h | (h << 4)) & 0x0F0F0F0Fu;
  h = (h | (h << 2)) & 0x33333333u;
  h = (h | (h << 1)) & 0x55555555u;
  return h;
}

// reverse the order of the L 2-bit groups held in NW words (groups keep their two bits in place) and complement them
// when CODES (A<->T, C<->G is a bitwise NOT); the result is masked to the read length
template <int NW, bool CODES>
__device__ __forceinline__ void fast_reverse(uint32_t (&v)[NW], uint32_t L, const uint32_t (&lenmask)[NW]) {
  const uint32_t s = 2u * (16u * NW - L);   // < 32
  uint32_t a[NW];
#pragma unroll
  for (int k = 0; k < NW; ++k) a[k] = __brev(v[NW - 1 - k]);
#pragma unroll
  for (int k = 0; k < NW; ++k) {
    const uint32_t an = k + 1 < NW ? a[k + 1] : 0u;
    const uint32_t x = __funnelshift_r(a[k], an, s);
    // brev swapped the two bits of every group: swap back
    const uint32_t y = ((x << 1) & 0xAAAAAAAAu) | ((x >> 1) & 0x55555555u);
    v[k] = (CODES ? ~y : y) & lenmask[k];
  }
}

// the same for a read of any length Lr <= 16 * NW: the shift may span whole words
template <int NW, bool CODES>
__device__ __forceinline__ void fast_reverse_any(uint32_t (&v)[NW], uint32_t Lr, const uint32_t (&lenmask)[NW]) {
  const uint32_t s = 2u * (16u * NW - Lr);   // < 32 * NW
  uint32_t a[NW + 1];
#pragma unroll
  for (int k = 0; k < NW; ++k) a[k] = __brev(v[NW - 1 - k]);
  a[NW] = 0u;
  if (NW > 2) {                              // whole-word part of the shift, two words then one
    const bool w2 = (s & 64u) != 0;
#pragma unroll
    for (int k = 0; k < NW; ++k) a[k] = w2 ? (k + 2 < NW ? a[k + 2 < NW ? k + 2 : 0] : 0u) : a[k];
  }
  if (NW > 1) {
    const bool w1 = (s & 32u) != 0;
#pragma unroll
    for (int k = 0; k < NW; ++k) a[k] = w1 ? a[k + 1] : a[k];
  }
#pragma unroll
  for (int k = 0; k < NW; ++k) {
    const uint32_t x = __funnelshift_r(a[k], a[k + 1], s & 31u);
    const uint32_t y = ((x << 1) & 0xAAAAAAAAu) | ((x >> 1) & 0x55555555u);
    v[k] = (CODES ? ~y : y) & lenmask[k];
  }
}

template <int NW, int NPL, int LT, bool RG>
__global__ void __launch_bounds__(FAST_THREADS, RG ? (NW <= 3 ? 4 : 3) : FAST_BLOCKS_PER_SM) profile_fast_kernel(const ProfileParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NC = fast_nc(NW, LT);
  constexpr uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t max_len = P.lay.max_len;
  const uint32_t L = LT > 0 ? (uint32_t)LT : P.b.uniform_len;
  const uint32_t bpr = (L + 3) >> 2;
  const FastStage lay = fast_stage_layout(L);
  const FastLayout fl = fast_layout(max_len, L, NW);
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* s_misc = reinterpret_cast<unsigned long long*>(smem_raw + fl.misc);
  // [0..3] sum of quality by read base over all positions, [4..7] same at invalid positions, [8] fast reads,
  // [12..15] mismatch quality by read base
  uint32_t* s_mm_cnt = reinterpret_cast<uint32_t*>(smem_raw + fl.mm_cnt);
  uint32_t* s_mm_q = reinterpret_cast<uint32_t*>(smem_raw + fl.mm_q);
  uint32_t* s_fast = reinterpret_cast<uint32_t*>(smem_raw + fl.fast);
  unsigned char* wbase = smem_raw + fl.warp0 + (size_t)warp * fl.warp_stride;
  uint32_t* s_inv = reinterpret_cast<uint32_t*>(wbase + fl.inv);        // [WT_READS][NW], zero between uses
  // 32-bit shared addresses of everything the loops touch
  const uint32_t a_smem = smem_u32(smem_raw);
  const uint32_t a_zero = a_smem + fl.zero;
  const uint32_t a_mm_cnt = a_smem + fl.mm_cnt;
  const uint32_t a_mm_q = a_smem + fl.mm_q + (lane & (FAST_QCOPIES - 1)) * 4;
  const uint32_t a_wbase = a_smem + fl.warp0 + warp * fl.warp_stride;
  const uint32_t a_bars = a_wbase + fl.bars;
  const uint32_t a_park = a_wbase + fl.park + lane * 4;                 // + ((h*2 + arr)*NW + k) * 128
  const uint32_t a_stage0 = a_wbase + fl.stage0;

  for (uint32_t k = threadIdx.x; k < fl.warp0 / 4; k += blockDim.x) reinterpret_cast<uint32_t*>(smem_raw)[k] = 0;
  for (uint32_t k = lane; k < WT_READS * NW; k += 32) s_inv[k] = 0;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < FAST_STAGES; ++s) mbar_init(reinterpret_cast<uint64_t*>(wbase + fl.bars) + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x < 4) sts32(a_smem + fl.tbl + threadIdx.x * 4, 0xFFu << (8 * threadIdx.x));
  __syncthreads();

  const uint64_t n_reads = P.b.n_reads;
  const uint32_t n_wt = P.n_tiles;                       // warp-tiles in the batch (the last may be partial)
  const uint32_t n_full = (uint32_t)(n_reads / WT_READS);
  const uint32_t gw = blockIdx.x * FAST_WARPS + warp;    // global warp id
  const uint32_t GW = gridDim.x * FAST_WARPS;
  auto issue = [&](uint32_t wt, uint32_t slot) {         // one lane only; partial tiles are staged by the warp itself
    if (wt >= n_full) return;
    const uint32_t dst = a_stage0 + slot * lay.total, bar = a_bars + slot * 8;
    const uint64_t r0 = (uint64_t)wt * WT_READS;
    const uint32_t bb = WT_READS * bpr, qb = WT_READS * L;
    mbar_expect_tx(bar, 3 * WT_READS * 4 + bb + qb);
    bulk_g2s(dst + lay.meta, P.b.meta + r0, WT_READS * 4, bar);
    bulk_g2s(dst + lay.start, P.b.ref_start + r0, WT_READS * 4, bar);
    bulk_g2s(dst + lay.cigar, P.b.cigar + r0, WT_READS * 4, bar);
    bulk_g2s(dst + lay.bases, P.b.bases2 + r0 * bpr, bb, bar);
    bulk_g2s(dst + lay.qual, P.b.qual + r0 * L, qb, bar);
  };
  if (elect_one()) {
#pragma unroll
    for (int s = 0; s < FAST_STAGES; ++s) {
      const uint32_t wt = gw + (uint32_t)s * GW;
      if (wt < n_wt) issue(wt, s);
    }
  }

  uint32_t lenmask[NW];
#pragma unroll
  for (int k = 0; k < NW; ++k) {
    const int rem = (int)L - 16 * k;
    lenmask[k] = rem >= 16 ? 0xFFFFFFFFu : (rem <= 0 ? 0u : ((1u << (2 * rem)) - 1u));
  }
  // PRMT tables (byte b = 0xFF) in vector registers: read back from shared memory so that they are no compile-time
  // constants, which would live in the uniform register file and cost a move at every use
  const uint32_t tbl1 = lds32(a_smem + fl.tbl + 4), tbl2 = lds32(a_smem + fl.tbl + 8), tbl3 = lds32(a_smem + fl.tbl + 12);
  const uint32_t ivmask0 = L >= 32 ? 0xFFFFFFFFu : ((1u << L) - 1u);
  const uint32_t ivmask1 = L > 32 ? (L >= 64 ? 0xFFFFFFFFu : ((1u << (L - 32)) - 1u)) : 0u;
  const uint32_t metaE = PS_MAKE_META(L, 1, 0), cgE = L << 4;      // the shape: length L, one op, L x M
  constexpr uint32_t kMetaMask = ~((uint32_t)(PS_RF_REVERSE | PS_RF_HAS_INVALID) << 24);
  const uint32_t Lcap = RG ? min(L, max_len) : L;                  // RG: longest read the rows and the histogram take

  Planes<NPL> pl[NC];
  uint32_t tot[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    tot[c] = 0;
#pragma unroll
    for (int p = 0; p < NPL; ++p) pl[c].p[p] = 0;
  }
  int qacc[4] = {0, 0, 0, 0}, qinv[4] = {0, 0, 0, 0};
  uint32_t n_fast = 0, since_flush = 0;
  constexpr uint32_t kFlushEvery = (1u << NPL) - 2u;   // reads a thread may add before a counter could overflow
  uint64_t c_lo = 1, c_hi = 0;                         // contig bounds cached from the previous warp-tile

  auto flush_vc = [&]() {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      tot[c] += vc_warp_total<NPL>(pl[c]);
#pragma unroll
      for (int p = 0; p < NPL; ++p) pl[c].p[p] = 0;
    }
    since_flush = 0;
    qacc[0] -= qacc[1] + qacc[2] + qacc[3];   // qacc[0] held the all-base total
#pragma unroll
    for (int b = 0; b < 4; ++b) {        // dp4a accumulated -q; keep the int32 far from overflow
      const int t = __reduce_add_sync(FULL, qacc[b]);
      const int u = __reduce_add_sync(FULL, qinv[b]);
      if (lane == 0 && t) atomicAdd(&s_misc[b], (unsigned long long)(long long)(-t));
      if (lane == 0 && u) atomicAdd(&s_misc[4 + b], (unsigned long long)(long long)u);
      qacc[b] = 0;
      qinv[b] = 0;
    }
  };

  // exception (N call) list of the first warp-tile's tile
  uint32_t e_lo = 0, e_hi = 0;
  if (gw < n_wt) { e_lo = __ldg(P.b.tile_exc_off + (gw >> 2)); e_hi = __ldg(P.b.tile_exc_off + (gw >> 2) + 1); }

  uint32_t it = 0;
  for (uint32_t wt = gw; wt < n_wt; wt += GW, ++it) {
    const uint32_t slot = it % FAST_STAGES;
    const uint32_t parity = (it / FAST_STAGES) & 1u;
    // this tile's N calls (issued before the wait so the latency overlaps it) and the next tile's list bounds
    const uint32_t ex = (e_lo + lane < e_hi) ? __ldg(P.b.exc + e_lo + lane) : 0xFFFFFFFFu;
    const uint32_t cur_lo = e_lo, cur_hi = e_hi;
    if (wt + GW < n_wt) {
      e_lo = __ldg(P.b.tile_exc_off + ((wt + GW) >> 2));
      e_hi = __ldg(P.b.tile_exc_off + ((wt + GW) >> 2) + 1);
    }
    const uint32_t a_sb = a_stage0 + slot * lay.total;
    unsigned char* sbw = wbase + fl.stage0 + (size_t)slot * lay.total;
    uint32_t n_here = WT_READS;
    if (wt < n_full) {
      mbar_wait(a_bars + slot * 8, parity);
    } else {   // the batch's last, partial warp-tile: bounds-checked cooperative copy instead of TMA
      const uint64_t r0 = (uint64_t)wt * WT_READS;
      n_here = (uint32_t)(n_reads - r0);
      uint32_t* d32 = reinterpret_cast<uint32_t*>(sbw);
      for (uint32_t k = lane; k < WT_READS; k += 32) {
        const bool in = k < n_here;
        d32[lay.meta / 4 + k] = in ? __ldg(P.b.meta + r0 + k) : 0u;
        d32[lay.start / 4 + k] = in ? __ldg(P.b.ref_start + r0 + k) : 0u;
        d32[lay.cigar / 4 + k] = in ? __ldg(P.b.cigar + r0 + k) : 0u;
      }
      const uint32_t* gb = reinterpret_cast<const uint32_t*>(P.b.bases2 + r0 * bpr);   // r0*bpr is a multiple of 64
      for (uint32_t k = lane; k < (n_here * bpr + 3) / 4; k += 32) d32[lay.bases / 4 + k] = __ldg(gb + k);
      const uint32_t* gq = reinterpret_cast<const uint32_t*>(P.b.qual + r0 * L);
      for (uint32_t k = lane; k < (n_here * L + 3) / 4; k += 32) d32[lay.qual / 4 + k] = __ldg(gq + k);
      __syncwarp();
    }
    // ---- record words and the reference window of this lane's two reads: requested first, so the loads are in flight
    //      while the warp looks at the contig bounds and the N calls.  The window offset is clamped to the reference, so
    //      the loads need no knowledge of the read's fate (a read outside the shape may carry any offset)
    uint32_t meta[2], g0[2], cg[2];
    uint32_t rw[2][NW + 1], ri[2][3], rsh[2];      // raw window words; funnel-shifted into place further down
    {
      const uint32_t g_last = (uint32_t)(P.ref.n_bases - 1);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t rit = lane + h * 32;
        meta[h] = lds32(a_sb + lay.meta + rit * 4);
        g0[h] = lds32(a_sb + lay.start + rit * 4);
        cg[h] = lds32(a_sb + lay.cigar + rit * 4);
        const uint32_t g = min(g0[h], g_last);
        rsh[h] = g & 31u;
#pragma unroll
        for (int k = 0; k <= NW; ++k) rw[h][k] = __ldg(P.ref.seq2 + (g >> 4) + k);
        ri[h][0] = __ldg(P.ref.inv + (g >> 5));
        ri[h][1] = __ldg(P.ref.inv + (g >> 5) + 1);
        ri[h][2] = (LT == 0 || LT > 32) ? __ldg(P.ref.inv + (g >> 5) + 2) : 0u;
      }
    }
    // contig bounds: reads starting and ending inside the contig of the tile's first read pass the range test
    {
      const uint64_t g = lds32(a_sb + lay.start);
      if (!(g >= c_lo && g < c_hi)) {
        if (g < P.ref.n_bases) {
          const uint32_t c = contig_of(P.ref, g);
          c_lo = __ldg(P.ref.contig_off + c);
          c_hi = __ldg(P.ref.contig_off + c + 1);
        } else { c_lo = 1; c_hi = 0; }
      }
    }
    // one unsigned compare per read: lo <= g0 and g0 + L <= hi  <=>  g0 - lo <= hi - lo - L  (offsets fit 32 bits)
    // (RG: span32 is the contig length and every read brings its own length to the test)
    const bool span_ok = RG ? c_hi > c_lo : (c_hi >= c_lo + L && L <= max_len);
    const uint32_t lo32 = (uint32_t)c_lo, span32 = span_ok ? (uint32_t)(c_hi - c_lo - (RG ? 0u : L)) : 0u;
    // scatter this warp-tile's N calls into the per-read invalid map
    if (cur_hi > cur_lo) {
      const uint32_t quarter = wt & 3u;
      uint32_t x = ex;
      for (uint32_t e = cur_lo; e < cur_hi; e += 32) {
        if (e != cur_lo) x = (e + lane < cur_hi) ? __ldg(P.b.exc + e + lane) : 0xFFFFFFFFu;
        if (x != 0xFFFFFFFFu && ((x >> 22) & 3u) == quarter) {
          const uint32_t rit = (x >> 16) & 63u, p = x & 0xFFFFu;
          const uint32_t mrit = lds32(a_sb + lay.meta + rit * 4);
          const uint32_t Lx = RG ? min(PS_META_LEN(mrit), L) : L;     // RG: rows hold the first L bases at most
          if (p < Lx) {
            atomicOr(&s_inv[rit * NW + (p >> 4)], 1u << (2u * (p & 15u)));
            // An N call is never counted, but the quality sums below run over ALL positions: clear the byte that pairs
            // with this base in the warp's copy of the qualities (index = distance from the 5' end: qualities are not
            // reversed with the bases, Q10), so that nothing has to be taken out again afterwards.
            const bool minus = (mrit & ((uint32_t)PS_RF_REVERSE << 24)) != 0;
            asm volatile("st.shared.u8 [%0], %1;" ::"r"(a_sb + lay.qual + rit * L + (minus ? Lx - 1u - p : p)), "r"(0u) : "memory");
          }
        }
      }
      __syncwarp();
    }

    // ================= the two reads of this lane, one straight-line body =======================================
    bool ok[2], rev[2], hasn[2], anyinv[2], punct[2];
    uint32_t rf[2][NW], iv[2][2], rd[2][NW], ve[2][NW];
    uint32_t a_qrow[2];
    uint32_t Lr[2], lm[2][RG ? NW : 1];          // RG: the read's own length and extent masks
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t rit = lane + h * 32;
#pragma unroll
      for (int k = 0; k < NW; ++k) rf[h][k] = __funnelshift_r(rw[h][k], rw[h][k + 1], (rsh[h] & 15u) * 2u);
      bool shaped;
      if (RG) {
        Lr[h] = PS_META_LEN(meta[h]);
        // one cigar op, no flag but strand / N calls, 1 <= Lr <= Lcap, the op is Lr x M
        shaped = (meta[h] & kMetaMask & 0xFFFF0000u) == (1u << 16) && Lr[h] - 1u < Lcap && cg[h] == (Lr[h] << 4);
        if (!shaped) Lr[h] = 1u;                    // keeps every shift below in range; the read adds nothing
#pragma unroll
        for (int k = 0; k < NW; ++k) {
          const int rem = min(max((int)Lr[h] - 16 * k, 0), 16);
          lm[h][k] = shl_clamp(1u, 2u * (uint32_t)rem) - 1u;        // rem == 16: shl by 32 gives 0, minus one = all ones
        }
        iv[h][0] = __funnelshift_r(ri[h][0], ri[h][1], rsh[h]) & (shl_clamp(1u, Lr[h]) - 1u);
        iv[h][1] = Lr[h] > 32u ? (__funnelshift_r(ri[h][1], ri[h][2], rsh[h]) & (shl_clamp(1u, Lr[h] - 32u) - 1u)) : 0u;
        // lo <= g0 and g0 + Lr <= hi with 32-bit offsets: d = g0 - lo may wrap to a huge value, which fails d <= span
        const uint32_t d = g0[h] - lo32;
        ok[h] = shaped && span_ok && d <= span32 && Lr[h] <= span32 - d && rit < n_here;
      } else {
        Lr[h] = L;
        iv[h][0] = __funnelshift_r(ri[h][0], ri[h][1], rsh[h]) & ivmask0;
        iv[h][1] = (LT == 0 || LT > 32) ? (__funnelshift_r(ri[h][1], ri[h][2], rsh[h]) & ivmask1) : 0u;
        shaped = ((meta[h] ^ metaE) & kMetaMask) == 0 && cg[h] == cgE;
        ok[h] = shaped && (g0[h] - lo32) <= span32 && span_ok && rit < n_here;
      }
      rev[h] = ok[h] && (meta[h] & ((uint32_t)PS_RF_REVERSE << 24)) != 0;
      hasn[h] = (meta[h] & ((uint32_t)PS_RF_HAS_INVALID << 24)) != 0 && rit < n_here;
      anyinv[h] = ok[h] && (iv[h][0] | iv[h][1]) != 0;
      punct[h] = anyinv[h];
      // ---- read codes (unaligned row in shared memory) ----------------------------------------------------
      const uint32_t boff = rit * bpr, bshift = (boff & 3u) * 8u;
      const uint32_t a_brow = a_sb + lay.bases + (boff & ~3u);
      uint32_t bw[NW + 1];
#pragma unroll
      for (int k = 0; k <= NW; ++k) bw[k] = lds32(a_brow + 4 * k);
      const uint32_t vmask = ok[h] ? 0x55555555u : 0u;
#pragma unroll
      for (int k = 0; k < NW; ++k) {
        const uint32_t lmk = RG ? lm[h][k] : lenmask[k];
        rd[h][k] = __funnelshift_r(bw[k], bw[k + 1], bshift) & lmk;
        ve[h][k] = lmk & vmask;
      }
      a_qrow[h] = ok[h] ? a_sb + lay.qual + rit * L : a_zero;    // a read outside the shape adds zeros
      n_fast += ok[h] ? 1u : 0u;
    }
    // ---- N / IUPAC in the reference window (rare) or in the read -> clear those positions --------------------------
    if (__any_sync(FULL, anyinv[0] | anyinv[1] | hasn[0] | hasn[1])) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (anyinv[h]) {
#pragma unroll
          for (int k = 0; k < NW; ++k) ve[h][k] &= ~fast_spread16(iv[h][k >> 1] >> (16 * (k & 1)));
        }
        if (hasn[h]) {     // the warp has OR-ed the read's N calls into its row of the invalid map
          uint32_t* row = s_inv + (lane + h * 32) * NW;
          punct[h] = ok[h];
#pragma unroll
          for (int k = 0; k < NW; ++k) { ve[h][k] &= ~row[k]; row[k] = 0; }
        }
      }
    }
    // ---- minus strand: reverse-complement both arrays (qualities stay forward, Q10) ------------------------------
    // (tested per half of the tile: clusters are single-stranded and reads come cluster by cluster, so 32 consecutive
    //  reads are on one strand far more often than 64)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (__any_sync(FULL, FAST_REV_SPLIT ? rev[h] : (rev[0] | rev[1]))) {
        uint32_t a[NW], b[NW];
#pragma unroll
        for (int k = 0; k < NW; ++k) { a[k] = rf[h][k]; b[k] = rd[h][k]; }
        if (RG) {
          uint32_t lmh[NW];
#pragma unroll
          for (int k = 0; k < NW; ++k) lmh[k] = lm[h][RG ? k : 0];
          fast_reverse_any<NW, true>(a, Lr[h], lmh);
          fast_reverse_any<NW, true>(b, Lr[h], lmh);
        } else {
          fast_reverse<NW, true>(a, L, lenmask);
          fast_reverse<NW, true>(b, L, lenmask);
        }
#pragma unroll
        for (int k = 0; k < NW; ++k) { rf[h][k] = rev[h] ? a[k] : rf[h][k]; rd[h][k] = rev[h] ? b[k] : rd[h][k]; }
        if (punct[h] && rev[h]) {   // the plain length mask is its own mirror image; only a punctured one needs reversing
          uint32_t v[NW];
#pragma unroll
          for (int k = 0; k < NW; ++k) v[k] = ve[h][k];
          if (RG) {
            uint32_t lmh[NW];
#pragma unroll
            for (int k = 0; k < NW; ++k) lmh[k] = lm[h][RG ? k : 0];
            fast_reverse_any<NW, false>(v, Lr[h], lmh);
          } else {
            fast_reverse<NW, false>(v, L, lenmask);
          }
#pragma unroll
          for (int k = 0; k < NW; ++k) ve[h][k] = v[k] & 0x55555555u;
        }
      }
    }
    // ---- match / mismatch masks, one-hot match words, codes parked for the mismatch loop --------------------------
    uint32_t xw[2][NC], mmv[2][NW];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int k = 0; k < NW; ++k) {
        const uint32_t x = rf[h][k] ^ rd[h][k];
        const uint32_t ne = (x | (x >> 1)) & 0x55555555u;
        const uint32_t m = ~ne & ve[h][k];
        mmv[h][k] = ne & ve[h][k];
        // counted lanes per position (c1 c0 = read code of a matching base):
        //   U: even bit E0 = match,        odd bit E2 = match & c1      (G or T)
        //   V: even bit E1 = match & c0,   odd bit E3 = match & c1 & c0 (T)      (C or T)
        // A = E0-E1-E2+E3, C = E1-E3, G = E2-E3, T = E3 are formed once, at the block flush.
        const uint32_t ms = m << 1, rds = rd[h][k] << 1;
        const uint32_t ac = m | (ms & rd[h][k]);
        const uint32_t gt = rd[h][k] & (m | (ms & rds));
        if (k == NW - 1 && NC == 2 * NW - 1) xw[h][2 * k] = ac | (gt << 16);
        else { xw[h][2 * k] = ac; xw[h][2 * k + 1 < NC ? 2 * k + 1 : 0] = gt; }
        sts32(a_park + ((h * 2 + 0) * NW + k) * 128, rf[h][k]);
        sts32(a_park + ((h * 2 + 1) * NW + k) * 128, rd[h][k]);
      }
    }
    // ---- quality sums by read base over ALL positions < L (corrected for mismatches / invalid at the end) ---------
    {
      constexpr int NCH = 2 * NW;                 // chunks of 8 positions
      const bool unaligned = !RG && (LT == 0 || (LT & 3));   // rows start at any byte unless L is a multiple of 4 (RG: of 16)
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        if (8 * c >= (int)L) break;               // L is uniform over the launch: no divergence
        const bool half = 8 * c + 4 >= (int)L;    // at most four positions left: one quality word, natural order
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t qsh = (a_qrow[h] & 3u) * 8u, a_q = (a_qrow[h] & ~3u) + 8 * c;
          uint32_t q0 = lds32(a_q), q1 = half ? 0u : lds32(a_q + 4);
          if (unaligned) {
            const uint32_t q2 = lds32(a_q + (half ? 4 : 8));
            if (half) q0 = __funnelshift_r(q0, q2, qsh);
            else { q0 = __funnelshift_r(q0, q1, qsh); q1 = __funnelshift_r(q1, q2, qsh); }
          }
          const int left = (int)L - 8 * c;        // positions of this chunk that exist
          // qacc[0] collects the sum over all bases (A = total - C - G - T at the flush)
          qacc[0] = dp4a_ss(q0, left >= 4 ? 0xFFFFFFFFu : (0xFFFFFFFFu >> (8 * (4 - left))), qacc[0]);
          const uint32_t codes = rd[h][c >> 1] >> (16 * (c & 1));     // PRMT reads the low 16 bits only
          if (half) {
            uint32_t s = codes & 0xFFu;             // four codes -> four selector nibbles
            s = (s | (s << 4)) & 0x0F0Fu;
            s = (s | (s << 2)) & 0x3333u;
            qacc[1] = dp4a_ss(q0, prmt(tbl1, tbl1, s), qacc[1]);
            qacc[2] = dp4a_ss(q0, prmt(tbl2, tbl2, s), qacc[2]);
            qacc[3] = dp4a_ss(q0, prmt(tbl3, tbl3, s), qacc[3]);
          } else {
            if (left < 8) qacc[0] = dp4a_ss(q1, 0xFFFFFFFFu >> (8 * (8 - left)), qacc[0]);
            else qacc[0] = dp4a_ss(q1, 0xFFFFFFFFu, qacc[0]);
            // nibble j of `codes` = codes of positions 2j+1 | 2j: with the same table in both PRMT operands only the low
            // two bits of a nibble pick the byte (bit 2 picks the copy, bit 3 replicates the sign of a 0x00 / 0xFF byte)
            const uint32_t qe = prmt(q0, q1, 0x6420), qo = prmt(q0, q1, 0x7531);
            const uint32_t so = codes >> 2;
            qacc[1] = dp4a_ss(qe, prmt(tbl1, tbl1, codes), qacc[1]);
            qacc[2] = dp4a_ss(qe, prmt(tbl2, tbl2, codes), qacc[2]);
            qacc[3] = dp4a_ss(qe, prmt(tbl3, tbl3, codes), qacc[3]);
            qacc[1] = dp4a_ss(qo, prmt(tbl1, tbl1, so), qacc[1]);
            qacc[2] = dp4a_ss(qo, prmt(tbl2, tbl2, so), qacc[2]);
            qacc[3] = dp4a_ss(qo, prmt(tbl3, tbl3, so), qacc[3]);
          }
        }
      }
    }
    // ---- mismatching positions, one at a time.  Words 0,1 share the even/odd bits of w0, words 2,3 of w1 -----------
    uint32_t tc_lo[2] = {0, 0}, tc_hi[2] = {0, 0};
    __syncwarp();      // parked words are read back by their own lane only; the fence orders the shared accesses
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t w0 = mmv[h][0] | (NW > 1 ? (mmv[h][NW > 1 ? 1 : 0] << 1) : 0u);
      uint32_t w1 = NW > 2 ? (mmv[h][NW > 2 ? 2 : 0] | (NW > 3 ? (mmv[h][NW > 3 ? 3 : 0] << 1) : 0u)) : 0u;
      const uint32_t a_pk = a_park + (h * 2 * NW) * 128;
      while (w0 | w1) {
        const bool first = NW <= 2 || w0 != 0;
        const uint32_t word = first ? w0 : w1;
        const uint32_t b = (uint32_t)__ffs((int)word) - 1u;
        const uint32_t rest = word & (word - 1u);
        if (first) w0 = rest; else w1 = rest;
        const uint32_t k = (first ? 0u : 2u) + (b & 1u), sh = b & ~1u;
        const uint32_t rfw = lds32(a_pk + k * 128), rdw = lds32(a_pk + (NW + k) * 128);
        const uint32_t i = 16u * k + (b >> 1);
        const uint32_t pair = ((rfw >> sh) & 3u) * 4u + ((rdw >> sh) & 3u);
        const int q = lds_s8(a_qrow[h] + i);
        red_s32(a_mm_cnt + (i * 16u + pair) * 4u, 1u);
        red_s32(a_mm_q + pair * (FAST_QCOPIES * 4u), (uint32_t)q);
        const uint32_t one = pair == 13u ? 1u : 0u;         // ref T, read C on the oriented strand
        tc_lo[h] |= shl_clamp(one, i);
        tc_hi[h] |= shl_clamp(one, i - 32u);               // i < 32 wraps to a huge amount: 0
      }
    }
    // ---- rare: invalid reference positions in the window -- the quality of every invalid position went into the
    //      all-position sums, take it out again -----------------------------------------------------------------------
    if (__any_sync(FULL, anyinv[0] | anyinv[1])) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (!anyinv[h]) continue;
#pragma unroll
        for (int k = 0; k < NW; ++k) {
          uint32_t mi = ((RG ? lm[h][RG ? k : 0] : lenmask[k]) & 0x55555555u) & ~ve[h][k];
          while (mi) {
            const uint32_t b = (uint32_t)__ffs((int)mi) - 1u;
            mi &= mi - 1u;
            const uint32_t bb = (rd[h][k] >> b) & 3u;
            const int q = lds_s8(a_qrow[h] + 16u * k + (b >> 1));
            qinv[0] += bb == 0u ? q : 0; qinv[1] += bb == 1u ? q : 0; qinv[2] += bb == 2u ? q : 0; qinv[3] += bb == 3u ? q : 0;
          }
        }
      }
    }
    // ---- outputs of the tile: T>C masks, deferred reads, counters -----------------------------------------------------
    if (P.t2c_mask != nullptr) {
      unsigned long long* mp = P.t2c_mask + ((uint64_t)wt * WT_READS + lane);
      const uint32_t hi0 = ok[0] ? (tc_hi[0] | 0x80000000u | ((uint32_t)rev[0] << 30)) : 0u;
      const uint32_t hi1 = ok[1] ? (tc_hi[1] | 0x80000000u | ((uint32_t)rev[1] << 30)) : 0u;
      if (lane < n_here) mp[0] = ((unsigned long long)hi0 << 32) | tc_lo[0];        // !ok: tc_lo is 0 (no events)
      if (lane + 32 < n_here) mp[32] = ((unsigned long long)hi1 << 32) | tc_lo[1];
    }
    if (P.okmap != nullptr) {          // -q: the histogram pass adds the qualities of exactly these reads
      const uint32_t b0 = __ballot_sync(FULL, ok[0]), b1 = __ballot_sync(FULL, ok[1]);
      if (lane == 0) { P.okmap[2 * (size_t)wt] = b0; P.okmap[2 * (size_t)wt + 1] = b1; }
    }
    if (__any_sync(FULL, (!ok[0] && lane < n_here) | (!ok[1] && lane + 32 < n_here))) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t rit = lane + h * 32;
        if (!ok[h] && rit < n_here)
          P.deferred[atomicAdd(P.deferred_count, 1u)] = (uint32_t)(P.first_read + (uint64_t)wt * WT_READS + rit);
      }
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) vc_add2<NPL>(pl[c].p, xw[0][c], xw[1][c]);
    since_flush += 2;
    if (since_flush >= kFlushEvery) flush_vc();

    __syncwarp();   // every lane is done with this stage buffer
    if (wt + FAST_STAGES * GW < n_wt) {
      if (elect_one()) issue(wt + FAST_STAGES * GW, slot);
    }
  }
  flush_vc();

  // ---- per-thread totals -> shared histograms ----------------------------------------------------------------
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (tot[c] == 0) continue;
    uint32_t i, base;
    if (c == 2 * (NW - 1) && NC == 2 * NW - 1) {      // packed last word: A|C in lanes 0..15, G|T in 16..31
      i = 16u * (NW - 1) + ((lane & 15u) >> 1);
      base = 2u * (lane & 1u) + (lane >> 4);        // U half: E0/E2, V half: E1/E3
    } else {
      i = 16u * (c >> 1) + (lane >> 1);
      base = 2u * (lane & 1u) + (c & 1u);
    }
    if (i < max_len) atomicAdd(&s_fast[i * 4 + base], tot[c]);
  }
  {
    const uint32_t t = __reduce_add_sync(FULL, n_fast);
    if (lane == 0 && t) atomicAdd(&s_misc[8], (unsigned long long)t);
  }
  __syncthreads();
  // ---- block flush ---------------------------------------------------------------------------------------------
  for (uint32_t k = threadIdx.x; k < max_len * 16; k += blockDim.x) {
    const uint32_t a = (k >> 2) & 3u, b = k & 3u, i = k >> 4;
    const unsigned long long cnt = a == b ? fast_base_count(s_fast + i * 4, a) : s_mm_cnt[k];
    if (cnt) atomicAdd(P.acc + P.lay.conv + k, cnt);
  }
  if (threadIdx.x < 16) {   // per (ref, read) pair: counts and mismatch quality over all positions
    const uint32_t a = threadIdx.x >> 2, b = threadIdx.x & 3u;
    unsigned long long cnt = 0;
    long long qs = 0;
    for (uint32_t i = 0; i < max_len; ++i)
      cnt += a == b ? fast_base_count(s_fast + i * 4, a) : s_mm_cnt[i * 16 + threadIdx.x];
    if (a != b)
      for (uint32_t c = 0; c < FAST_QCOPIES; ++c) qs += (long long)(int)s_mm_q[threadIdx.x * FAST_QCOPIES + c];
    if (cnt) {
      atomicAdd(P.acc + P.lay.qcnt + threadIdx.x, cnt);   // fast reads never hold I/D: every counted base has a quality
      atomicAdd(P.acc + P.lay.ctr + PS_PC_TOTAL_BASES_CHECKED, cnt);
    }
    if (a != b && qs) {
      atomicAdd(P.acc + P.lay.qsum + threadIdx.x, (unsigned long long)qs);
      atomicAdd(&s_misc[12 + b], (unsigned long long)qs);             // mismatch quality by read base
    }
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    const uint32_t b = threadIdx.x;
    const long long v = (long long)s_misc[b] - (long long)s_misc[4 + b] - (long long)s_misc[12 + b];
    if (v) atomicAdd(P.acc + P.lay.qsum + b * 5, (unsigned long long)v);
  }
  if (threadIdx.x == 8 && s_misc[8]) {
    atomicAdd(P.acc + P.lay.ctr + PS_PC_NUM_READS_PROCESSED, s_misc[8]);
    atomicAdd(P.fault + 1, s_misc[8]);   // debug word: reads that took the fast path
  }
}

// a block may add this many reads before the 32-bit shared mismatch-quality cells could overflow
// (64 positions x |q| <= 128 x 2^17 reads = 2^30)
#define FAST_MAX_READS_PER_BLOCK (1u << 17)

template <int NW, int NPL, int LT, bool RG = false>
cudaError_t launch_fast(ps_ctx* ctx, const ProfileParams& P, uint32_t n_wt, cudaStream_t stream) {
  const size_t smem = fast_layout(P.lay.max_len, P.b.uniform_len, NW).total + 128;
  auto kern = profile_fast_kernel<NW, NPL, LT, RG>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, FAST_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  uint32_t grid = (uint32_t)ctx->sm_count * (uint32_t)per_sm;
  const uint32_t need = (n_wt + FAST_WARPS - 1) / FAST_WARPS;
  if (grid > need) grid = need;
  // keep every block under FAST_MAX_READS_PER_BLOCK by splitting very large batches into several launches
  uint64_t per_block = FAST_MAX_READS_PER_BLOCK;
  if (const char* ev = getenv("PARASUITE_B200_FAST_READS_PER_BLOCK")) {   // tests: split batches of test size too
    // whole tiles only, so that every launch starts on a tile of the exception table
    const long v = atol(ev);
    if (v >= PS_TILE_READS && v <= (long)FAST_MAX_READS_PER_BLOCK && v % PS_TILE_READS == 0) per_block = (uint64_t)v;
  }
  const uint64_t per_launch = (uint64_t)grid * per_block / WT_READS;
  for (uint64_t first = 0; first < n_wt; first += per_launch) {
    ProfileParams Q = P;
    const uint64_t cnt = std::min<uint64_t>(per_launch, n_wt - first);
    Q.n_tiles = (uint32_t)cnt;
    const uint64_t r0 = first * WT_READS;
    Q.b.meta += r0; Q.b.ref_start += r0; Q.b.cigar += r0;
    Q.b.bases2 += r0 * ((P.b.uniform_len + 3) / 4);
    Q.b.qual += r0 * P.b.uniform_len;
    Q.b.tile_exc_off += r0 / PS_TILE_READS;
    Q.b.n_reads = std::min<uint64_t>(P.b.n_reads - r0, cnt * WT_READS);
    Q.first_read = P.first_read + r0;    // offset added to deferred read indices
    if (Q.t2c_mask) Q.t2c_mask += r0;
    if (Q.okmap) Q.okmap += r0 / 32;
    kern<<<grid, FAST_THREADS, smem, stream>>>(Q);
    ctx->launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
