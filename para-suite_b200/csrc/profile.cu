// K1: error-profile count kernels.  Replace the loop ErrorProfiling.java:146-409 (reference:
// /root/reference/src/src/utils/errorprofile/ErrorProfiling.java) for one SoA batch.
//
// profile_fast_kernel   the common PAR-CLIP shape: uniform read length L <= 64, one M/=/X cigar op (L == R).
//   * persistent CTAs of 4 warps (5 per SM); every WARP owns a 2-stage ring of cp.async.bulk (TMA) copies with its own
//     mbarriers (64 reads per warp-tile: meta, ref_start, cigar, 2-bit bases, qualities are contiguous runs in HBM),
//     so there is no block barrier in the main loop;
//   * one thread per read, all per-base work bit-parallel on 2-bit packed words:
//       match counts   -> per-thread bit-sliced ("vertical") counters, one-hot (A|C, G|T) x position lanes,
//                         merged across the warp with a carry-save butterfly every 2^P-2 reads; no atomics
//       mismatches     -> rare: two native 32-bit shared atomics (count, quality sum) per mismatching base
//       quality sums   -> dp4a of the quality bytes against 0/-1 byte masks built with PRMT from the codes
//   * reads that do not fit the fast shape (flags, other cigars, contig edges) are appended to a dense list for
//     profile_deferred_kernel (thread per read, the literal routine).
// profile_generic_kernel  every CIGAR / flag / length: lane-per-read prologue, warp-per-read count loop
//     (lanes = alignment columns), warp-tiles from an atomic counter.
//
// Counts land in per-block shared-memory histograms and are flushed once per block with 64-bit global atomics
// into the accumulator vector (internal.h ProfileLayout) -- the unit of the multi-GPU all-reduce.
#include <algorithm>
#include <cstdlib>

#include "device_common.cuh"

namespace {

struct ProfileParams {
  DeviceBatch b;
  DeviceRef ref;
  ProfileLayout lay;
  unsigned long long* acc;    // int64 accumulators (two's complement adds)
  unsigned long long* fault;
  uint64_t ordinal0;
  uint64_t first_read;        // generic kernel: first read it covers
  uint32_t n_tiles;           // generic kernel: tiles from first_read on;  fast kernel: number of super-tiles
  uint32_t flush_reads;       // generic kernel: a warp empties its 32-bit per-lane sums after this many columns per lane (2^23)
  uint32_t* deferred;         // fast kernel: reads that need the generic routine (processed by profile_deferred_kernel)
  unsigned int* deferred_count;
  unsigned int* deferred_count_next;   // the counter of the run's next batch: cleared by this batch's deferred kernel
                                       // (two counters take turns, so no memset sits in front of the fast kernel)
  unsigned long long* t2c_mask;        // fast kernel, optional: one T>C mask word per read (profile_fast.cuh), for the pileup
  uint32_t* okmap;                     // fast kernel, optional (-q): bit r%32 of word r/32 = read r took the fast path
  const uint32_t* off3;                // deferred kernel on a re-laid ragged batch: [3][n_reads] in-tile offsets of every read
                                       // (bytes of bases, bytes of qualities, cigar elements), written by the repack kernel
  unsigned long long* ts;              // fast and deferred kernels, optional: stamp pair of the timed section
};

// shared-memory histograms of the generic path
struct GenericSmem {
  unsigned long long* s_q;    // [32] qualityPerMismatch sums | counts
  unsigned long long* s_ctr;  // [8]
  uint32_t* s_conv;           // [max_len*16]
  uint32_t* s_indel;          // [2*max_len] insertionsPerPos | deletionsPerPos (hot addresses: never global atomics)
};

// ---------------------------------------------------------------------------------------------------------
// Generic per-read routine: literal restatement of ErrorProfiling.java:155-408 on packed data.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_shared_add(uint32_t saddr, uint32_t v) {   // native shared-memory reduction
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}

__device__ __noinline__ void profile_read_generic(const ProfileParams& P, const GenericSmem& S, uint64_t tile,
                                                  uint32_t rit, uint64_t r, uint32_t meta, ReadOffsets off) {
  const uint32_t max_len = P.lay.max_len;
  const uint32_t flags = PS_META_FLAGS(meta), L = PS_META_LEN(meta), ncig = PS_META_NCIGAR(meta);
  const uint64_t ordinal = P.ordinal0 + r;
  // filters :155-166 (first match wins)
  if (flags & PS_RF_UNMAPPED) { atomicAdd(&S.s_ctr[PS_PC_UNMAPPED], 1ull); return; }
  if (flags & PS_RF_DUPLICATE) { atomicAdd(&S.s_ctr[PS_PC_DUPLICATES], 1ull); return; }
  if (flags & PS_RF_POS_ZERO) { atomicAdd(&S.s_ctr[PS_PC_START_ZERO], 1ull); return; }
  if (flags & PS_RF_CIGAR_OVERFLOW) { raise_fault(P.fault, ordinal, PS_FAULT_CIGAR_OPS); return; }   // not representable

  const uint32_t* cig = P.b.cigar + off.cigar;
  uint32_t R = 0;
  bool has_indel = false;
  for (uint32_t e = 0; e < ncig; ++e) {
    uint32_t c = __ldg(cig + e), op = c & 15u;
    if (op_consumes_ref(op)) R += c >> 4;
    has_indel |= (op == 1u) | (op == 2u);
  }
  const uint64_t g0 = __ldg(P.b.ref_start + r);
  {  // :169-172 FASTA fetch range
    bool bad = (flags & PS_RF_REF_RANGE) || g0 >= P.ref.n_bases;
    if (!bad) {
      uint32_t c = contig_of(P.ref, g0);
      bad = g0 + R > __ldg(P.ref.contig_off + c + 1);
    }
    if (bad) { raise_fault(P.fault, ordinal, PS_THROW_REF_RANGE); return; }
  }
  atomicAdd(&S.s_ctr[PS_PC_NUM_READS_PROCESSED], 1ull);                        // :174
  if (R == 0) { raise_fault(P.fault, ordinal, PS_THROW_EMPTY_REF); return; }

  const uint32_t ml = L > R ? L : R;
  const bool walked = L != R;
  bool skip = false;
  if (walked) {   // :194-299, pass 1: bounds (skip), indel side effects, uncaught exceptions
    int64_t pr = 0, pq = 0, pm = 0;
    for (uint32_t e = 0; e < ncig; ++e) {
      const uint32_t c = __ldg(cig + e), op = c & 15u;
      const int64_t n = c >> 4;
      if (op_is_match(op)) {
        // any z with z+pm >= ml, z+pr >= R or z+pq >= L throws inside the try -> skip
        if (n > 0 && (pm + n > (int64_t)ml || pr + n > (int64_t)R || pq + n > (int64_t)L)) skip = true;
        pm += n; pr += n; pq += n;
      } else if (op == 3u) {
        pr += n; pq += n;
      } else if (op == 1u || op == 2u) {
        if (n > 0 && pm + n > (int64_t)ml) { raise_fault(P.fault, ordinal, PS_THROW_INDEL_FILL); return; }
        pm += n;
        if (op == 1u) pq += n; else pr += n;
        uint32_t* arr = S.s_indel + (op == 1u ? 0u : max_len);
        for (int64_t q = 1; q <= n; ++q) {
          if (pm + q >= (int64_t)max_len) { raise_fault(P.fault, ordinal, PS_THROW_INDEL_POS); return; }
          atomicAdd(arr + (pm + q), 1u);
        }
        if (n > 1) atomicAdd(&S.s_ctr[PS_PC_LONGER_INDELS], 1ull);
      }
    }
    atomicAdd(&S.s_ctr[PS_PC_INDEL_READ], 1ull);                               // :296
  }
  if (skip) { atomicAdd(&S.s_ctr[PS_PC_SKIPPED_READS], 1ull); return; }        // :303-306

  // count loop :349-408 over the (virtual) temp arrays.  Every effect is a commutative sum, so the M/=/X blocks are
  // taken in cigar order on either strand (minus strand: i = ml-1-column, both bases complemented) and 16 bases at a
  // time: one funnel shift each for the reference codes, the invalid bits and the read codes.
  const bool rev = flags & PS_RF_REVERSE;
  const bool has_inv = flags & PS_RF_HAS_INVALID;
  ExcRange xr{0, 0};
  if (has_inv) xr = read_exc_range(P.b, tile, rit);
  const uint32_t qual_len = (flags & PS_RF_QUAL_MISSING) ? 0u : L;
  const uint8_t* rb = P.b.bases2 + off.base;
  const uint8_t* rq = P.b.qual + off.qual;
  int q_acc0 = 0, q_acc1 = 0, q_acc2 = 0, q_acc3 = 0;          // |q| <= 128, <= 65535 bases: no overflow
  uint32_t q_cnt0 = 0, q_cnt1 = 0, q_cnt2 = 0, q_cnt3 = 0;
  uint32_t checked = 0;
  uint32_t f_key = 0xFFFFFFFFu;   // first uncaught exception of the count loop: min over (i << 1 | QUAL_RANGE)
  const uint32_t s_conv32 = (uint32_t)__cvta_generic_to_shared(S.s_conv);
  {
    int64_t pr = 0, pq = 0, pm = 0;
    const uint32_t n_ops = walked ? ncig : 1u;
    for (uint32_t e = 0; e < n_ops; ++e) {
      int64_t n;
      if (!walked) n = L;                                      // L == R: ungapped compare (Q1)
      else {
        const uint32_t c = __ldg(cig + e), op = c & 15u;
        n = c >> 4;
        if (op == 3u) { pr += n; pq += n; continue; }
        if (op == 1u) { pm += n; pq += n; continue; }
        if (op == 2u) { pm += n; pr += n; continue; }
        if (!op_is_match(op)) continue;
      }
      for (int64_t z0 = 0; z0 < n; z0 += 16) {
        const uint32_t cnt = (uint32_t)(n - z0 < 16 ? n - z0 : 16);
        const uint64_t g = g0 + (uint64_t)(pr + z0);
        const uint32_t p = (uint32_t)(pq + z0);
        const uint32_t rw = __funnelshift_r(__ldg(P.ref.seq2 + (g >> 4)), __ldg(P.ref.seq2 + (g >> 4) + 1), (uint32_t)(g & 15u) * 2u);
        const uint32_t iw = __funnelshift_r(__ldg(P.ref.inv + (g >> 5)), __ldg(P.ref.inv + (g >> 5) + 1), (uint32_t)(g & 31u));
        const uintptr_t ba = reinterpret_cast<uintptr_t>(rb + (p >> 2));
        const uint32_t* bw = reinterpret_cast<const uint32_t*>(ba & ~(uintptr_t)3);
        const uint32_t rdw = __funnelshift_r(__ldg(bw), __ldg(bw + 1), (uint32_t)(ba & 3u) * 8u + (p & 3u) * 2u);
        uint32_t valid = (cnt == 16 ? 0x55555555u : ((1u << (2u * cnt)) - 1u) & 0x55555555u) & ~spread16_even(iw);
        if (has_inv)
          for (uint32_t x = xr.e0; x < xr.e1; ++x) {
            const uint32_t d = (__ldg(P.b.exc + x) & 0xFFFFu) - p;
            if (d < cnt) valid &= ~(1u << (2u * d));
          }
        const uint32_t col0 = (uint32_t)(pm + z0);                    // columns < ml <= 65535 + 65535
        // positions of this chunk: i = ibase + istep * k, k = 0 .. cnt-1
        const uint32_t ibase = rev ? ml - 1u - col0 : col0;
        const int istep = rev ? -1 : 1;
        const uint32_t i_max = rev ? ibase : ibase + cnt - 1u;
        const uint32_t flip = rev ? 15u : 0u;                         // complementing both bases: pair -> 15 - pair
        if (i_max < max_len && (has_indel || i_max < qual_len)) {     // no exception can be raised in this chunk
          while (valid) {
            const uint32_t k2 = (uint32_t)__ffs((int)valid) - 1u;
            valid &= valid - 1u;
            const uint32_t ra = (rw >> k2) & 3u, rb2 = (rdw >> k2) & 3u;
            const uint32_t pair = (ra * 4u + rb2) ^ flip;             // 15 - x == x ^ 15 for x < 16
            const uint32_t i = ibase + (uint32_t)(istep * (int)(k2 >> 1));
            red_shared_add(s_conv32 + (i * 16u + pair) * 4u, 1u);
            ++checked;
            if (!has_indel) {
              const int qv = (int)(signed char)__ldg(rq + i);   // qualities are NOT reversed (Q10)
              if (ra == rb2) {
                const uint32_t a = pair >> 2;
                if (a == 0) { q_acc0 += qv; q_cnt0++; } else if (a == 1) { q_acc1 += qv; q_cnt1++; }
                else if (a == 2) { q_acc2 += qv; q_cnt2++; } else { q_acc3 += qv; q_cnt3++; }
              } else {
                atomicAdd(&S.s_q[pair], (unsigned long long)(long long)qv);
                atomicAdd(&S.s_q[16 + pair], 1ull);
              }
            }
          }
        } else {
          while (valid) {
            const uint32_t k2 = (uint32_t)__ffs((int)valid) - 1u;
            valid &= valid - 1u;
            const uint32_t pair = (((rw >> k2) & 3u) * 4u + ((rdw >> k2) & 3u)) ^ flip;
            const uint32_t i = ibase + (uint32_t)(istep * (int)(k2 >> 1));
            if (i >= max_len) { f_key = min(f_key, i << 1); continue; }                 // :377
            red_shared_add(s_conv32 + (i * 16u + pair) * 4u, 1u);
            ++checked;
            if (!has_indel) {
              if (i >= qual_len) { f_key = min(f_key, (i << 1) | 1u); continue; }       // :388
              const int qv = (int)(signed char)__ldg(rq + i);
              if ((pair >> 2) == (pair & 3u)) {
                const uint32_t a = pair >> 2;
                if (a == 0) { q_acc0 += qv; q_cnt0++; } else if (a == 1) { q_acc1 += qv; q_cnt1++; }
                else if (a == 2) { q_acc2 += qv; q_cnt2++; } else { q_acc3 += qv; q_cnt3++; }
              } else {
                atomicAdd(&S.s_q[pair], (unsigned long long)(long long)qv);
                atomicAdd(&S.s_q[16 + pair], 1ull);
              }
            }
          }
        }
      }
      pm += n; pr += n; pq += n;
    }
  }
  uint32_t f_i = f_key == 0xFFFFFFFFu ? 0xFFFFFFFFu : f_key >> 1;
  uint32_t f_code = (f_key & 1u) ? PS_THROW_QUAL_RANGE : PS_THROW_POS_MAXLEN;
  bool live = f_key == 0xFFFFFFFFu;
  if (P.lay.infer_q) {   // :402-407 touches baseQualitiesPerPos[i] / readQualities[i] for EVERY i < ml
    const uint32_t iq = max_len < qual_len ? max_len : qual_len;
    if (ml > iq && iq < f_i) {
      f_i = iq;
      f_code = max_len <= qual_len ? PS_THROW_POS_MAXLEN : PS_THROW_QUAL_RANGE;
      live = false;
    }
  }
  if (f_i != 0xFFFFFFFFu) raise_fault(P.fault, ordinal, f_code);
  if (!live) return;
  if (q_cnt0) { atomicAdd(&S.s_q[0], (unsigned long long)(long long)q_acc0); atomicAdd(&S.s_q[16], (unsigned long long)q_cnt0); }
  if (q_cnt1) { atomicAdd(&S.s_q[5], (unsigned long long)(long long)q_acc1); atomicAdd(&S.s_q[21], (unsigned long long)q_cnt1); }
  if (q_cnt2) { atomicAdd(&S.s_q[10], (unsigned long long)(long long)q_acc2); atomicAdd(&S.s_q[26], (unsigned long long)q_cnt2); }
  if (q_cnt3) { atomicAdd(&S.s_q[15], (unsigned long long)(long long)q_acc3); atomicAdd(&S.s_q[31], (unsigned long long)q_cnt3); }
  atomicAdd(&S.s_ctr[PS_PC_TOTAL_BASES_CHECKED], (unsigned long long)checked);
  if (P.lay.infer_q)
    for (uint32_t i = 0; i < ml; ++i) atomicAdd(P.acc + P.lay.qhist + (size_t)i * 256 + __ldg(rq + i), 1ull);
}

__device__ __forceinline__ void flush_generic(const ProfileParams& P, const GenericSmem& S) {
  for (uint32_t k = threadIdx.x; k < P.lay.max_len * 16; k += blockDim.x)
    if (S.s_conv[k]) atomicAdd(P.acc + P.lay.conv + k, (unsigned long long)S.s_conv[k]);
  for (uint32_t k = threadIdx.x; k < 2 * P.lay.max_len; k += blockDim.x)   // ins and del are adjacent in the layout
    if (S.s_indel[k]) atomicAdd(P.acc + P.lay.ins + k, (unsigned long long)S.s_indel[k]);
  if (threadIdx.x < 32 && S.s_q[threadIdx.x]) atomicAdd(P.acc + P.lay.qsum + threadIdx.x, S.s_q[threadIdx.x]);
  if (threadIdx.x < PS_PC_COUNT && S.s_ctr[threadIdx.x])
    atomicAdd(P.acc + P.lay.ctr + threadIdx.x, S.s_ctr[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------------------
// General kernel: one WARP per read, lanes = alignment columns.
// All lanes walk the cigar together (uniform control flow, broadcast loads); inside an M/=/X block lane l takes columns
// l, l+32, ...: consecutive reference bases, read bases and qualities per lane, conflict-free native shared-memory
// reductions into a [pair][position] histogram.  Matching-base quality sums and the base counter live in per-lane
// registers for the whole kernel.  Same statements as profile_read_generic (ErrorProfiling.java:155-408).
// ---------------------------------------------------------------------------------------------------------
struct WarpAcc {          // 32-bit per lane, emptied into the block's 64-bit cells before 2^23 columns per lane have gone in
  int q_acc[4];
  uint32_t q_cnt[4];
  uint32_t checked;
  uint32_t mm_events;      // mismatch-quality events this lane has put into the warp's 32-bit cells since their last flush
  uint32_t reads;          // columns per lane (upper bound) the warp has counted since the last flush: a column adds at most 128
};

// Mismatch qualities (sum and count by pair, ErrorProfiling.java:392-397) first go to 32 warp-private 32-bit cells with
// native shared reductions -- a 64-bit shared atomicAdd is a compare-and-swap loop, and reads that compare shifted
// sequence (soft clips, Q-quirk) bring a hundred such events each -- and from there to the block's 64-bit cells before a
// cell could overflow (|q| <= 128, 2^18 events per lane).
#ifndef PS_FLUSH_INLINE
#define PS_FLUSH_INLINE __forceinline__
#endif
__device__ PS_FLUSH_INLINE void warp_q_flush(const GenericSmem& S, uint32_t wq32, WarpAcc& A) {
  __syncwarp();
  const uint32_t lane = threadIdx.x & 31;
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(wq32 + lane * 4u));
  if (v) {
    atomicAdd(&S.s_q[lane], lane < 16 ? (unsigned long long)(long long)(int)v : (unsigned long long)v);
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(wq32 + lane * 4u), "r"(0u) : "memory");
  }
  A.mm_events = 0;
  // the per-lane registers: matching-base quality sums and counts (by base), bases checked
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    long long t = A.q_acc[b];
    unsigned long long c = A.q_cnt[b];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) { t += __shfl_xor_sync(0xFFFFFFFFu, t, d); c += __shfl_xor_sync(0xFFFFFFFFu, c, d); }
    if (lane == 0 && c) { atomicAdd(&S.s_q[b * 5], (unsigned long long)t); atomicAdd(&S.s_q[16 + b * 5], c); }
    A.q_acc[b] = 0; A.q_cnt[b] = 0;
  }
  {
    unsigned long long c = A.checked;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, d);
    if (lane == 0 && c) atomicAdd(&S.s_ctr[PS_PC_TOTAL_BASES_CHECKED], c);
    A.checked = 0;
  }
  A.reads = 0;
  __syncwarp();
}

// what the count loop needs to know about a read that reached it
struct ReadPlan {
  uint64_t g0;
  uint32_t ml;          // 0: nothing to count (filtered, skipped, or the JVM died on this record)
  uint32_t bits;        // bit 0: the cigar string holds I or D; bit 1: L != R (the read was walked)
};

// Prologue of one read by ONE lane (32 reads of a warp-tile at a time): filters, FASTA range, cigar bounds, indel side
// effects, uncaught exceptions of the walk (ErrorProfiling.java:155-306).
// (the three run counters nearly every read touches -- processed, indel read, longer indel -- go to per-lane registers
// `ctr`, summed once at the end of the kernel: a 64-bit shared atomicAdd is a compare-and-swap loop, and the 32 lanes
// of a warp would all spin on the same cell)
__device__ __forceinline__ ReadPlan profile_read_prologue(const ProfileParams& P, const GenericSmem& S, uint64_t r, uint32_t meta,
                                                          const ReadOffsets& off, uint32_t (&ctr)[3]) {
  ReadPlan plan;
  plan.g0 = 0; plan.ml = 0; plan.bits = 0;
  const uint32_t max_len = P.lay.max_len;
  const uint32_t flags = PS_META_FLAGS(meta), L = PS_META_LEN(meta), ncig = PS_META_NCIGAR(meta);
  const uint64_t ordinal = P.ordinal0 + r;
  // filters :155-166 (first match wins)
  if (flags & PS_RF_UNMAPPED) { atomicAdd(&S.s_ctr[PS_PC_UNMAPPED], 1ull); return plan; }
  if (flags & PS_RF_DUPLICATE) { atomicAdd(&S.s_ctr[PS_PC_DUPLICATES], 1ull); return plan; }
  if (flags & PS_RF_POS_ZERO) { atomicAdd(&S.s_ctr[PS_PC_START_ZERO], 1ull); return plan; }
  if (flags & PS_RF_CIGAR_OVERFLOW) { raise_fault(P.fault, ordinal, PS_FAULT_CIGAR_OPS); return plan; }   // not representable
  const uint32_t* cig = P.b.cigar + off.cigar;
  uint32_t R = 0;
  bool has_indel = false;
  for (uint32_t e = 0; e < ncig; ++e) {
    const uint32_t c = __ldg(cig + e), op = c & 15u;
    if (op_consumes_ref(op)) R += c >> 4;
    has_indel |= (op == 1u) | (op == 2u);
  }
  const uint64_t g0 = __ldg(P.b.ref_start + r);
  {  // :169-172 FASTA fetch range
    bool bad = (flags & PS_RF_REF_RANGE) || g0 >= P.ref.n_bases;
    if (!bad) {
      const uint32_t c = contig_of(P.ref, g0);
      bad = g0 + R > __ldg(P.ref.contig_off + c + 1);
    }
    if (bad) { raise_fault(P.fault, ordinal, PS_THROW_REF_RANGE); return plan; }
  }
  ++ctr[0];                        // :174
  if (R == 0) { raise_fault(P.fault, ordinal, PS_THROW_EMPTY_REF); return plan; }
  const uint32_t ml = L > R ? L : R;
  if (L != R) {   // :194-299, pass 1: bounds (skip), indel side effects, uncaught exceptions
    bool skip = false;
    int64_t pr = 0, pq = 0, pm = 0;
    for (uint32_t e = 0; e < ncig; ++e) {
      const uint32_t c = __ldg(cig + e), op = c & 15u;
      const int64_t n = c >> 4;
      if (op_is_match(op)) {
        if (n > 0 && (pm + n > (int64_t)ml || pr + n > (int64_t)R || pq + n > (int64_t)L)) skip = true;
        pm += n; pr += n; pq += n;
      } else if (op == 3u) {
        pr += n; pq += n;
      } else if (op == 1u || op == 2u) {
        if (n > 0 && pm + n > (int64_t)ml) { raise_fault(P.fault, ordinal, PS_THROW_INDEL_FILL); return plan; }
        pm += n;
        if (op == 1u) pq += n; else pr += n;
        uint32_t* arr = S.s_indel + (op == 1u ? 0u : max_len);
        for (int64_t q = 1; q <= n; ++q) {
          if (pm + q >= (int64_t)max_len) { raise_fault(P.fault, ordinal, PS_THROW_INDEL_POS); return plan; }
          atomicAdd(arr + (pm + q), 1u);
        }
        if (n > 1) ++ctr[2];
      }
    }
    ++ctr[1];                               // :296
    if (skip) { atomicAdd(&S.s_ctr[PS_PC_SKIPPED_READS], 1ull); return plan; } // :303-306
  }
  // does [g0, g0 + R) hold an invalid reference base at all?  (a few mask words per read here, instead of a load and a
  // test per column in the count loop; reads with long N gaps keep the per-column test)
  bool ref_clean = false;
  if (R <= 512u) {
    const uint64_t last = g0 + R - 1u, w0 = g0 >> 5, w1 = last >> 5;
    uint32_t any = 0;
    for (uint64_t w = w0; w <= w1; ++w) {
      uint32_t m = 0xFFFFFFFFu;
      if (w == w0) m &= 0xFFFFFFFFu << (uint32_t)(g0 & 31u);
      if (w == w1) m &= 0xFFFFFFFFu >> (31u - (uint32_t)(last & 31u));
      any |= __ldg(P.ref.inv + w) & m;
    }
    ref_clean = any == 0;
  }
  plan.g0 = g0; plan.ml = ml; plan.bits = (has_indel ? 1u : 0u) | (L != R ? 2u : 0u) | (ref_clean ? 4u : 0u);
  return plan;
}

// Count loop of one read by the WHOLE warp (ErrorProfiling.java:349-408).
__device__ __forceinline__ void profile_read_warp(const ProfileParams& P, const GenericSmem& S, uint32_t convT, uint32_t pad,
                                                  uint32_t wq32, uint64_t r, uint32_t meta, ReadOffsets off, ReadPlan plan,
                                                  WarpAcc& A) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t max_len = P.lay.max_len;
  const uint32_t flags = PS_META_FLAGS(meta), L = PS_META_LEN(meta), ncig = PS_META_NCIGAR(meta);
  const uint64_t ordinal = P.ordinal0 + r;
  const uint32_t* cig = P.b.cigar + off.cigar;
  const uint64_t g0 = plan.g0;
  const uint32_t ml = plan.ml;
  const bool has_indel = (plan.bits & 1u) != 0, walked = (plan.bits & 2u) != 0, ref_clean = (plan.bits & 4u) != 0;
  // the read's window of the reference: word pointers once, 32-bit offsets per column
  const uint32_t* inv_w = P.ref.inv + (g0 >> 5);
  const uint32_t* seq_w = P.ref.seq2 + (g0 >> 4);
  const uint32_t g_in32 = (uint32_t)(g0 & 31u), g_in16 = (uint32_t)(g0 & 15u);
  // count loop :349-408
  const bool rev = flags & PS_RF_REVERSE;
  const bool has_inv = flags & PS_RF_HAS_INVALID;
  ExcRange xr{0, 0};
  if (has_inv) xr = read_exc_range(P.b, r / PS_TILE_READS, (uint32_t)(r % PS_TILE_READS));
  const uint32_t qual_len = (flags & PS_RF_QUAL_MISSING) ? 0u : L;
  const uint8_t* rb = P.b.bases2 + off.base;
  const uint8_t* rq = P.b.qual + off.qual;
  const uint32_t flip = rev ? 15u : 0u;           // complementing both bases: pair -> 15 - pair
  uint32_t f_key = 0xFFFFFFFFu;                   // first uncaught exception: min over (i << 1 | QUAL_RANGE)
  int qa0 = 0, qa1 = 0, qa2 = 0, qa3 = 0;
  uint32_t qc0 = 0, qc1 = 0, qc2 = 0, qc3 = 0, checked = 0;
  {
    uint32_t pr = 0, pq = 0, pm = 0;              // the read was not skipped: every block lies inside ml, R and L
    const uint32_t n_ops = walked ? ncig : 1u;
    for (uint32_t e = 0; e < n_ops; ++e) {
      uint32_t n;
      if (!walked) n = L;                         // L == R: ungapped compare (Q1)
      else {
        const uint32_t c = __ldg(cig + e), op = c & 15u;
        n = c >> 4;
        if (op == 3u) { pr += n; pq += n; continue; }
        if (op == 1u) { pm += n; pq += n; continue; }
        if (op == 2u) { pm += n; pr += n; continue; }
        if (!op_is_match(op)) continue;
      }
      for (uint32_t z = lane; z < n; z += 32) {
        const uint32_t p = pq + z, col = pm + z, gi = g_in32 + pr + z, gs = g_in16 + pr + z;
        bool ok = ref_clean || !((__ldg(inv_w + (gi >> 5)) >> (gi & 31u)) & 1u);
        if (ok && has_inv) ok = !read_pos_invalid(P.b, xr, p);
        if (!ok) continue;
        const uint32_t ra = (__ldg(seq_w + (gs >> 4)) >> (2u * (gs & 15u))) & 3u;
        const uint32_t rd = ((uint32_t)__ldg(rb + (p >> 2)) >> (2u * (p & 3u))) & 3u;
        const uint32_t pair = (ra * 4u + rd) ^ flip;
        const uint32_t i = rev ? ml - 1u - col : col;
        if (i >= max_len) { f_key = min(f_key, i << 1); continue; }                 // :377
        red_shared_add(convT + (pair * pad + i) * 4u, 1u);
        ++checked;
        if (!has_indel) {
          if (i >= qual_len) { f_key = min(f_key, (i << 1) | 1u); continue; }       // :388
          const int qv = (int)(signed char)__ldg(rq + i);   // qualities are NOT reversed (Q10)
          if (ra == rd) {
            const uint32_t a = pair >> 2;
            if (a == 0) { qa0 += qv; qc0++; } else if (a == 1) { qa1 += qv; qc1++; }
            else if (a == 2) { qa2 += qv; qc2++; } else { qa3 += qv; qc3++; }
          } else {
            red_shared_add(wq32 + pair * 4u, (uint32_t)qv);
            red_shared_add(wq32 + (16u + pair) * 4u, 1u);
            ++A.mm_events;
          }
        }
      }
      pm += n; pr += n; pq += n;
    }
  }
  if (__any_sync(0xFFFFFFFFu, A.mm_events >= (1u << 18)) || A.reads >= P.flush_reads) warp_q_flush(S, wq32, A);
  f_key = __reduce_min_sync(0xFFFFFFFFu, f_key);
  uint32_t f_i = f_key == 0xFFFFFFFFu ? 0xFFFFFFFFu : f_key >> 1;
  uint32_t f_code = (f_key & 1u) ? PS_THROW_QUAL_RANGE : PS_THROW_POS_MAXLEN;
  if (P.lay.infer_q) {   // :402-407 touches baseQualitiesPerPos[i] / readQualities[i] for EVERY i < ml
    const uint32_t iq = max_len < qual_len ? max_len : qual_len;
    if (ml > iq && iq < f_i) { f_i = iq; f_code = max_len <= qual_len ? PS_THROW_POS_MAXLEN : PS_THROW_QUAL_RANGE; }
  }
  if (f_i != 0xFFFFFFFFu) { if (lane == 0) raise_fault(P.fault, ordinal, f_code); return; }
  A.q_acc[0] += qa0; A.q_acc[1] += qa1; A.q_acc[2] += qa2; A.q_acc[3] += qa3;
  A.q_cnt[0] += qc0; A.q_cnt[1] += qc1; A.q_cnt[2] += qc2; A.q_cnt[3] += qc3;
  A.checked += checked;
  A.reads += (ml + 31u) >> 5;                    // columns a lane may have counted for this read
  if (P.lay.infer_q)
    for (uint32_t i = lane; i < ml; i += 32) atomicAdd(P.acc + P.lay.qhist + (size_t)i * 256 + __ldg(rq + i), 1ull);
}

// Shared memory: s_q[32] u64 | s_ctr[16] u64 | histogram [16][pad] u32 (pad = max_len | 1) | s_indel[2*max_len] u32
// Work unit = a warp-tile of 32 consecutive reads, handed out by an atomic counter: no block barrier in the loop.  The
// tile's per-read stream offsets come from one warp scan; the warp then takes the 32 reads one after the other.
#ifndef PS_GENERIC_BLOCKS
#define PS_GENERIC_BLOCKS 4
#endif
__global__ void __launch_bounds__(PS_BLOCK_THREADS, PS_GENERIC_BLOCKS) profile_generic_kernel(const __grid_constant__ ProfileParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  GenericSmem S;
  const uint32_t max_len = P.lay.max_len, pad = max_len | 1u;
  S.s_q = reinterpret_cast<unsigned long long*>(smem_raw);
  S.s_ctr = S.s_q + 32;
  S.s_conv = reinterpret_cast<uint32_t*>(S.s_ctr + 16);      // transposed here: [pair][pad]
  S.s_indel = S.s_conv + 16 * pad;
  uint32_t* s_wq = S.s_indel + 2 * max_len;                  // [warps][32] warp-private mismatch-quality cells
  for (uint32_t k = threadIdx.x; k < 16 * pad + 2 * max_len + (PS_BLOCK_THREADS / 32) * 32; k += blockDim.x) S.s_conv[k] = 0;
  if (threadIdx.x < 48) S.s_q[threadIdx.x] = 0;   // s_q and s_ctr are contiguous
  __syncthreads();
  const uint32_t convT = (uint32_t)__cvta_generic_to_shared(S.s_conv);
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t wq32 = (uint32_t)__cvta_generic_to_shared(s_wq) + (threadIdx.x >> 5) * 128u;
  uint4* wstate = reinterpret_cast<uint4*>((reinterpret_cast<uintptr_t>(s_wq + (PS_BLOCK_THREADS / 32) * 32) + 15u) & ~(uintptr_t)15u) +
                  (threadIdx.x >> 5) * 96u;
  WarpAcc A;
#pragma unroll
  for (int b = 0; b < 4; ++b) { A.q_acc[b] = 0; A.q_cnt[b] = 0; }
  A.checked = 0;
  A.mm_events = 0;
  A.reads = 0;
  uint32_t ctr[3] = {0, 0, 0};      // processed, indel reads, longer indels
  unsigned int* counter = reinterpret_cast<unsigned int*>(P.fault + 3);   // zeroed by the launcher
  for (;;) {
    unsigned int wt = 0;
    if (lane == 0) wt = atomicAdd(counter, 1u);
    wt = __shfl_sync(0xFFFFFFFFu, wt, 0);
    if (wt >= P.n_tiles) break;
    const uint64_t q = P.first_read + (uint64_t)wt * 32u, r = q + lane;
    const bool in_range = r < P.b.n_reads;
    const uint32_t meta = in_range ? __ldg(P.b.meta + r) : 0;
    const ReadOffsets off = warp_read_offsets(P.b, q, r, in_range, meta);
    ReadPlan plan;
    plan.g0 = 0; plan.ml = 0; plan.bits = 0;
    if (in_range) plan = profile_read_prologue(P, S, r, meta, off, ctr);
    uint32_t todo = __ballot_sync(0xFFFFFFFFu, plan.ml != 0);
    // what the lanes found goes to the warp's rows in shared memory: the count loop fetches a read's row with three
    // broadcast loads, and none of it stays in registers across the loop (the kernel runs at 64 registers per thread)
    __syncwarp();
    wstate[lane * 3 + 0] = make_uint4((uint32_t)off.base, (uint32_t)(off.base >> 32), (uint32_t)off.qual, (uint32_t)(off.qual >> 32));
    wstate[lane * 3 + 1] = make_uint4((uint32_t)off.cigar, (uint32_t)(off.cigar >> 32), (uint32_t)plan.g0, (uint32_t)(plan.g0 >> 32));
    wstate[lane * 3 + 2] = make_uint4(plan.ml, plan.bits, meta, 0u);
    __syncwarp();
    while (todo) {
      const int j = __ffs((int)todo) - 1;
      todo &= todo - 1;
      const uint4 s0 = wstate[j * 3 + 0], s1 = wstate[j * 3 + 1], s2 = wstate[j * 3 + 2];
      ReadOffsets oj;
      oj.base = (uint64_t)s0.x | ((uint64_t)s0.y << 32);
      oj.qual = (uint64_t)s0.z | ((uint64_t)s0.w << 32);
      oj.cigar = (uint64_t)s1.x | ((uint64_t)s1.y << 32);
      ReadPlan pj;
      pj.g0 = (uint64_t)s1.z | ((uint64_t)s1.w << 32);
      pj.ml = s2.x;
      pj.bits = s2.y;
      profile_read_warp(P, S, convT, pad, wq32, q + j, s2.z, oj, pj, A);
      __syncwarp();
    }
  }
  warp_q_flush(S, wq32, A);                    // per-lane registers -> shared
  {
    const int which[3] = {PS_PC_NUM_READS_PROCESSED, PS_PC_INDEL_READ, PS_PC_LONGER_INDELS};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const uint32_t t = __reduce_add_sync(0xFFFFFFFFu, ctr[k]);    // a lane sees far fewer than 2^32 / 32 reads
      if (lane == 0 && t) atomicAdd(&S.s_ctr[which[k]], (unsigned long long)t);
    }
  }
  __syncthreads();
  // flush (the histogram is [pair][position] here)
  for (uint32_t k = threadIdx.x; k < max_len * 16; k += blockDim.x) {
    const uint32_t v = S.s_conv[(k & 15u) * pad + (k >> 4)];
    if (v) atomicAdd(P.acc + P.lay.conv + k, (unsigned long long)v);
  }
  for (uint32_t k = threadIdx.x; k < 2 * max_len; k += blockDim.x)
    if (S.s_indel[k]) atomicAdd(P.acc + P.lay.ins + k, (unsigned long long)S.s_indel[k]);
  if (threadIdx.x < 32 && S.s_q[threadIdx.x]) atomicAdd(P.acc + P.lay.qsum + threadIdx.x, S.s_q[threadIdx.x]);
  if (threadIdx.x < PS_PC_COUNT && S.s_ctr[threadIdx.x]) atomicAdd(P.acc + P.lay.ctr + threadIdx.x, S.s_ctr[threadIdx.x]);
}

// Reads the fast kernel could not take (flags, other cigars, contig edges): a dense list, so every thread of a
// warp has work instead of 31 lanes waiting for one slow read.  Only uniform batches reach this kernel.
__global__ void __launch_bounds__(PS_BLOCK_THREADS) profile_deferred_kernel(const __grid_constant__ ProfileParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  GenericSmem S;
  S.s_q = reinterpret_cast<unsigned long long*>(smem_raw);
  S.s_ctr = S.s_q + 32;
  S.s_conv = reinterpret_cast<uint32_t*>(S.s_ctr + 16);
  S.s_indel = S.s_conv + P.lay.max_len * 16;
  for (uint32_t k = threadIdx.x; k < P.lay.max_len * 18; k += blockDim.x) S.s_conv[k] = 0;
  if (threadIdx.x < 48) S.s_q[threadIdx.x] = 0;
  pdl_wait();      // the list and its count come from the fast kernel
  pdl_launch_dependents();
  if (P.ts && threadIdx.x == 0) stamp_start(P.ts);
  __syncthreads();
  const unsigned int n = *P.deferred_count;
  if (blockIdx.x == 0 && threadIdx.x == 0) *P.deferred_count_next = 0;
  const uint32_t bpr = (P.b.uniform_len + 3) >> 2;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const uint64_t r = P.deferred[k];
    ReadOffsets off;
    if (P.off3 != nullptr) {      // ragged batch: tile offset + the in-tile offset the repack kernel left
      const uint64_t t = r / PS_TILE_READS, n_all = P.b.n_reads;
      off.base = (P.b.uniform_len ? t * PS_TILE_READS * bpr : __ldg(P.b.tile_base_off + t)) + __ldg(P.off3 + r);
      off.qual = (P.b.uniform_len ? t * PS_TILE_READS * (uint64_t)P.b.uniform_len : __ldg(P.b.tile_qual_off + t)) + __ldg(P.off3 + n_all + r);
      off.cigar = (P.b.uniform_ncigar ? t * PS_TILE_READS * (uint64_t)P.b.uniform_ncigar : __ldg(P.b.tile_cigar_off + t)) +
                  __ldg(P.off3 + 2 * n_all + r);
    } else {
      off.base = r * (uint64_t)bpr;
      off.qual = r * (uint64_t)P.b.uniform_len;
      off.cigar = r * (uint64_t)P.b.uniform_ncigar;
    }
    profile_read_generic(P, S, r / PS_TILE_READS, (uint32_t)(r % PS_TILE_READS), r, __ldg(P.b.meta + r), off);
  }
  __syncthreads();
  flush_generic(P, S);
  if (P.ts && threadIdx.x == 0) stamp_end(P.ts + 1);
}

// ---------------------------------------------------------------------------------------------------------
// Ragged batch -> rows of S positions for the fast kernel (profile_fast.cuh, RG): one block per tile of 256 reads.
// A block scan over the metas gives every read's place in the three streams (left in `off3` for the deferred kernel);
// then every thread moves its own read: aligned word loads + funnel shifts out of the streams (neighbouring lanes read
// neighbouring rows, so the loads hit the same lines), 16-byte stores into its row, zero beyond the read's end.  Reads
// longer than S get a zero row: the fast kernel hands them to the deferred kernel, which works on the original streams.
// ---------------------------------------------------------------------------------------------------------
struct RepackParams {
  DeviceBatch b;          // the batch as uploaded
  uint64_t first_read;    // chunk [first_read, first_read + n_reads), first_read a multiple of PS_TILE_READS
  uint64_t n_reads;
  uint32_t S;             // row length in positions: a multiple of 16, <= 64
  uint32_t* bases_out;    // [n_reads][S/16] words
  uint32_t* qual_out;     // [n_reads][S/4] words
  uint32_t* op0_out;      // [n_reads] the read's cigar op when it has exactly one, else ~0
  uint32_t* off3;         // [3][b.n_reads]
};

// One stream row -> NWORDS output words: bytes [a, a + len) of `stream`, zero behind them.  The row starts at any byte:
// aligned word loads, funnel shifts; a word is only requested when it holds a wanted byte.
template <int NWORDS>
__device__ __forceinline__ void repack_row(const uint8_t* stream, uint64_t a, uint32_t len, uint32_t (&o)[NWORDS]) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(stream) + (a >> 2);
  const uint32_t sk = (uint32_t)(a & 3u), need = sk + len;      // bytes counted from the aligned start
  uint32_t prev = len ? __ldg(w) : 0u;
#pragma unroll
  for (int k = 0; k < NWORDS; ++k) {
    const uint32_t nxt = 4u * (uint32_t)(k + 1) < need ? __ldg(w + k + 1) : 0u;
    const uint32_t v = __funnelshift_r(prev, nxt, sk * 8u);
    const int have = (int)len - 4 * k;
    o[k] = have >= 4 ? v : (have <= 0 ? 0u : (v & ((1u << (8 * have)) - 1u)));
    prev = nxt;
  }
}

template <int NW>     // S = 16 * NW
__global__ void __launch_bounds__(PS_TILE_READS) profile_repack_kernel(const __grid_constant__ RepackParams P) {
  __shared__ unsigned long long s_wsum[PS_TILE_READS / 32];
  const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint64_t tile = P.first_read / PS_TILE_READS + blockIdx.x;
  const uint64_t r = tile * PS_TILE_READS + t, r_end = P.first_read + P.n_reads;
  const bool in = r < r_end;
  const uint32_t meta = in ? __ldg(P.b.meta + r) : 0u;
  const uint32_t L = PS_META_LEN(meta), nc = PS_META_NCIGAR(meta);
  // L | bytes of bases << 25 | cigar ops << 48, like warp_read_offsets
  const unsigned long long mine = (unsigned long long)L | ((unsigned long long)((L + 3) >> 2) << 25) | ((unsigned long long)nc << 48);
  unsigned long long inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, inc, d);
    if (lane >= (uint32_t)d) inc += y;
  }
  if (lane == 31) s_wsum[warp] = inc;
  __syncthreads();
  unsigned long long pre = 0;
  for (uint32_t w = 0; w < warp; ++w) pre += s_wsum[w];
  if (!in) return;
  const unsigned long long ex = pre + inc - mine;
  const uint32_t relq = (uint32_t)(ex & 0x1FFFFFFu), relb = (uint32_t)((ex >> 25) & 0x7FFFFFu), relc = (uint32_t)(ex >> 48);
  const uint64_t B0 = P.b.uniform_len ? tile * PS_TILE_READS * (uint64_t)((P.b.uniform_len + 3) >> 2) : __ldg(P.b.tile_base_off + tile);
  const uint64_t Q0 = P.b.uniform_len ? tile * PS_TILE_READS * (uint64_t)P.b.uniform_len : __ldg(P.b.tile_qual_off + tile);
  const uint64_t C0 = P.b.uniform_ncigar ? tile * PS_TILE_READS * (uint64_t)P.b.uniform_ncigar : __ldg(P.b.tile_cigar_off + tile);
  P.off3[r] = relb;
  P.off3[P.b.n_reads + r] = relq;
  P.off3[2 * P.b.n_reads + r] = relc;
  const uint64_t row = r - P.first_read;
  P.op0_out[row] = nc == 1u ? __ldg(P.b.cigar + C0 + relc) : 0xFFFFFFFFu;
  const uint32_t Lr = L <= 16u * NW ? L : 0u;              // longer reads: a zero row (the deferred kernel takes them)
  {  // qualities: one row of 16 * NW bytes, written as NW 16-byte stores
    uint4* dst = reinterpret_cast<uint4*>(P.qual_out) + row * NW;
#pragma unroll
    for (int g = 0; g < NW; ++g) {
      uint32_t o[4];
      const uint32_t done = 16u * (uint32_t)g;
      repack_row<4>(P.b.qual, Q0 + relq + done, Lr > done ? Lr - done : 0u, o);
      dst[g] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
  {  // bases: NW words
    uint32_t o[NW];
    repack_row<NW>(P.b.bases2, B0 + relb, (Lr + 3u) >> 2, o);
    uint32_t* dst = P.bases_out + row * NW;
#pragma unroll
    for (int k = 0; k < NW; ++k) dst[k] = o[k];
  }
}

#include "profile_fast.cuh"

}  // namespace

static cudaError_t launch_generic(ps_ctx* ctx, ProfileParams P, uint64_t first_read, cudaStream_t stream) {
  if (first_read >= P.b.n_reads) return cudaSuccess;
  P.first_read = first_read;
  const uint64_t n_wt = (P.b.n_reads - first_read + 31) / 32;
  if (n_wt > 0xFFFFFFF0ull) return cudaErrorInvalidValue;
  P.n_tiles = (uint32_t)n_wt;
  P.flush_reads = 1u << 23;          // columns per lane: |quality| <= 128, so a sum stays below 2^30 + one read
  if (const char* e = getenv("PARASUITE_B200_GENERIC_FLUSH_READS")) {   // tests: exercise the flush in the middle of a launch
    const long v = atol(e);
    if (v >= 1 && v <= (1l << 23)) P.flush_reads = (uint32_t)v;
  }
  size_t smem = 48 * 8 + ((size_t)(ctx->layout.max_len | 1u) * 16 + 2 * (size_t)ctx->layout.max_len) * 4 +
                (PS_BLOCK_THREADS / 32) * 32 * 4 +     // + the warps' 32-bit mismatch-quality cells
                (PS_BLOCK_THREADS / 32) * 32 * 48 + 16; // + the warps' lane-per-read state (48 bytes per read, 16-byte aligned)
  int per_sm = 0;
  cudaError_t e = fn_blocks_per_sm(ctx, reinterpret_cast<const void*>(profile_generic_kernel), PS_BLOCK_THREADS, smem, &per_sm);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  uint32_t grid = (uint32_t)ctx->sm_count * (uint32_t)per_sm;
  const uint32_t need = (P.n_tiles + PS_BLOCK_THREADS / 32 - 1) / (PS_BLOCK_THREADS / 32);
  if (grid > need) grid = need;
  e = cudaMemsetAsync(P.fault + 3, 0, 4, stream);     // warp-tile counter
  if (e != cudaSuccess) return e;
  profile_generic_kernel<<<grid, PS_BLOCK_THREADS, smem, stream>>>(P);
  ctx->launches++;
  return cudaGetLastError();
}

static cudaError_t launch_deferred(ps_ctx* ctx, const ProfileParams& P, cudaStream_t stream) {
  size_t smem = 48 * 8 + (size_t)ctx->layout.max_len * 18 * 4;
  int per_sm = 0;
  cudaError_t e = fn_blocks_per_sm(ctx, reinterpret_cast<const void*>(profile_deferred_kernel), PS_BLOCK_THREADS, smem, &per_sm);
  if (e != cudaSuccess) return e;
  e = launch_chained(ctx, profile_deferred_kernel, (uint32_t)ctx->sm_count, PS_BLOCK_THREADS, smem, stream, P);
  ctx->launches++;
  return e;
}

// `-q` on the fast path: baseQualitiesPerPos[i].add(readQualities[i]) for every i < L (ErrorProfiling.java:402-407) of the
// reads the fast kernel counted (its ok-map), as a histogram [position][byte] in shared memory.  Rows of `stride` bytes
// (the uniform batch itself, or the re-laid rows of a ragged one); lane = read, so a warp walks 32 neighbouring rows.
// Rows of the histogram are 257 words apart: equal qualities at neighbouring positions fall into different banks.
namespace {
__global__ void __launch_bounds__(256) profile_qhist_kernel(const uint8_t* __restrict__ qual, const uint32_t* __restrict__ meta,
                                                            const uint32_t* __restrict__ okmap, uint64_t n_reads, uint32_t stride,
                                                            uint32_t uniform_L, uint32_t max_len, unsigned long long* acc_qhist) {
  extern __shared__ uint32_t s_hist[];          // [max_len][257]
  for (uint32_t k = threadIdx.x; k < max_len * 257u; k += blockDim.x) s_hist[k] = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t n_groups = (n_reads + 31) / 32;
  for (uint64_t g = (uint64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); g < n_groups; g += (uint64_t)gridDim.x * (blockDim.x / 32)) {
    const uint64_t r = g * 32 + lane;
    const uint32_t okw = __ldg(okmap + g);
    if (r >= n_reads || !((okw >> lane) & 1u)) continue;
    const uint32_t L = uniform_L ? uniform_L : PS_META_LEN(__ldg(meta + r));
    const uint8_t* row = qual + r * (uint64_t)stride;
    if ((stride & 3u) == 0) {
      const uint32_t* w = reinterpret_cast<const uint32_t*>(row);
      for (uint32_t i = 0; i < L; i += 4) {
        const uint32_t v = __ldg(w + (i >> 2));
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j)
          if (i + j < L) atomicAdd(&s_hist[(i + j) * 257u + ((v >> (8u * j)) & 255u)], 1u);
      }
    } else {
      for (uint32_t i = 0; i < L; ++i) atomicAdd(&s_hist[i * 257u + __ldg(row + i)], 1u);
    }
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < max_len * 256u; k += blockDim.x) {
    const uint32_t v = s_hist[(k >> 8) * 257u + (k & 255u)];
    if (v) atomicAdd(acc_qhist + k, (unsigned long long)v);
  }
}
}  // namespace

static cudaError_t launch_qhist(ps_ctx* ctx, const uint8_t* qual, const uint32_t* meta, const uint32_t* okmap, uint64_t n_reads,
                                uint32_t stride, uint32_t uniform_L, unsigned long long* acc, cudaStream_t stream) {
  const uint32_t max_len = ctx->layout.max_len;
  const size_t smem = (size_t)max_len * 257 * 4;
  int per_sm = 0;
  cudaError_t e = fn_blocks_per_sm(ctx, reinterpret_cast<const void*>(profile_qhist_kernel), 256, smem, &per_sm);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const uint64_t need = (n_reads + 255) / 256;
  // a block's 32-bit cells see at most n_reads / grid reads each: keep that below 2^31
  uint32_t grid = (uint32_t)std::min<uint64_t>(need, (uint64_t)ctx->sm_count * per_sm);
  grid = std::max<uint32_t>(grid, (uint32_t)std::min<uint64_t>(need, n_reads / (1ull << 31) + 1));
  profile_qhist_kernel<<<grid, 256, smem, stream>>>(qual, meta, okmap, n_reads, stride, uniform_L, max_len,
                                                      acc + ctx->layout.qhist);
  ctx->launches++;
  return cudaGetLastError();
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

cudaError_t launch_profile(ps_ctx* ctx, const DeviceBatch& b, uint64_t ordinal0, cudaStream_t stream,
                           unsigned long long* t2c_mask, bool* mask_written) {
  if (mask_written) *mask_written = false;
  if (b.n_reads == 0) {
    timer_begin(ctx, stream);
    timer_end(ctx, stream);
    return cudaSuccess;
  }
  ProfileParams P;
  P.b = b;
  P.ref = ctx->ref;
  P.lay = ctx->layout;
  P.acc = static_cast<unsigned long long*>(ctx->acc.p);
  P.fault = static_cast<unsigned long long*>(ctx->fault.p);
  P.ordinal0 = ordinal0;
  P.first_read = 0;
  P.n_tiles = 0;
  P.deferred = nullptr;
  P.t2c_mask = nullptr;
  P.off3 = nullptr;
  P.okmap = nullptr;
  P.ts = nullptr;
  // both counters are zero at the start of a run (ps_profile_begin clears the words behind the fault word)
  P.deferred_count = reinterpret_cast<unsigned int*>(P.fault + 2) + (ctx->profile_batches & 1u);
  P.deferred_count_next = reinterpret_cast<unsigned int*>(P.fault + 2) + ((ctx->profile_batches + 1u) & 1u);
  uint64_t done = 0;
  const uint32_t L = b.uniform_len;
  // -q: the fast kernels count as usual and leave a map of the reads they took; profile_qhist_kernel adds those reads'
  // qualities to the per-position histogram (the deferred kernel does it for the others)
  const bool q_ok = !ctx->layout.infer_q || ctx->layout.max_len <= 64;
  const bool fast_ok = L >= 1 && L <= 64 && b.uniform_ncigar == 1 && q_ok && ctx->layout.max_len <= 256 &&
                       aligned16(b.meta) && aligned16(b.ref_start) && aligned16(b.cigar) && aligned16(b.bases2) &&
                       aligned16(b.qual) && b.n_reads < 0xFFFFFFFFull;
  if (fast_ok) {
    cudaError_t ee = ctx->deferred.reserve((size_t)b.n_reads * 4);
    if (ee != cudaSuccess) return ee;
    P.deferred = static_cast<uint32_t*>(ctx->deferred.p);
    // bits 62 and 63 of a mask word are flags: the mask is offered for L <= 62 only
    if (t2c_mask && L <= 62) { P.t2c_mask = t2c_mask; if (mask_written) *mask_written = true; }
    if (ctx->layout.infer_q) {
      if ((ee = ctx->rg_okmap.reserve(((size_t)b.n_reads + 63) / 64 * 8 + 64)) != cudaSuccess) return ee;
      P.okmap = static_cast<uint32_t*>(ctx->rg_okmap.p);
    }
    ctx->profile_batches++;
    // the fast and the deferred kernel are chained (launch_chained): their section's time comes from their stamps
    timer_begin_chained(ctx, stream);
    P.ts = ctx->cur_ts;
    const uint32_t n_wt = (uint32_t)((b.n_reads + WT_READS - 1) / WT_READS);   // the fast kernel takes every read
    const uint32_t nw = (L + 15) / 16;
    cudaError_t e;
    // read lengths sequencers commonly leave get an instantiation with the length as a compile-time constant (static loop
    // bounds, the last word's counters packed): 20-25 % faster than the run-time-length ones
    if (L == 36) e = launch_fast<3, 6, 36>(ctx, P, n_wt, stream);
    else if (L == 50) e = launch_fast<4, 5, 50>(ctx, P, n_wt, stream);
    else if (L == 51) e = launch_fast<4, 5, 51>(ctx, P, n_wt, stream);
    else if (L == 40) e = launch_fast<3, 6, 40>(ctx, P, n_wt, stream);
    else if (L == 32) e = launch_fast<2, 6, 32>(ctx, P, n_wt, stream);
    else if (nw == 1) e = launch_fast<1, 6, 0>(ctx, P, n_wt, stream);
    else if (nw == 2) e = launch_fast<2, 6, 0>(ctx, P, n_wt, stream);
    else if (nw == 3) e = launch_fast<3, 5, 0>(ctx, P, n_wt, stream);
    else e = launch_fast<4, 5, 0>(ctx, P, n_wt, stream);
    if (e != cudaSuccess) return e;
    if (P.okmap && (e = launch_qhist(ctx, b.qual, b.meta, P.okmap, b.n_reads, L, L, P.acc, stream)) != cudaSuccess) return e;
    e = launch_deferred(ctx, P, stream);
    timer_end(ctx, stream);
    return e;
  }
  // Ragged batches of short reads (adapter-trimmed PAR-CLIP reads as an aligner leaves them): re-lay them as rows of
  // S = 16 * ceil(max_read_length / 16) positions and run the fast kernel with per-read lengths.  Reads of another
  // shape (several cigar ops, clips, longer than S) go to the deferred kernel on the original streams; the test on the
  // op count keeps batches of mostly gapped alignments on the warp-per-read kernel.
  const uint32_t max_len = ctx->layout.max_len;
  const bool ragged_ok = max_len >= 1 && max_len <= 64 && b.n_reads < 0xFFFFFFFFull &&
                         aligned16(b.meta) && aligned16(b.ref_start) && (b.uniform_len == 0 || b.uniform_len <= 64) &&
                         (reinterpret_cast<uintptr_t>(b.bases2) & 3u) == 0 && (reinterpret_cast<uintptr_t>(b.qual) & 3u) == 0 &&
                         b.cigar_count * 2 <= b.n_reads * 3 && getenv("PARASUITE_B200_NO_RAGGED_FAST") == nullptr;
  if (ragged_ok) {
    // rows as short as the batch allows when its producer says how long the longest read is
    const uint32_t Lmax = b.max_len ? std::min(b.max_len, max_len) : max_len;
    const uint32_t S = (Lmax + 15u) / 16u * 16u, nw = S / 16u;
    uint64_t chunk = 1ull << 23;                              // reads re-laid per pass (bounds the scratch rows)
    if (const char* ev = getenv("PARASUITE_B200_RAGGED_CHUNK")) {
      const uint64_t v = strtoull(ev, nullptr, 10) / PS_TILE_READS * PS_TILE_READS;
      if (v >= PS_TILE_READS && v <= (1ull << 26)) chunk = v;
    }
    chunk = std::min<uint64_t>((b.n_reads + PS_TILE_READS - 1) / PS_TILE_READS * PS_TILE_READS, chunk);
    cudaError_t e;
    if ((e = ctx->deferred.reserve((size_t)b.n_reads * 4)) != cudaSuccess) return e;
    if ((e = ctx->rg_off.reserve((size_t)b.n_reads * 12)) != cudaSuccess) return e;
    if ((e = ctx->rg_bases.reserve((size_t)chunk * (S / 4) + 64)) != cudaSuccess) return e;
    if ((e = ctx->rg_qual.reserve((size_t)chunk * S + 64)) != cudaSuccess) return e;
    if ((e = ctx->rg_op0.reserve((size_t)chunk * 4 + 64)) != cudaSuccess) return e;
    P.deferred = static_cast<uint32_t*>(ctx->deferred.p);
    P.off3 = static_cast<const uint32_t*>(ctx->rg_off.p);
    if (ctx->layout.infer_q) {
      if ((e = ctx->rg_okmap.reserve(((size_t)chunk + 63) / 64 * 8 + 64)) != cudaSuccess) return e;
      P.okmap = static_cast<uint32_t*>(ctx->rg_okmap.p);
    }
    ctx->profile_batches++;
    timer_begin(ctx, stream);
    for (uint64_t c0 = 0; c0 < b.n_reads; c0 += chunk) {
      const uint64_t cn = std::min<uint64_t>(chunk, b.n_reads - c0);
      RepackParams R;
      R.b = b; R.first_read = c0; R.n_reads = cn; R.S = S;
      R.bases_out = static_cast<uint32_t*>(ctx->rg_bases.p);
      R.qual_out = static_cast<uint32_t*>(ctx->rg_qual.p);
      R.op0_out = static_cast<uint32_t*>(ctx->rg_op0.p);
      R.off3 = static_cast<uint32_t*>(ctx->rg_off.p);
      const uint32_t rgrid = (uint32_t)((cn + PS_TILE_READS - 1) / PS_TILE_READS);
      if (nw == 1) profile_repack_kernel<1><<<rgrid, PS_TILE_READS, 0, stream>>>(R);
      else if (nw == 2) profile_repack_kernel<2><<<rgrid, PS_TILE_READS, 0, stream>>>(R);
      else if (nw == 3) profile_repack_kernel<3><<<rgrid, PS_TILE_READS, 0, stream>>>(R);
      else profile_repack_kernel<4><<<rgrid, PS_TILE_READS, 0, stream>>>(R);
      ctx->launches++;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
      ProfileParams Q = P;
      Q.b.n_reads = cn;
      Q.b.meta = b.meta + c0; Q.b.ref_start = b.ref_start + c0;
      Q.b.cigar = R.op0_out;
      Q.b.bases2 = reinterpret_cast<const uint8_t*>(R.bases_out);
      Q.b.qual = reinterpret_cast<const uint8_t*>(R.qual_out);
      Q.b.tile_exc_off = b.tile_exc_off + c0 / PS_TILE_READS;
      Q.b.uniform_len = S; Q.b.uniform_ncigar = 1;
      Q.first_read = c0;
      Q.off3 = nullptr;
      const uint32_t n_wt = (uint32_t)((cn + WT_READS - 1) / WT_READS);
      // (the row length S = 16 * nw is a compile-time constant of these instantiations)
      if (nw == 1) e = launch_fast<1, 6, 16, true>(ctx, Q, n_wt, stream);
      else if (nw == 2) e = launch_fast<2, 6, 32, true>(ctx, Q, n_wt, stream);
      else if (nw == 3) e = launch_fast<3, 5, 48, true>(ctx, Q, n_wt, stream);
      else e = launch_fast<4, 5, 64, true>(ctx, Q, n_wt, stream);
      if (e != cudaSuccess) return e;
      if (P.okmap && (e = launch_qhist(ctx, Q.b.qual, Q.b.meta, P.okmap, cn, S, 0, P.acc, stream)) != cudaSuccess) return e;
    }
    e = launch_deferred(ctx, P, stream);
    timer_end(ctx, stream);
    return e;
  }
  timer_begin(ctx, stream);
  const cudaError_t e = launch_generic(ctx, P, done, stream);
  timer_end(ctx, stream);
  return e;
}
