// Device helpers shared by the profile, pileup and track kernels (sm_100a).
#pragma once
#include <cstdint>

#include "internal.h"

// ---- chained launches (launch_chained, internal.h) ---------------------------------------------------------------
// Both are no-ops in a grid launched without programmatic stream serialization.  pdl_wait returns once the preceding
// grid of the stream has completed and its writes are visible; every chained kernel calls it before its first access to
// anything an earlier kernel writes or reads, and on every path before it exits (the next grid's wait covers only this
// one).  pdl_launch_dependents lets the next grid become resident; that grid still waits for this one to complete.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Timer stamps of the chained kernels (no event may sit between them): %globaltimer in ns.  A pair of words that start
// at 0 holds [0] = ~(earliest start), [1] = latest end, both kept with atomicMax.
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void stamp_start(unsigned long long* w) { atomicMax(w, ~globaltimer_ns()); }
__device__ __forceinline__ void stamp_end(unsigned long long* w) { atomicMax(w, globaltimer_ns()); }

// 2-bit reference code at global offset g (undefined where the invalid bit is set)
__device__ __forceinline__ uint32_t ref_code_at(const DeviceRef& ref, uint64_t g) {
  return (__ldg(ref.seq2 + (g >> 4)) >> (2 * (g & 15))) & 3u;
}
__device__ __forceinline__ bool ref_invalid_at(const DeviceRef& ref, uint64_t g) {
  return (__ldg(ref.inv + (g >> 5)) >> (g & 31)) & 1u;
}
// 2-bit read code at position p of a read whose packed bases start at `b`
__device__ __forceinline__ uint32_t read_code_at(const uint8_t* b, uint32_t p) {
  return (__ldg(b + (p >> 2)) >> (2 * (p & 3))) & 3u;
}

__device__ __forceinline__ void raise_fault(unsigned long long* fault, uint64_t ordinal, uint32_t code) {
  atomicMin(fault, (unsigned long long)((ordinal << 8) | code));
}

// contig index of global offset g (contig_off has n_contigs+1 entries, ascending)
__device__ __forceinline__ uint32_t contig_of(const DeviceRef& ref, uint64_t g) {
  uint32_t lo = 0, hi = ref.n_contigs;  // invariant: contig_off[lo] <= g < contig_off[hi]
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (__ldg(ref.contig_off + mid) <= g) lo = mid; else hi = mid;
  }
  return lo;
}

struct ContigCache {         // contig bounds of the last read looked up by this thread
  uint64_t lo = 1, hi = 0;
  uint32_t idx = 0;
  uint32_t rank = 0;         // position of contig idx in the input's sort order (the pileup keys)
};
struct ContigCache32 {       // same in 32 bits (the global coordinate space is < 2^32 bases: set_contigs in ctx.cu)
  uint32_t lo = 0, hi = 0;     // empty: hi - lo == 0, no offset passes the one-compare range test
  uint32_t idx = 0;
  uint32_t rank = 0;
};
__device__ __forceinline__ bool contig_lookup(const DeviceRef& ref, uint32_t g0, ContigCache32& c) {
  if (g0 - c.lo < c.hi - c.lo) return true;       // lo <= g0 < hi in one unsigned compare
  if (g0 >= ref.n_bases) return false;
  c.idx = contig_of(ref, g0);
  c.lo = (uint32_t)__ldg(ref.contig_off + c.idx);
  c.hi = (uint32_t)__ldg(ref.contig_off + c.idx + 1);
  c.rank = __ldg(ref.contig_rank + c.idx);
  return true;
}
__device__ __forceinline__ bool contig_lookup(const DeviceRef& ref, uint64_t g0, ContigCache& c) {
  if (g0 >= c.lo && g0 < c.hi) return true;
  if (g0 >= ref.n_bases) return false;
  c.idx = contig_of(ref, g0);
  c.lo = __ldg(ref.contig_off + c.idx);
  c.hi = __ldg(ref.contig_off + c.idx + 1);
  c.rank = __ldg(ref.contig_rank + c.idx);
  return true;
}

// per-read stream offsets (bytes of packed bases, bytes of qualities, cigar elements)
struct ReadOffsets {
  uint64_t base, qual, cigar;
};

// Stream offsets of the reads of one warp chunk [q, q+32) (lane l holds read r = q + l; `in` = r exists), without a
// block barrier: tile tables + the metas between the tile start and the chunk + a warp scan.  A chunk may straddle one
// tile boundary.  Warp-collective: all 32 lanes must call.
__device__ __forceinline__ ReadOffsets warp_read_offsets(const DeviceBatch& b, uint64_t q, uint64_t r, bool in, uint32_t meta) {
  ReadOffsets o;
  if (b.uniform_len && b.uniform_ncigar) {
    o.base = r * (uint64_t)((b.uniform_len + 3) >> 2);
    o.qual = r * (uint64_t)b.uniform_len;
    o.cigar = r * (uint64_t)b.uniform_ncigar;
    return o;
  }
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t t0 = q / PS_TILE_READS;
  // L | bytes << 25 | cigar ops << 48 (a tile holds 256 reads of L <= 65535 and <= 255 ops: no field overflows)
  auto pack = [](uint32_t m) {
    const uint64_t L = PS_META_LEN(m);
    return L | (((L + 3) >> 2) << 25) | ((uint64_t)PS_META_NCIGAR(m) << 48);
  };
  uint64_t pre = 0;
  for (uint64_t j = t0 * PS_TILE_READS + lane; j < q; j += 32) pre += pack(__ldg(b.meta + j));
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) pre += __shfl_xor_sync(0xFFFFFFFFu, pre, d);
  const uint64_t mine = in ? pack(meta) : 0ull;
  uint64_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t y = __shfl_up_sync(0xFFFFFFFFu, inc, d);
    if (lane >= (uint32_t)d) inc += y;
  }
  const uint64_t ex = inc - mine;
  const uint64_t my_tile = r / PS_TILE_READS;
  const uint32_t crossed = __ballot_sync(0xFFFFFFFFu, my_tile != t0);
  uint64_t rel = pre + ex, tile = t0;
  if (crossed) {
    const int bl = __ffs((int)crossed) - 1;            // first lane of the next tile
    const uint64_t exb = __shfl_sync(0xFFFFFFFFu, ex, bl);
    if (my_tile != t0) { rel = ex - exb; tile = t0 + 1; }
  }
  o.base = 0; o.qual = 0; o.cigar = 0;
  if (!in) return o;
  if (b.uniform_len) {
    o.base = r * (uint64_t)((b.uniform_len + 3) >> 2);
    o.qual = r * (uint64_t)b.uniform_len;
  } else {
    o.base = __ldg(b.tile_base_off + tile) + ((rel >> 25) & 0x7FFFFFu);
    o.qual = __ldg(b.tile_qual_off + tile) + (rel & 0x1FFFFFFu);
  }
  o.cigar = b.uniform_ncigar ? r * (uint64_t)b.uniform_ncigar : __ldg(b.tile_cigar_off + tile) + (rel >> 48);
  return o;
}

// 16 bits -> the even bits of a 32-bit word
__device__ __forceinline__ uint32_t spread16_even(uint32_t h) {
  h &= 0xFFFFu;
  h = (h | (h << 8)) & 0x00FF00FFu;
  h = (h | (h << 4)) & 0x0F0F0F0Fu;
  h = (h | (h << 2)) & 0x33333333u;
  h = (h | (h << 1)) & 0x55555555u;
  return h;
}

// Exception list (non-ACGT base calls) of one read: the tile's list is sorted by (read_in_tile << 16 | position), so a
// read's entries are one contiguous run [e0, e1), found once per read with two binary searches.
struct ExcRange { uint32_t e0, e1; };
__device__ __forceinline__ uint32_t exc_lower_bound(const uint32_t* exc, uint32_t lo, uint32_t hi, uint32_t key) {
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(exc + mid) < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ ExcRange read_exc_range(const DeviceBatch& b, uint64_t tile, uint32_t rit) {
  const uint32_t lo = __ldg(b.tile_exc_off + tile), hi = __ldg(b.tile_exc_off + tile + 1);
  ExcRange r;
  r.e0 = exc_lower_bound(b.exc, lo, hi, rit << 16);
  r.e1 = exc_lower_bound(b.exc, r.e0, hi, (rit + 1u) << 16);
  return r;
}
// is position p of the read listed as an invalid base?  (a read holds a handful of entries at most)
__device__ __forceinline__ bool read_pos_invalid(const DeviceBatch& b, ExcRange r, uint32_t p) {
  for (uint32_t e = r.e0; e < r.e1; ++e)
    if ((__ldg(b.exc + e) & 0xFFFFu) == p) return true;
  return false;
}
// the listed positions p < 64 of read r as a forward bit mask (bit p): the bit-parallel T>C paths clear them, whatever
// code the producer stored there.  Call for reads with PS_RF_HAS_INVALID only.  One search for the read's first entry,
// then a scan over its (few) entries.
__device__ __forceinline__ unsigned long long read_exc_mask64(const DeviceBatch& b, uint64_t r) {
  const uint64_t tile = r / PS_TILE_READS;
  const uint32_t rit = (uint32_t)(r % PS_TILE_READS), hi = __ldg(b.tile_exc_off + tile + 1);
  unsigned long long m = 0;
  for (uint32_t e = exc_lower_bound(b.exc, __ldg(b.tile_exc_off + tile), hi, rit << 16); e < hi; ++e) {
    const uint32_t v = __ldg(b.exc + e);
    if ((v >> 16) != rit) break;
    if ((v & 0xFFFFu) < 64u) m |= 1ull << (v & 0xFFFFu);
  }
  return m;
}

// even bits of c -> low 16 bits
__device__ __forceinline__ uint32_t even_bits(uint32_t c) {
  c &= 0x55555555u;
  c = (c | (c >> 1)) & 0x33333333u;
  c = (c | (c >> 2)) & 0x0F0F0F0Fu;
  c = (c | (c >> 4)) & 0x00FF00FFu;
  c = (c | (c >> 8)) & 0x0000FFFFu;
  return c;
}

// Bit-parallel T>C events of a read of length L <= 64 whose one M/=/X op covers it, in genome orientation (bit j = read
// position j): ref T (11) and read C (01) on the plus strand, ref A (00) and read G (10) on the minus strand.  w: the
// reference words from g0 >> 4 on, bw: the read's words, bsh: the bit offset of its first base in bw[0].  The positions
// over a reference N, from L on, and (has_exc: the read has entries in `exc`) of listed N calls are cleared: the codes
// stored there are arbitrary.  ref_n: the reference-N window of the read, same orientation.
struct T2cWord { unsigned long long t2c, ref_n; };
template <int NW>
__device__ __forceinline__ T2cWord t2c_word(const DeviceRef& ref, const DeviceBatch& b, uint64_t r, uint32_t g0, uint32_t L,
                                            bool rev, bool has_exc, const uint32_t (&w)[NW + 1],
                                            const uint32_t (&bw)[NW + 1], uint32_t bsh) {
  const uint32_t sh = (g0 & 15u) * 2u, ii = g0 >> 5, s1 = g0 & 31u;
  const uint32_t i0 = __ldg(ref.inv + ii), i1 = __ldg(ref.inv + ii + 1), i2 = NW > 2 ? __ldg(ref.inv + ii + 2) : 0u;
  unsigned long long m = 0;
#pragma unroll
  for (int j = 0; j < NW; ++j) {
    const uint32_t rf = __funnelshift_r(w[j], w[j + 1], sh);
    const uint32_t rd = __funnelshift_r(bw[j], bw[j + 1], bsh);
    const uint32_t h = rev ? (~(rf | (rf >> 1)) & (rd >> 1) & ~rd) : (rf & (rf >> 1) & rd & ~(rd >> 1));
    m |= (unsigned long long)even_bits(h) << (16 * j);
  }
  T2cWord t;
  t.ref_n = (unsigned long long)__funnelshift_r(i0, i1, s1) |
            ((unsigned long long)(NW > 2 ? __funnelshift_r(i1, i2, s1) : 0u) << 32);
  m &= ~t.ref_n;
  m &= L >= 64 ? ~0ull : ((1ull << L) - 1ull);
  if (has_exc && m) m &= ~read_exc_mask64(b, r);      // only a read with a candidate event needs its list
  t.t2c = m;
  return t;
}
