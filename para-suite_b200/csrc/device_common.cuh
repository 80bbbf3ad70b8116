// Device helpers shared by the profile and pileup kernels (sm_100a).
#pragma once
#include <cstdint>

#include "internal.h"

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

// htsjdk Cigar.getReferenceLength: M, D, N, =, X consume the reference
__device__ __forceinline__ bool op_consumes_ref(uint32_t op) { return (0x18Du >> op) & 1u; }   // bits 0,2,3,7,8
__device__ __forceinline__ bool op_is_match(uint32_t op) { return (0x181u >> op) & 1u; }       // M, =, X

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
