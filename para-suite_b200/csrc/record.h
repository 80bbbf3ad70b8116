// The CIGAR rules the tools share, on the host and on the device: which ops consume the reference, which are alignment
// blocks, the shape of a record's CIGAR and the walk over its alignment blocks.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

// htsjdk Cigar.getReferenceLength: M, D, N, =, X consume the reference
__host__ __device__ __forceinline__ bool op_consumes_ref(uint32_t op) { return (0x18Du >> op) & 1u; }   // bits 0,2,3,7,8
__host__ __device__ __forceinline__ bool op_is_match(uint32_t op) { return (0x181u >> op) & 1u; }       // M, =, X

__host__ __device__ __forceinline__ uint32_t cigar_at(const uint32_t* cig, uint32_t e) {
#ifdef __CUDA_ARCH__
  return __ldg(cig + e);
#else
  return cig[e];
#endif
}

// Span: the type the reference length is summed in.  The kernels and the pileup keys take 32 bits, as Java's int does;
// the clust writer's sequence assembly sums in 64.
template <typename Span = uint32_t>
struct CigarShape {
  Span ref_span;       // reference length (M, D, N, =, X)
  uint32_t aligned;    // bases in M/=/X blocks
  uint32_t blocks;     // M/=/X ops
  bool skip;           // an I or D together with an N: the pileup drops the record (PileupClusters.java:152-157)
};

template <typename Span = uint32_t>
__host__ __device__ __forceinline__ CigarShape<Span> cigar_shape(const uint32_t* cig, uint32_t ncig) {
  CigarShape<Span> s{0, 0, 0, false};
  bool hasI = false, hasD = false, hasN = false;
  for (uint32_t e = 0; e < ncig; ++e) {
    const uint32_t c = cigar_at(cig, e), op = c & 15u;
    hasI |= op == 1u; hasD |= op == 2u; hasN |= op == 3u;
    if (op_consumes_ref(op)) s.ref_span += c >> 4;
    if (op_is_match(op)) { s.aligned += c >> 4; ++s.blocks; }
  }
  s.skip = (hasI || hasD) && hasN;
  return s;
}

// Alignment blocks (SAMUtils.getAlignmentBlocks): S and I advance the read, D and N the reference, M/=/X both, H and P
// nothing.  f(read_pos, ref_off, len) runs for every M/=/X block in CIGAR order; it returns false to stop the walk.
template <typename F>
__host__ __device__ __forceinline__ void for_each_block(const uint32_t* cig, uint32_t ncig, F&& f) {
  int64_t rdp = 0, rfp = 0;
  for (uint32_t e = 0; e < ncig; ++e) {
    const uint32_t c = cigar_at(cig, e), op = c & 15u;
    const int64_t n = c >> 4;
    if (op == 4u || op == 1u) { rdp += n; continue; }
    if (op == 2u || op == 3u) { rfp += n; continue; }
    if (!op_is_match(op)) continue;
    if (!f(rdp, rfp, n)) return;
    rdp += n; rfp += n;
  }
}
