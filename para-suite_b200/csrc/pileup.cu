// K2/K3: T>C conversion pileup.  Replaces the loop PileupClusters.java:137-500 and
// calculateClusterInformation :585-673 (reference: /root/reference/src/src/utils/pileupclusters/).
//
// Three stages over one coordinate-sorted SoA batch; every output record is assembled on the device:
//
//   flag stage         the only ORDERED step, kept as light as possible (12 B/read: meta, ref_start, cigar):
//       per read       filter (P1), (contig, start, end)
//       running max    of (contig, end) over all earlier reads = the cluster end the Java loop holds (tempClusterEnd)
//                      -> boundary flag (clusterEnd - start) < 5 or contig changed (P2)
//       prefix sum     of the flags = cluster slot; the opening read's index goes to cl_first[slot]
//     one-op-per-read batches: pl_flag_kernel<16, true> (no dependency between tiles: the running max in front of a
//     tile is taken over a halo of 128 reads and recorded), pl_flag_scan_kernel (one block: exact prefixes over the
//     tile table, every assumption checked -- a failed one makes the host repeat the call with the exact kernel),
//     pl_flag_expand_kernel (flag words + tile prefix -> cl_first).  Other batches and the fallback:
//     pl_flag_kernel<.., false>, two decoupled look-backs over 16-byte single-word descriptors.
//   pl_cluster_kernel  one block = 64 consecutive clusters = one contiguous run of reads, no inter-block dependency:
//       thread per read      T>C bit mask over the concatenated alignment blocks (P3) -- bit-parallel on 2-bit packed
//                            words for the PAR-CLIP shape (uniform length, one M op), a literal CIGAR walk otherwise --
//                            decoded into shared memory; T>C positions ORed into the cluster's 64-position key set
//       per cluster          reads, T>C count, end, 51-bit position mask, strand state (P4, P6)
//       thread per read      mutationMap values, first-insertion key and baseCoveredMap at the keys (P3, P7): native
//                            shared-memory atomics, slot = rank of the key in the key set (position order)
//       thread per cluster   64-byte record and the sites; the block takes ONE run of site slots with one atomic
//       warp per cluster     what does not fit (> 1024 reads, > 6 keys, keys > 64 apart): warp ballots for <= 32 reads,
//                            else a streaming sweep over a sliding ring of positions, else window tables
//   pl_compact_kernel  site runs into (cluster, position) order; the prefix over the per-cluster site counts comes from
//                      per-tile totals the cluster kernel adds up (a look-back past 2 M cluster slots)
//
// The flush-time logic (SNP filter, anchor site, text rows: :178-344) stays on the host side of the boundary.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "device_common.cuh"
#include "lookback.cuh"

void timer_begin(ps_ctx* ctx, cudaStream_t st);
void timer_end(ps_ctx* ctx, cudaStream_t st);
int stage_batch(ps_ctx* ctx, const ps_read_batch* hb, bool with_qual, StagedBatch** out);

namespace {

constexpr int PL_THREADS = 256;
constexpr int PL_WARPS = PL_THREADS / 32;
// pl_cluster_kernel tuning (overridable with -D for side-by-side variants: tools/build_variants.sh)
#ifndef CB_THREADS_
#define CB_THREADS_ 128
#endif
#ifndef CB_CLUSTERS_
#define CB_CLUSTERS_ 64
#endif
#ifndef CB_CHUNK_
#define CB_CHUNK_ 1024
#endif
#ifndef CB_BLOCKS_PER_SM
#define CB_BLOCKS_PER_SM 8
#endif
constexpr int CB_THREADS = CB_THREADS_;               // threads per block of pl_cluster_kernel
constexpr int CB_WARPS = CB_THREADS / 32;
constexpr int CB_CLUSTERS = CB_CLUSTERS_;             // clusters per block of pl_cluster_kernel
constexpr int CB_CHUNK = CB_CHUNK_;                   // reads decoded into shared memory at a time
constexpr int CB_SITES = 6;                           // distinct T>C positions per cluster kept in shared memory
#ifndef FLAG_THREADS_
#define FLAG_THREADS_ 128
#endif
#ifndef FLAG_ITEMS_
#define FLAG_ITEMS_ 16
#endif
#ifndef FLAG_BLOCKS_PER_SM
#define FLAG_BLOCKS_PER_SM 4
#endif
constexpr int FLAG_THREADS = FLAG_THREADS_;           // threads per block of pl_flag_kernel
constexpr int FLAG_WARPS = FLAG_THREADS / 32;
constexpr int PL_FLAG_ITEMS = FLAG_ITEMS_;            // reads per thread of pl_flag_kernel on the vector path
constexpr int PL_WINDOW = 128;                        // positions per window

struct PlState {                  // device-side run state (one per call)
  unsigned long long fault;       // min over (ordinal << 8 | code); ~0 = none
  unsigned long long skipped;     // skippedDueIndel (:156)
  unsigned long long dstr;        // doubleStranded (:496)
  unsigned long long n_sites;     // site slots handed out by pl_cluster_kernel (>= the number of sites: upper bounds)
  unsigned long long n_sites_final;   // distinct (cluster, position), written by pl_compact_kernel
  unsigned int n_flags;           // clusters opened
  unsigned int unsorted;
  unsigned int tile_ctr_flag;
  unsigned int tile_ctr_compact;
  unsigned int first_slot1;       // first read of slot 1 (end of the head partial); n_reads if there is no slot 1
  unsigned int spec_failed;       // the speculative flag pass used a carry-in that pl_flag_scan_kernel found too small
  ps_cluster head, open;          // final records of slot 0 and of the last slot (written by pl_compact_kernel)
  // PARASUITE_B200_DEBUG, counted by the warp routine over clusters with at least one T>C event: [0] clusters the
  // ballot form could not take (the streaming sweep starts on them), [1] of those, the ones the sweep gave up on,
  // [2] window passes the window loop made over them (one per PL_WINDOW positions from the first event to the last)
  unsigned long long dbg[3];
  // timer stamps of the chained kernels (device_common.cuh), cleared by pl_init_state: ~start of the flag, cluster and
  // compaction stages (earliest block past its pdl_wait), end of the compaction
  unsigned long long ts[4];
};

struct PlRead {              // what the pileup needs from one read
  unsigned long long mask;   // T>C by index i over the strand-oriented concatenated blocks
  int32_t start, end;        // alignment start / end (1-based, contig coordinates)
  int32_t lo, hi;            // checkPosition interval (baseCoveredMap support)
  uint32_t contig;
  bool kept, rev;
};

// ---------------------------------------------------------------------------------------------------------
// pl_flag_kernel
// ---------------------------------------------------------------------------------------------------------
struct FlagParams {
  DeviceBatch b;
  DeviceRef ref;
  PlState* st;
  LbDesc* d_max;
  LbDesc* d_cnt;
  unsigned int epoch;
  uint32_t n_tiles;
  unsigned long long carry_key;
  const unsigned long long* carry_keys;   // device: keys of the preceding shards (may be null)
  uint32_t carry_keys_n;
  uint32_t* cl_first;       // [cap_cl + 2] first read of each slot; slot 0 = reads continuing the carry-in cluster
  uint64_t cap_cl;
  // speculative three-kernel path (pl_flag_kernel<.., true>, pl_flag_scan_kernel, pl_flag_expand_kernel)
  unsigned long long* tile_ein;   // [n_tiles] carry-in every tile assumed: maximum over the FLAG_HALO reads in front of it
  unsigned long long* tile_agg;   // [n_tiles] maximum over the tile's own reads
  uint32_t* tile_cnt;             // [n_tiles] boundary flags per tile, then (scan kernel) their exclusive prefix
  uint32_t* flag_words;           // one word per thread (bit j = read j of the thread)
  uint32_t scan_in_expand;        // no pl_flag_scan_kernel: the expand kernel sums the tile counts itself
  uint32_t stamp;                 // stamp PlState::ts
};

// (rank of the contig + 1) << 32 | end of a kept record, 0 otherwise (PileupClusters.java:146-158).  The rank is the
// contig's position in the input's sort order (DeviceRef::contig_rank), so that the running maximum of the keys follows
// the records across a contig change whatever order the file lists its contigs in.
template <bool COUNT = true>
__device__ __forceinline__ unsigned long long pl_key(const FlagParams& P, uint64_t r, uint32_t meta, const uint32_t* cig,
                                                     uint32_t g0, ContigCache& cc, int32_t& start) {
  const uint32_t flags = PS_META_FLAGS(meta);
  start = 0;
  if (flags & PS_RF_UNMAPPED) return 0;                                      // :146
  const CigarShape<> s = cigar_shape(cig, PS_META_NCIGAR(meta));
  if (s.skip) {                                                              // :152-157
    if (COUNT) atomicAdd(&P.st->skipped, 1ull);
    return 0;
  }
  if (flags & (PS_RF_POS_ZERO | PS_RF_CIGAR_OVERFLOW)) return 0;   // the JVM dies on the first, the second cannot be held:
                                                                   // pl_cluster_kernel raises the fault
  if (!contig_lookup(P.ref, g0, cc)) return 0;    // likewise
  start = (int32_t)((uint64_t)g0 - cc.lo) + 1;
  const int32_t end = start + (int32_t)s.ref_span - 1;
  return ((unsigned long long)(cc.rank + 1) << 32) | (uint32_t)end;
}

// same for a record with exactly one cigar op `cg` (a lone I or D next to no N is kept: :152-157 needs both)
template <typename CC>
__device__ __forceinline__ unsigned long long pl_key1(const FlagParams& P, uint32_t meta, uint32_t cg, uint32_t g0,
                                                      CC& cc, int32_t& start) {
  // straight-line on purpose (16 reads per thread are unrolled around this: early returns cost a convergence
  // barrier each); only the contig table walk of a cache miss is a branch
  const uint32_t flags = PS_META_FLAGS(meta);
  bool ok = (flags & (PS_RF_UNMAPPED | PS_RF_POS_ZERO | PS_RF_CIGAR_OVERFLOW)) == 0;
  if (ok) ok = contig_lookup(P.ref, g0, cc);
  const uint32_t R = op_consumes_ref(cg & 15u) ? cg >> 4 : 0u;
  const int32_t s = (int32_t)(g0 - (uint32_t)cc.lo) + 1;      // offsets inside a contig fit 32 bits (the whole reference does)
  start = ok ? s : 0;
  const unsigned long long key = ((unsigned long long)(cc.rank + 1) << 32) | (uint32_t)(s + (int32_t)R - 1);
  return ok ? key : 0ull;
}

// max over the records of a batch of (contig rank, end): what a following shard needs as carry-in (region sharding: the
// exclusive prefix-max of these keys over the shards replaces Java's (tempClusterChr, tempClusterEnd) at the cut)
__global__ void __launch_bounds__(PL_THREADS) pl_maxkey_kernel(const __grid_constant__ FlagParams P, unsigned long long* out) {
  ContigCache cc;
  unsigned long long best = 0;
  const uint64_t n = P.b.n_reads;
  for (uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); q < n; q += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = q + (threadIdx.x & 31u);
    const bool in = r < n;
    const uint32_t meta = in ? __ldg(P.b.meta + r) : PS_MAKE_META(0, 0, PS_RF_UNMAPPED);
    const ReadOffsets off = warp_read_offsets(P.b, q, r, in, meta);
    if (!in) continue;
    int32_t start;
    const unsigned long long k = pl_key<false>(P, r, meta, P.b.cigar + off.cigar, __ldg(P.b.ref_start + r), cc, start);
    best = k > best ? k : best;
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, best, d); best = o > best ? o : best; }
  if ((threadIdx.x & 31u) == 0 && best) atomicMax(out, best);
}

// block-wide exclusive scan over one 64-bit value per thread (PL_THREADS threads); also returns the block total
template <typename Op, int WARPS = PL_WARPS>
__device__ __forceinline__ unsigned long long block_exclusive(unsigned long long v, Op op, unsigned long long identity,
                                                              unsigned long long* warp_tot /* [WARPS] smem */,
                                                              unsigned long long& total) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, x, d);
    if (lane >= (uint32_t)d) x = op(y, x);
  }
  if (lane == 31) warp_tot[warp] = x;
  __syncthreads();
  unsigned long long prefix = identity, tot = identity;
#pragma unroll
  for (uint32_t w = 0; w < (uint32_t)WARPS; ++w) {
    const unsigned long long t = warp_tot[w];
    if (w < warp) prefix = op(prefix, t);
    tot = op(tot, t);
  }
  total = tot;
  unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, x, 1);
  if (lane == 0) up = identity;
  __syncthreads();
  return op(prefix, up);
}

// ITEMS == PL_FLAG_ITEMS: every read has one cigar op and the streams are 16-byte aligned (vector loads);
// ITEMS == 1: any batch (per-read cigar offsets from the tile tables)
// SPEC (vector path only): the two chained look-backs are what the exact kernel waits for (every tile needs the running
// maximum of ALL earlier tiles, then the flag count of all earlier tiles).  In a coordinate-sorted batch the running
// maximum in front of a tile is, bar a record reaching over more than FLAG_HALO of its successors, the maximum over the
// FLAG_HALO reads in front of it: the speculative variant loads those next to its own reads (no dependency between
// tiles at all), records the carry-in it assumed, its own aggregate, flag bits and a per-tile count;
// pl_flag_scan_kernel (one block) takes the exact prefixes over the tile table and checks every assumption (a failed
// one makes the host repeat the call with the exact variant); pl_flag_expand_kernel writes cl_first.
constexpr int FLAG_HALO = FLAG_THREADS;     // one read in front of the tile per thread
template <int ITEMS, bool SPEC>
__global__ void __launch_bounds__(FLAG_THREADS, FLAG_BLOCKS_PER_SM) pl_flag_kernel(const __grid_constant__ FlagParams P) {
  constexpr int TILE = FLAG_THREADS * ITEMS;
  static_assert(!SPEC || ITEMS > 1, "the speculative pass is built for the vector path");
  __shared__ unsigned long long s_wtot[FLAG_WARPS];
  __shared__ unsigned long long s_halo[FLAG_WARPS];
  __shared__ unsigned int s_tile;
  __shared__ unsigned long long s_pre;
  pdl_wait();
  pdl_launch_dependents();
  if (P.stamp && threadIdx.x == 0) stamp_start(&P.st->ts[0]);

  if constexpr (!SPEC) {      // the look-backs need forward progress: tile numbers in the order the blocks start
    if (threadIdx.x == 0) s_tile = atomicAdd(&P.st->tile_ctr_flag, 1u);
    __syncthreads();
  }
  const uint32_t tile = SPEC ? blockIdx.x : s_tile;
  const uint64_t n = P.b.n_reads;
  const uint64_t r0 = (uint64_t)tile * TILE + (uint64_t)threadIdx.x * ITEMS;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  unsigned long long key[ITEMS];
  int32_t start[ITEMS];
  typename std::conditional<(ITEMS > 1), ContigCache32, ContigCache>::type cc;
  [[maybe_unused]] uint32_t h_meta = PS_MAKE_META(0, 0, PS_RF_UNMAPPED), h_start = 0, h_cig = 0;
  if constexpr (SPEC) {       // one read of the halo per thread, requested together with the tile's own reads
    const uint64_t t0 = (uint64_t)tile * TILE;
    if (t0 + threadIdx.x >= (uint64_t)FLAG_HALO) {
      const uint64_t hr = t0 + threadIdx.x - FLAG_HALO;          // < t0 <= n
      h_meta = __ldg(P.b.meta + hr); h_start = __ldg(P.b.ref_start + hr); h_cig = __ldg(P.b.cigar + hr);
    }
  }
  if constexpr (ITEMS > 1) {
    static_assert(ITEMS % 4 == 0, "vector loads take 4 reads at a time");
#pragma unroll
    for (int g = 0; g < ITEMS; g += 4) {
      uint32_t metas[4], starts[4], cigs[4];
      const uint64_t rg = r0 + g;
      if (rg + 4 <= n) {
        const uint4 m4 = __ldg(reinterpret_cast<const uint4*>(P.b.meta + rg));
        const uint4 s4 = __ldg(reinterpret_cast<const uint4*>(P.b.ref_start + rg));
        const uint4 c4 = __ldg(reinterpret_cast<const uint4*>(P.b.cigar + rg));
        metas[0] = m4.x; metas[1] = m4.y; metas[2] = m4.z; metas[3] = m4.w;
        starts[0] = s4.x; starts[1] = s4.y; starts[2] = s4.z; starts[3] = s4.w;
        cigs[0] = c4.x; cigs[1] = c4.y; cigs[2] = c4.z; cigs[3] = c4.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool in = rg + j < n;
          metas[j] = in ? __ldg(P.b.meta + rg + j) : PS_MAKE_META(0, 0, PS_RF_UNMAPPED);
          starts[j] = in ? __ldg(P.b.ref_start + rg + j) : 0u;
          cigs[j] = in ? __ldg(P.b.cigar + rg + j) : 0u;
        }
      }
      // four reads at a time: when none of them needs the contig table (all kept ones lie in the cached contig -- every
      // group but a thread's first, bar contig changes) keys and starts are straight-line code
      bool need = false;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        need |= ((PS_META_FLAGS(metas[j]) & (PS_RF_UNMAPPED | PS_RF_POS_ZERO | PS_RF_CIGAR_OVERFLOW)) == 0) & !(starts[j] - cc.lo < cc.hi - cc.lo);
      if (!need) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool ok = (PS_META_FLAGS(metas[j]) & (PS_RF_UNMAPPED | PS_RF_POS_ZERO | PS_RF_CIGAR_OVERFLOW)) == 0;
          const uint32_t R = op_consumes_ref(cigs[j] & 15u) ? cigs[j] >> 4 : 0u;
          const int32_t st = (int32_t)(starts[j] - cc.lo) + 1;
          start[g + j] = ok ? st : 0;
          key[g + j] = ok ? (((unsigned long long)(cc.rank + 1) << 32) | (uint32_t)(st + (int32_t)R - 1)) : 0ull;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) key[g + j] = pl_key1(P, metas[j], cigs[j], starts[j], cc, start[g + j]);
      }
    }
  } else {
    const bool in_range = r0 < n;
    const uint32_t meta = in_range ? __ldg(P.b.meta + r0) : PS_MAKE_META(0, 0, PS_RF_UNMAPPED);
    const ReadOffsets off = warp_read_offsets(P.b, (uint64_t)tile * TILE + (threadIdx.x & ~31u), r0, in_range, meta);
    key[0] = in_range ? pl_key(P, r0, meta, P.b.cigar + off.cigar, __ldg(P.b.ref_start + r0), cc, start[0]) : 0ull;
    if (!in_range) start[0] = 0;
  }

  // ---- look-back #1: running max of (contig rank, end) -----------------------------------------------------------
  unsigned long long tmax = 0;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) tmax = key[j] > tmax ? key[j] : tmax;
  if constexpr (SPEC) {
    int32_t hs;
    unsigned long long hk = pl_key1(P, h_meta, h_cig, h_start, cc, hs);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, hk, d); hk = o > hk ? o : hk; }
    if (lane == 0) s_halo[warp] = hk;           // read after the barriers of the scan below
  }
  unsigned long long block_max;
  const unsigned long long ex_max = block_exclusive<LbMax, FLAG_WARPS>(tmax, LbMax(), 0ull, s_wtot, block_max);
  if (warp == 0) {
    if constexpr (SPEC) {
      unsigned long long pre = lane < FLAG_WARPS ? s_halo[lane] : 0ull;
#pragma unroll
      for (int d = FLAG_WARPS / 2; d >= 1; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, pre, d); pre = o > pre ? o : pre; }
      if (lane == 0) { s_pre = pre; P.tile_ein[tile] = pre; P.tile_agg[tile] = block_max; }
    } else if (tile == 0) {
      if (lane == 0) { lb_publish(&P.d_max[0], block_max, 2u, P.epoch); s_pre = 0; }
    } else {
      if (lane == 0) lb_publish(&P.d_max[tile], block_max, 1u, P.epoch);
      const unsigned long long pre = lb_exclusive_prefix(P.d_max, (int)tile, P.epoch, LbMax(), 0ull);
      if (lane == 0) {
        lb_publish(&P.d_max[tile], pre > block_max ? pre : block_max, 2u, P.epoch);
        s_pre = pre;
      }
    }
  }
  __syncthreads();
  unsigned long long E = s_pre > ex_max ? s_pre : ex_max;
  E = E > P.carry_key ? E : P.carry_key;
  for (uint32_t k = 0; k < P.carry_keys_n; ++k) {        // a handful of shards: every thread reads them (L1 broadcast)
    const unsigned long long ck = __ldg(P.carry_keys + k);
    E = E > ck ? E : ck;
  }

  // ---- boundary flags (:175-176) ---------------------------------------------------------------------------------
  uint32_t fl = 0, nfl = 0;
  bool unsorted = false;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const unsigned long long my = key[j];
    const bool kept = my != 0;
    const uint32_t pc = (uint32_t)(E >> 32), mc = (uint32_t)(my >> 32);
    // tempClusterEnd = 0, tempClusterChr = "" (:118-120) | contig changed | (clusterEnd - start) < 5; predicated, no branches
    const bool f = kept & ((E == 0) | (pc != mc) | (((int64_t)(int32_t)(uint32_t)E - (int64_t)start[j]) < 5));
    unsorted |= kept & (pc > mc);                       // contig order went backwards: not coordinate sorted (in the
                                                        // order the keys follow: ps_reference_set_contig_order)
    E = my > E ? my : E;                                // my == 0 leaves E alone
    fl |= (uint32_t)f << j;
    nfl += (uint32_t)f;
  }
  if (unsorted) P.st->unsorted = 1u;
  if constexpr (SPEC) {
    P.flag_words[(size_t)tile * FLAG_THREADS + threadIdx.x] = fl;
    const uint32_t wsum = __reduce_add_sync(0xFFFFFFFFu, nfl);
    if (lane == 0) s_wtot[warp] = wsum;          // the scan is done with s_wtot (its second barrier is behind us)
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t c = 0;
#pragma unroll
      for (int w = 0; w < FLAG_WARPS; ++w) c += (uint32_t)s_wtot[w];
      P.tile_cnt[tile] = c;
    }
    return;
  }
  __syncthreads();   // s_pre is reused below

  // ---- look-back #2: cluster slots ---------------------------------------------------------------------------------
  unsigned long long block_cnt;
  const unsigned long long ex_cnt = block_exclusive<LbSum, FLAG_WARPS>((unsigned long long)nfl, LbSum(), 0ull, s_wtot, block_cnt);
  if (warp == 0) {
    if (tile == 0) {
      if (lane == 0) { lb_publish(&P.d_cnt[0], block_cnt, 2u, P.epoch); s_pre = 0; }
    } else {
      if (lane == 0) lb_publish(&P.d_cnt[tile], block_cnt, 1u, P.epoch);
      const unsigned long long pre = lb_exclusive_prefix(P.d_cnt, (int)tile, P.epoch, LbSum(), 0ull);
      if (lane == 0) {
        lb_publish(&P.d_cnt[tile], pre + block_cnt, 2u, P.epoch);
        s_pre = pre;
      }
    }
  }
  __syncthreads();
  uint64_t slot = s_pre + ex_cnt;     // flags before this thread's first read
  if (tile == 0 && threadIdx.x == 0) P.cl_first[0] = 0;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j)
    if ((fl >> j) & 1u) {
      ++slot;
      if (slot < P.cap_cl) P.cl_first[slot] = (uint32_t)(r0 + j);
      if (slot == 1) P.st->first_slot1 = (unsigned int)(r0 + j);
    }
  if (tile == P.n_tiles - 1 && threadIdx.x == FLAG_THREADS - 1) {
    if (slot + 1 <= P.cap_cl) P.cl_first[slot + 1] = (uint32_t)n;   // slots 0 .. n_flags, the last one is the open cluster
    P.st->n_flags = (unsigned int)slot;
  }
}

// One block over the tile table of the speculative flag pass: exact running maximum in front of every tile (checked
// against the carry-in the tile assumed) and exclusive prefix of the per-tile flag counts.
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 8;        // consecutive tiles per thread and round
__global__ void __launch_bounds__(SCAN_THREADS) pl_flag_scan_kernel(const __grid_constant__ FlagParams P) {
  __shared__ unsigned long long s_wtot[SCAN_THREADS / 32];
  pdl_wait();
  pdl_launch_dependents();
  unsigned long long carry = P.carry_key;
  for (uint32_t k = 0; k < P.carry_keys_n; ++k) {
    const unsigned long long ck = __ldg(P.carry_keys + k);
    carry = carry > ck ? carry : ck;
  }
  unsigned long long run_max = 0, run_cnt = 0;
  bool bad = false;
  for (uint64_t c0 = 0; c0 < P.n_tiles; c0 += (uint64_t)SCAN_THREADS * SCAN_ITEMS) {
    const uint64_t t0 = c0 + (uint64_t)threadIdx.x * SCAN_ITEMS;
    unsigned long long agg[SCAN_ITEMS], ein[SCAN_ITEMS];
    uint32_t cnt[SCAN_ITEMS];
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
      const bool in = t0 + j < P.n_tiles;
      agg[j] = in ? P.tile_agg[t0 + j] : 0ull;
      ein[j] = in ? P.tile_ein[t0 + j] : 0ull;
      cnt[j] = in ? P.tile_cnt[t0 + j] : 0u;
    }
    unsigned long long tmax = 0, tcnt = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) { tmax = agg[j] > tmax ? agg[j] : tmax; tcnt += cnt[j]; }
    unsigned long long tot_max, tot_cnt;
    unsigned long long m = block_exclusive<LbMax, SCAN_THREADS / 32>(tmax, LbMax(), 0ull, s_wtot, tot_max);
    unsigned long long c = block_exclusive<LbSum, SCAN_THREADS / 32>(tcnt, LbSum(), 0ull, s_wtot, tot_cnt) + run_cnt;
    m = m > run_max ? m : run_max;
    m = m > carry ? m : carry;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j)
      if (t0 + j < P.n_tiles) {
        const unsigned long long used = ein[j] > carry ? ein[j] : carry;
        bad |= m != used;                         // m = exact running maximum in front of tile t0 + j
        P.tile_cnt[t0 + j] = (uint32_t)c;
        m = agg[j] > m ? agg[j] : m;
        c += cnt[j];
      }
    run_max = run_max > tot_max ? run_max : tot_max;
    run_cnt += tot_cnt;
  }
  if (bad) P.st->spec_failed = 1u;
  if (threadIdx.x == 0) {
    P.cl_first[0] = 0;
    if (run_cnt + 1 <= P.cap_cl) P.cl_first[run_cnt + 1] = (uint32_t)P.b.n_reads;   // slots 0 .. n_flags, the last one is the open cluster
    P.st->n_flags = (unsigned int)run_cnt;
  }
}

// cl_first from the flag bits and the per-tile prefix (same tiling as the flag kernel).
// P.scan_in_expand (tile tables of up to kFlagSumTiles entries): there is no scan kernel in front of this one; every
// block adds up the counts of the tiles in front of it itself and checks its own tile's assumption LOCALLY --
// assumed(t) == max(assumed(t-1), aggregate(t-1)) for every t is, by induction from assumed(0) = carry, the same as
// assumed(t) == exact running maximum -- and the last tile's block writes the totals.
template <int ITEMS>
__global__ void __launch_bounds__(FLAG_THREADS) pl_flag_expand_kernel(const __grid_constant__ FlagParams P) {
  __shared__ unsigned long long s_wtot[FLAG_WARPS];
  __shared__ unsigned long long s_base;
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tile = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t fl = P.flag_words[(size_t)tile * FLAG_THREADS + threadIdx.x];
  unsigned long long part = 0;
  if (P.scan_in_expand)
    for (uint32_t t = threadIdx.x; t < tile; t += FLAG_THREADS) part += P.tile_cnt[t];
  unsigned long long total;
  const unsigned long long ex = block_exclusive<LbSum, FLAG_WARPS>((unsigned long long)__popc(fl), LbSum(), 0ull, s_wtot, total);
  unsigned long long base;
  if (P.scan_in_expand) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, d);
    if (lane == 0) s_wtot[warp] = part;          // block_exclusive is done with s_wtot
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long b = 0;
#pragma unroll
      for (int w = 0; w < FLAG_WARPS; ++w) b += s_wtot[w];
      s_base = b;
      unsigned long long carry = P.carry_key;
      for (uint32_t k = 0; k < P.carry_keys_n; ++k) {
        const unsigned long long ck = __ldg(P.carry_keys + k);
        carry = carry > ck ? carry : ck;
      }
      if (tile > 0) {
        unsigned long long used = P.tile_ein[tile], prev = P.tile_ein[tile - 1];
        const unsigned long long agg = P.tile_agg[tile - 1];
        used = used > carry ? used : carry;
        prev = prev > carry ? prev : carry;
        prev = prev > agg ? prev : agg;
        if (used != prev) P.st->spec_failed = 1u;
      }
      if (tile == P.n_tiles - 1) {
        const unsigned long long n_flags = b + total;
        P.cl_first[0] = 0;
        if (n_flags + 1 <= P.cap_cl) P.cl_first[n_flags + 1] = (uint32_t)P.b.n_reads;   // slots 0 .. n_flags, the last one is the open cluster
        P.st->n_flags = (unsigned int)n_flags;
      }
    }
    __syncthreads();
    base = s_base;
  } else {
    base = P.tile_cnt[tile];                     // exclusive prefix, left by pl_flag_scan_kernel
  }
  if (total == 0) return;
  uint64_t slot = base + ex;
  const uint64_t r0 = (uint64_t)tile * (FLAG_THREADS * ITEMS) + (uint64_t)threadIdx.x * ITEMS;
  for (uint32_t w = fl; w; w &= w - 1) {          // about one flag per thread: walk the set bits, not the 16 reads
    const uint32_t j = (uint32_t)__ffs((int)w) - 1u;
    ++slot;
    if (slot < P.cap_cl) P.cl_first[slot] = (uint32_t)(r0 + j);
    if (slot == 1) P.st->first_slot1 = (unsigned int)(r0 + j);
  }
}

// ---------------------------------------------------------------------------------------------------------
// per-read decode for pl_cluster_kernel
// ---------------------------------------------------------------------------------------------------------
struct ClusterParams {
  DeviceBatch b;
  DeviceRef ref;
  PlState* st;
  uint32_t first_id;
  const uint32_t* cl_first;
  ps_cluster* cl;
  ps_site* sites;           // pl_cluster_kernel: sites grouped by block in completion order; pl_compact_kernel orders them
  uint64_t cap_cl, cap_sites;
  unsigned int* tile_sites;   // [slots / COMPACT_TILE] sites per tile of pl_compact_kernel (zeroed by the host), or nullptr
  const unsigned long long* t2c_mask;   // optional: one T>C mask word per read, left by profile_fast_kernel for THIS batch
                                        // (bit 63 valid, bit 62 minus strand, bits 0..61 mask by strand-oriented index)
  uint32_t stamp;                       // pl_cluster_kernel: stamp PlState::ts
};
#ifndef COMPACT_ITEMS_
#define COMPACT_ITEMS_ 2
#endif
constexpr int COMPACT_ITEMS = COMPACT_ITEMS_;
constexpr int COMPACT_TILE = PL_THREADS * COMPACT_ITEMS;     // cluster slots per block of pl_compact_kernel
static_assert(COMPACT_TILE % CB_CLUSTERS == 0, "a block of pl_cluster_kernel lies inside one tile of pl_compact_kernel");

// Literal per-read routine (any CIGAR, any flag): PileupClusters.java:146-158, :585-673
__device__ __noinline__ void pl_decode_generic(const ClusterParams& P, uint64_t r, uint32_t meta, uint64_t off_base,
                                               uint64_t off_cigar, PlRead& x) {
  const uint32_t flags = PS_META_FLAGS(meta), L = PS_META_LEN(meta), ncig = PS_META_NCIGAR(meta);
  const uint32_t* cig = P.b.cigar + off_cigar;
  x.kept = false; x.mask = 0; x.start = 0; x.end = 0; x.lo = 1; x.hi = 0; x.rev = false; x.contig = 0;
  if (flags & PS_RF_UNMAPPED) return;                                        // :146
  if (flags & PS_RF_CIGAR_OVERFLOW) { raise_fault(&P.st->fault, r, PS_FAULT_CIGAR_OPS); return; }   // not representable
  const CigarShape<> sh = cigar_shape(cig, ncig);
  const uint32_t alen = sh.aligned;
  if (sh.skip) return;                                                       // :152-157 (counted by pl_flag_kernel)
  if (flags & PS_RF_POS_ZERO) { raise_fault(&P.st->fault, r, PS_THROW_REF_RANGE); return; }
  const uint64_t g0 = __ldg(P.b.ref_start + r);
  if (g0 >= P.ref.n_bases) { raise_fault(&P.st->fault, r, PS_THROW_REF_RANGE); return; }
  const uint32_t contig = contig_of(P.ref, g0);
  const uint64_t c_lo = __ldg(P.ref.contig_off + contig), c_hi = __ldg(P.ref.contig_off + contig + 1);
  const int32_t start = (int32_t)(g0 - c_lo) + 1;
  const int32_t end = start + (int32_t)sh.ref_span - 1;
  const bool rev = flags & PS_RF_REVERSE;
  const bool has_inv = flags & PS_RF_HAS_INVALID;
  const uint8_t* rb = P.b.bases2 + off_base;
  x.kept = true; x.start = start; x.end = end; x.rev = rev; x.contig = contig;
  if (rev) { x.hi = end; x.lo = end - (int32_t)alen + 1; }
  else { x.lo = start; x.hi = start + (int32_t)alen - 1; }
  // the reference slices every block (read bases, then FASTA) before it looks at a single base (:593-604)
  uint32_t code = 0;
  for_each_block(cig, ncig, [&](int64_t rdp, int64_t rfp, int64_t n) {
    if (rdp + n > (int64_t)L) code = PS_THROW_BLOCK_RANGE;
    else if ((flags & PS_RF_REF_RANGE) || g0 + (uint64_t)(rfp + n) > c_hi) code = PS_THROW_REF_RANGE;
    return code == 0;
  });
  if (code) { raise_fault(&P.st->fault, r, code); return; }
  uint32_t j = 0;             // index over the concatenated blocks (forward orientation)
  unsigned long long mask = 0;
  bool over = false;
  for_each_block(cig, ncig, [&](int64_t rdp, int64_t rfp, int64_t n) {
    for (int64_t z = 0; z < n; ++z, ++j) {
      const uint64_t g = g0 + (uint64_t)(rfp + z);
      const uint32_t p = (uint32_t)(rdp + z);
      if (ref_invalid_at(P.ref, g)) continue;
      const uint32_t a = ref_code_at(P.ref, g), bb = read_code_at(rb, p);
      // minus strand: both arrays are reverse-complemented, so ref T & read C there is ref A & read G here
      const bool hit = rev ? (a == 0u && bb == 2u) : (a == 3u && bb == 1u);
      if (!hit) continue;
      if (has_inv && read_pos_invalid(P.b, read_exc_range(P.b, r / PS_TILE_READS, (uint32_t)(r % PS_TILE_READS)), p)) continue;
      const uint32_t i = rev ? alen - 1 - j : j;
      if (i >= 51u) { raise_fault(&P.st->fault, r, PS_THROW_MASK51); over = true; return false; }   // boolean[51] (:654)
      mask |= 1ull << i;
    }
    return true;
  });
  if (!over) x.mask = mask;
}

// PAR-CLIP shape: uniform length L <= 64, one M/=/X op of length L.  The T>C word in strand orientation
// (i = alignedLength - 1 - j on the minus strand); bw: the read's words, loaded ahead (pl_load_raw)
template <int NW>
__device__ __forceinline__ unsigned long long t2c_mask_fast(const DeviceRef& ref, uint32_t g0, uint32_t L, bool rev,
                                                            const uint32_t (&bw)[NW + 1], uint32_t bshift,
                                                            const DeviceBatch& b, uint64_t r, bool has_inv) {
  uint32_t w[NW + 1];
#pragma unroll
  for (int k = 0; k <= NW; ++k) w[k] = __ldg(ref.seq2 + (g0 >> 4) + k);
  unsigned long long m = t2c_word<NW>(ref, b, r, g0, L, rev, has_inv, w, bw, bshift).t2c;
  if (rev) m = __brevll(m) >> (64u - L);
  return m;
}

// the words of one record that do not depend on anything else: loaded one read ahead of their use (PAR-CLIP shape).
// MK: the profile kernel left a T>C mask word per read (ClusterParams::t2c_mask): the record is its offset and that word
template <int NW, bool MK>
struct PlRaw {
  uint32_t meta, g0, cg;
  uint32_t bw[NW > 0 ? NW + 1 : 1];
};
template <int NW>
struct PlRaw<NW, true> {
  uint32_t g0;
  unsigned long long mk;
};
template <int NW, bool MK>
__device__ __forceinline__ PlRaw<NW, MK> pl_load_raw(const ClusterParams& P, uint64_t r, bool in) {
  PlRaw<NW, MK> w;
  if constexpr (MK) {
    w.g0 = in ? __ldg(P.b.ref_start + r) : 0u;
    w.mk = in ? __ldg(P.t2c_mask + r) : 0ull;
  } else {
    w.meta = in ? __ldg(P.b.meta + r) : 0u;
    w.g0 = 0; w.cg = 0;
    if constexpr (NW > 0) {
#pragma unroll
      for (int k = 0; k <= NW; ++k) w.bw[k] = 0;
      if (in) {
        w.g0 = __ldg(P.b.ref_start + r);
        w.cg = __ldg(P.b.cigar + r);
        const uint64_t boff = r * (uint64_t)((P.b.uniform_len + 3) >> 2);
        const uint32_t* src = reinterpret_cast<const uint32_t*>(P.b.bases2 + (boff & ~3ull));
#pragma unroll
        for (int k = 0; k <= NW; ++k) w.bw[k] = __ldg(src + k);
      }
    }
  }
  return w;
}

// one lane decodes read r (r < n); NW > 0: the batch has the PAR-CLIP shape and most reads take the bit-parallel path
template <int NW, bool MK, typename CC>
__device__ __forceinline__ void pl_decode(const ClusterParams& P, uint64_t q, uint64_t r, bool in, const PlRaw<NW, MK>& raw,
                                          CC& cc, PlRead& x) {
  x.kept = false; x.mask = 0; x.start = 0; x.end = 0; x.lo = 1; x.hi = 0; x.rev = false; x.contig = 0;
  if constexpr (MK) {
    static_assert(NW > 0, "mask words exist for the PAR-CLIP shape only");
    if (!in) return;
    const uint32_t L = P.b.uniform_len, bpr = (L + 3) >> 2;
    const unsigned long long mk = raw.mk;
    // a valid word: the profile kernel saw flags in {REVERSE, HAS_INVALID}, one M op of length L and the whole read
    // inside one contig -- everything the bit-parallel path below asks for
    if ((mk >> 63) && contig_lookup(P.ref, raw.g0, cc)) {
      const unsigned long long m = mk & ((1ull << 62) - 1ull);
      const int32_t start = (int32_t)((uint64_t)raw.g0 - cc.lo) + 1, end = start + (int32_t)L - 1;
      if (L > 51u && (m >> 51)) { raise_fault(&P.st->fault, r, PS_THROW_MASK51); return; }
      x.kept = true; x.mask = m; x.start = start; x.end = end; x.lo = start; x.hi = end; x.rev = (mk >> 62) & 1ull;
      x.contig = cc.idx;
      return;
    }
    PlRead t;
    pl_decode_generic(P, r, __ldg(P.b.meta + r), r * (uint64_t)bpr, r, t);
    x = t;
  } else {
    const uint32_t meta = raw.meta;
    if constexpr (NW > 0) {
      if (!in) return;
      const uint32_t L = P.b.uniform_len, bpr = (L + 3) >> 2;
      const uint32_t flags = PS_META_FLAGS(meta), g0 = raw.g0, cg = raw.cg;
      // N calls are cleared from the mask by their `exc` entries (the code stored under them is arbitrary);
      // duplicates are not filtered by this tool and qualities are never read
      constexpr uint32_t kHarmless = PS_RF_REVERSE | PS_RF_HAS_INVALID | PS_RF_DUPLICATE | PS_RF_QUAL_MISSING;
      bool fast = (flags & ~kHarmless) == 0 && op_is_match(cg & 15u) && (cg >> 4) == L && PS_META_LEN(meta) == L;
      fast = fast && contig_lookup(P.ref, g0, cc) && (uint64_t)g0 + L <= cc.hi;
      if (fast) {
        const bool rev = (flags & PS_RF_REVERSE) != 0;
        const uint64_t boff = r * (uint64_t)bpr;
        unsigned long long m = t2c_mask_fast<NW>(P.ref, g0, L, rev, raw.bw, (uint32_t)(boff & 3u) * 8u, P.b, r,
                                                 (flags & PS_RF_HAS_INVALID) != 0);
        const int32_t start = (int32_t)((uint64_t)g0 - cc.lo) + 1, end = start + (int32_t)L - 1;
        if (L > 51u && (m >> 51)) { raise_fault(&P.st->fault, r, PS_THROW_MASK51); return; }
        x.kept = true; x.mask = m; x.start = start; x.end = end; x.lo = start; x.hi = end; x.rev = rev; x.contig = cc.idx;
        return;
      }
      PlRead t;               // the literal routine takes its result by address: keep x itself in registers
      pl_decode_generic(P, r, meta, r * (uint64_t)bpr, r, t);
      x = t;
    } else {
      const ReadOffsets off = warp_read_offsets(P.b, q, r, in, meta);    // warp-collective
      if (in) pl_decode_generic(P, r, meta, off.base, off.cigar, x);
    }
  }
}
template <int NW, bool MK = false>
__device__ __forceinline__ void pl_decode(const ClusterParams& P, uint64_t q, uint64_t r, bool in, ContigCache& cc, PlRead& x) {
  pl_decode<NW, MK>(P, q, r, in, pl_load_raw<NW, MK>(P, r, in), cc, x);
}

// ---------------------------------------------------------------------------------------------------------
// pl_cluster_kernel
// ---------------------------------------------------------------------------------------------------------
struct WarpTables {     // one window of PL_WINDOW positions
  int32_t diff[PL_WINDOW];            // +1 at lo, -1 after hi  -> prefix sum = baseCoveredMap
  uint32_t cnt[PL_WINDOW];            // mutationMap
  unsigned long long first[PL_WINDOW];   // min over events of (read << 6 | i) = first insertion
};

constexpr int PL_RING = 256;          // positions of the sliding window of the streaming sweep (power of two)
struct WarpRing {
  int32_t diff[PL_RING];
  uint32_t cnt[PL_RING];
  unsigned long long first[PL_RING];
};

__device__ __forceinline__ uint32_t warp_or(uint32_t v) { return __reduce_or_sync(0xFFFFFFFFu, v); }

// One cluster = reads [f, fe) (slot `slot`), whole warp.  Fills *rec (shared memory) when `fill`, writes up to `cap`
// sites to `dest` in position order and returns the number of sites the cluster has.
template <int NW, bool MK>
__device__ __noinline__ uint32_t pl_cluster(const ClusterParams& P, uint32_t slot, uint32_t f, uint32_t fe, WarpTables& T,
                                            WarpRing& G, ps_cluster* rec, bool fill, ps_site* dest, uint32_t cap,
                                            unsigned long long& dstr, unsigned long long* site_base = nullptr) {
  const uint32_t lane = threadIdx.x & 31;
  ContigCache cc;
  PlRead x;
  // ---- aggregates (P3 counters, P4, P6) ----------------------------------------------------------------------
  uint32_t reads = 0, t2c = 0, minus = 0, first_rev = 0, contig = 0;
  int32_t end = INT32_MIN, cstart = 0, ev_min = INT32_MAX, ev_max = INT32_MIN;
  unsigned long long mask = 0, first_read = f;
  bool have_first = false;
  for (uint32_t q = f; q < fe; q += 32) {
    const uint32_t r = q + lane;
    pl_decode<NW, MK>(P, q, r, r < fe, cc, x);
    const uint32_t kb = __ballot_sync(0xFFFFFFFFu, x.kept);
    if (kb == 0) continue;
    if (!have_first) {
      const int fl = __ffs((int)kb) - 1;
      first_read = q + fl;
      cstart = __shfl_sync(0xFFFFFFFFu, x.start, fl);
      contig = __shfl_sync(0xFFFFFFFFu, x.contig, fl);
      first_rev = __shfl_sync(0xFFFFFFFFu, (uint32_t)x.rev, fl);
      have_first = true;
    }
    reads += __popc(kb);
    minus += __popc(__ballot_sync(0xFFFFFFFFu, x.kept && x.rev));
    end = max(end, __reduce_max_sync(0xFFFFFFFFu, x.kept ? x.end : INT32_MIN));
    const uint32_t any = __ballot_sync(0xFFFFFFFFu, x.mask != 0);
    if (any) {
      t2c += __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popcll(x.mask));
      mask |= (unsigned long long)warp_or((uint32_t)x.mask) | ((unsigned long long)warp_or((uint32_t)(x.mask >> 32)) << 32);
      int32_t lo_e = INT32_MAX, hi_e = INT32_MIN;
      if (x.mask) {
        const int ia = __ffsll((long long)x.mask) - 1, ib = 63 - __clzll((long long)x.mask);
        lo_e = x.rev ? x.hi - ib : x.lo + ia;
        hi_e = x.rev ? x.hi - ia : x.lo + ib;
      }
      ev_min = min(ev_min, __reduce_min_sync(0xFFFFFFFFu, lo_e));
      ev_max = max(ev_max, __reduce_max_sync(0xFFFFFFFFu, hi_e));
    }
  }
  if (fill && lane == 0) {
    const uint32_t maf = slot ? minus - first_rev : minus;   // slot 0 continues a cluster opened by the preceding shard
    rec->first_read = first_read;
    rec->running_id = slot ? P.first_id + slot : 0;          // runningID++ then "cl_<id>_<chr>" (:355): first cluster is cl_2
    rec->contig = contig;
    rec->start = cstart;
    rec->end = reads ? end : 0;
    rec->num_reads = reads;
    rec->num_t2c = t2c;
    rec->minus_after_first = maf;
    rec->first_reverse = (uint8_t)first_rev;
    // StrandOrientation state at flush (P6): minus-first -> "-"; plus-first -> "+/-" once a minus member came
    rec->combined_strand = first_rev ? 1 : (maf ? 2 : 0);
    rec->reserved = 0;
    rec->mask51 = mask;
    rec->site_begin = 0;
    rec->site_end = 0;
    if (slot && !first_rev) dstr += maf;                     // doubleStranded++ (:494-498), incl. the never-flushed last cluster
  }
  if (t2c == 0) return 0;
  if (site_base) {
    // the caller wants the sites written in ONE pass: take an upper bound of slots (events, or positions between the
    // first and the last event) from the block-order site array; pl_compact_kernel drops the unused ones
    const unsigned long long ub = min((unsigned long long)t2c, (unsigned long long)((int64_t)ev_max - (int64_t)ev_min + 1));
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&P.st->n_sites, ub);
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    *site_base = base;
    dest = P.sites + base;
    cap = base < P.cap_sites ? (uint32_t)min(ub, P.cap_sites - base) : 0u;
  }

  // ---- sites: one chunk of reads, all events inside one window -> warp ballots, no shared memory ----------------
  if (fe - f <= 32 && (int64_t)ev_max - (int64_t)ev_min < PL_WINDOW) {
    // x still holds this lane's read
    uint32_t pm[4] = {0, 0, 0, 0};
    unsigned long long m = x.mask;
    while (m) {
      const int i = __ffsll((long long)m) - 1;
      m &= m - 1;
      const uint32_t rel = (uint32_t)((x.rev ? x.hi - i : x.lo + i) - ev_min);   // checkPosition (:638-643)
      const uint32_t bit = 1u << (rel & 31u);
      const uint32_t w = rel >> 5;
      pm[0] |= w == 0 ? bit : 0u; pm[1] |= w == 1 ? bit : 0u; pm[2] |= w == 2 ? bit : 0u; pm[3] |= w == 3 ? bit : 0u;
    }
    uint32_t n_sites = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      uint32_t u = warp_or(pm[w]);
      while (u) {
        const int b = __ffs((int)u) - 1;
        u &= u - 1;
        const int32_t pos = ev_min + 32 * w + b;
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, (pm[w] >> b) & 1u);
        const int fl = __ffs((int)bal) - 1;
        const uint32_t cov = __popc(__ballot_sync(0xFFFFFFFFu, x.kept && x.lo <= pos && pos <= x.hi));
        const uint32_t i_me = (uint32_t)(x.rev ? x.hi - pos : pos - x.lo);
        const uint32_t i_first = __shfl_sync(0xFFFFFFFFu, i_me, fl);
        if (lane == 0 && n_sites < cap) {
          ps_site s;
          s.pos = pos; s.t2c = __popc(bal); s.cov = cov; s.reserved = 0;
          s.order_key = ((unsigned long long)(f + fl) << 6) | i_first;
          dest[n_sites] = s;
        }
        ++n_sites;
      }
    }
    return n_sites;
  }

  if (lane == 0) atomicAdd(&P.st->dbg[0], 1ull);
  // ---- sites: streaming sweep (any number of reads, one decode per read) ------------------------------------------
  // Records are sorted by start and no read touches a position before its own start, so every position before the
  // start of the read being added is final: a ring of PL_RING positions slides along the cluster, finished positions
  // are emitted (in position order) and their slots recycled.  Gives up -- and leaves the cluster to the window loop
  // below -- if starts ever go backwards (input not sorted inside a contig) or a single read is longer than the ring.
  {
    for (uint32_t k = lane; k < PL_RING; k += 32) { G.diff[k] = 0; G.cnt[k] = 0; G.first[k] = ~0ull; }
    __syncwarp();
    uint32_t written = 0;
    int32_t wlo = 0, carry = 0;          // first position not yet emitted; coverage just before it
    bool started = false, ok = true;
    auto flush_to = [&](int32_t upto) {  // emit positions [wlo, upto)
      const int64_t stop = min((int64_t)upto, (int64_t)wlo + PL_RING);     // nothing beyond the ring was ever touched
      for (int64_t p0 = wlo; p0 < stop; p0 += 32) {
        const int64_t pp = p0 + lane;
        const bool in = pp < stop;
        const uint32_t sl = (uint32_t)pp & (PL_RING - 1);
        int32_t c = in ? G.diff[sl] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int32_t y = __shfl_up_sync(0xFFFFFFFFu, c, d);
          if (lane >= (uint32_t)d) c += y;
        }
        c += carry;
        carry = __shfl_sync(0xFFFFFFFFu, c, 31);
        const uint32_t n = in ? G.cnt[sl] : 0u;
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, n != 0);
        const uint32_t at = written + __popc(bal & ((1u << lane) - 1u));
        if (n && at < cap) {
          ps_site s;
          s.pos = (int32_t)pp; s.t2c = n; s.cov = (uint32_t)c; s.reserved = 0; s.order_key = G.first[sl];
          dest[at] = s;
        }
        written += __popc(bal);
        if (in) { G.diff[sl] = 0; G.cnt[sl] = 0; G.first[sl] = ~0ull; }
      }
      wlo = upto;
      __syncwarp();
    };
    for (uint32_t q = f; q < fe && ok; q += 32) {
      const uint32_t r = q + lane;
      pl_decode<NW, MK>(P, q, r, r < fe, cc, x);
      uint32_t pending = __ballot_sync(0xFFFFFFFFu, x.kept);
      while (pending) {
        const bool mine = (pending >> lane) & 1u;
        const int32_t bstart = __reduce_min_sync(0xFFFFFFFFu, mine ? x.start : INT32_MAX);
        if (!started) { wlo = bstart; started = true; }
        if (bstart < wlo) { ok = false; break; }
        flush_to(bstart);
        const uint32_t fits = __ballot_sync(0xFFFFFFFFu, mine && (int64_t)x.hi + 2 - (int64_t)wlo <= PL_RING && x.lo >= wlo);
        const uint32_t first_pending = (uint32_t)__ffs((int)pending) - 1u;
        if (!((fits >> first_pending) & 1u)) { ok = false; break; }        // one read longer than the ring
        const uint32_t misfit = pending & ~fits;
        const uint32_t take = misfit ? pending & ((1u << ((uint32_t)__ffs((int)misfit) - 1u)) - 1u) : pending;
        if ((take >> lane) & 1u) {
          unsigned long long m = x.mask;
          while (m) {
            const int i = __ffsll((long long)m) - 1;
            m &= m - 1;
            const uint32_t sl = (uint32_t)(x.rev ? x.hi - i : x.lo + i) & (PL_RING - 1);
            atomicAdd(&G.cnt[sl], 1u);
            atomicMin(&G.first[sl], ((unsigned long long)r << 6) | (unsigned)i);
          }
          atomicAdd(&G.diff[(uint32_t)x.lo & (PL_RING - 1)], 1);
          atomicAdd(&G.diff[(uint32_t)(x.hi + 1) & (PL_RING - 1)], -1);
        }
        __syncwarp();
        pending &= ~take;
      }
    }
    if (ok) {
      // tail: every touched position lies inside the ring
      if (started) flush_to((int32_t)min((int64_t)INT32_MAX, (int64_t)wlo + PL_RING));
      return written;
    }
  }

  // ---- sites: per-warp tables, one window of positions at a time (quadratic in the worst case; only reached by
  //      clusters the sweep above gave up on) ---------------------------------------------------------------------------
  uint32_t written = 0;
  if (lane == 0) atomicAdd(&P.st->dbg[1], 1ull);
  for (int64_t w0 = ev_min; w0 <= ev_max; w0 += PL_WINDOW) {
    const int64_t w1 = w0 + PL_WINDOW - 1;
    if (lane == 0) atomicAdd(&P.st->dbg[2], 1ull);
    for (uint32_t k = lane; k < PL_WINDOW; k += 32) { T.diff[k] = 0; T.cnt[k] = 0; T.first[k] = ~0ull; }
    __syncwarp();
    for (uint32_t q = f; q < fe; q += 32) {
      const uint32_t r = q + lane;
      pl_decode<NW, MK>(P, q, r, r < fe, cc, x);
      if (!x.kept || (int64_t)x.hi < w0 || (int64_t)x.lo > w1) continue;
      unsigned long long m = x.mask;
      while (m) {
        const int i = __ffsll((long long)m) - 1;
        m &= m - 1;
        const int64_t d = (int64_t)(x.rev ? x.hi - i : x.lo + i) - w0;
        if (d >= 0 && d < PL_WINDOW) {
          atomicAdd(&T.cnt[d], 1u);
          atomicMin(&T.first[d], ((unsigned long long)r << 6) | (unsigned)i);
        }
      }
      atomicAdd(&T.diff[(int64_t)x.lo > w0 ? (int64_t)x.lo - w0 : 0], 1);
      if ((int64_t)x.hi < w1) atomicAdd(&T.diff[(int64_t)x.hi + 1 - w0], -1);
    }
    __syncwarp();
    int32_t carry = 0;
    for (uint32_t k0 = 0; k0 < PL_WINDOW; k0 += 32) {
      int32_t c = T.diff[k0 + lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int32_t y = __shfl_up_sync(0xFFFFFFFFu, c, d);
        if (lane >= (uint32_t)d) c += y;
      }
      c += carry;
      carry = __shfl_sync(0xFFFFFFFFu, c, 31);
      const uint32_t n = T.cnt[k0 + lane];
      const uint32_t bal = __ballot_sync(0xFFFFFFFFu, n != 0);
      const uint32_t at = written + __popc(bal & ((1u << lane) - 1u));
      if (n && at < cap) {
        ps_site s;
        s.pos = (int32_t)(w0 + k0 + lane);
        s.t2c = n;
        s.cov = (uint32_t)c;
        s.reserved = 0;
        s.order_key = T.first[k0 + lane];
        dest[at] = s;
      }
      written += __popc(bal);
    }
    __syncwarp();
  }
  return written;
}

// Shared-memory plan of pl_cluster_kernel (dynamic): decoded reads of one chunk, per-cluster site tables
struct ClusterSmem {
  unsigned long long* mask;   // [CB_CHUNK] T>C mask | rev << 62 | kept << 63
  int32_t *lo, *hi, *end;     // [CB_CHUNK]
  unsigned long long* umask;  // [CB_CLUSTERS] mutationMap key set: bit p = position base + p holds a T>C
  uint32_t *scnt, *scov, *skey;   // [CB_SITES * CB_CLUSTERS] site s of cluster k at [s * CB_CLUSTERS + k]
  int32_t* base;              // [CB_CLUSTERS] position of bit 0 of umask = start of the read that opened the cluster
  uint32_t* ovf;              // [CB_CLUSTERS] != 0: the cluster does not fit the tables
  uint8_t* cid;               // [CB_CHUNK] cluster (index inside the chunk) of each read
  uint32_t* first;            // [CB_CLUSTERS + 1] cl_first of the block's clusters
  uint32_t* fb;               // [CB_CLUSTERS] clusters left to the warp routine
};
constexpr size_t kClusterAliasBytes = (size_t)CB_CHUNK * (8 + 3 * 4 + 1) + (size_t)CB_CLUSTERS * (8 + CB_SITES * 12 + 2 * 4);
constexpr size_t kClusterSmemBytes = kClusterAliasBytes + (size_t)CB_CLUSTERS * 2 * 4 + 64;
static_assert(kClusterAliasBytes >= CB_WARPS * (sizeof(WarpTables) + sizeof(WarpRing) + sizeof(ps_cluster)),
              "fallback tables alias the read arrays and the site tables (not first / fb)");
static_assert(CB_CLUSTERS <= 256 && CB_THREADS % CB_CLUSTERS == 0 && CB_CHUNK % 4 == 0,
              "cluster index is one byte; CB_SPLIT threads per cluster");
constexpr int CB_SPLIT = CB_THREADS / CB_CLUSTERS;    // threads that share one cluster in the per-cluster phases
static_assert(CB_SPLIT >= 1 && CB_SPLIT <= 32 && (CB_SPLIT & (CB_SPLIT - 1)) == 0, "the CB_SPLIT threads of a cluster are neighbouring lanes");

__device__ __forceinline__ unsigned long long bits_below(int n) { return n >= 64 ? ~0ull : (1ull << n) - 1ull; }

// checkPosition (:638-643) for all T>C indices of a read at once: index ib lies at position lo + ib (plus strand) or
// hi - ib (minus strand).  Returns false when a position falls outside [base, base + 64).
__device__ __forceinline__ bool t2c_positions(unsigned long long mask, bool rev, int32_t lo, int32_t hi, int32_t base,
                                              unsigned long long& bits) {
  bits = 0;
  if (!rev) {
    const int32_t s = lo - base;
    if ((uint32_t)s > 63u) return false;
    bits = mask << s;
    return (bits >> s) == mask;
  }
  const unsigned long long rv = __brevll(mask);          // index ib -> bit 63 - ib; wanted: bit (hi - base) - ib
  const int32_t d = hi - base - 63;
  if (d >= 0) {
    if (d > 63) return false;
    bits = rv << d;
    return (bits >> d) == rv;
  }
  if (d < -63) return false;
  bits = rv >> -d;
  return (bits << -d) == rv;
}

// One block = CB_CLUSTERS consecutive clusters = one contiguous run of reads, taken in chunks of CB_CHUNK reads.
//   pre CB_SPLIT threads per CLUSTER: cluster of every read; origin of the key set = start of the opening read
//   A   thread per READ:    decode (T>C mask, interval, strand) into shared memory -- full lanes whatever the cluster
//                           sizes are -- and OR of the read's T>C positions (two shifts) into its cluster's
//                           64-position key set: shared atomics
//   B0  CB_SPLIT threads per CLUSTER: counters over the cluster's decoded reads (P3 counters, P4, P6)
//   B2  thread per READ:    per T>C: mutationMap count and first-insertion key (min); baseCoveredMap: the keys a read's
//                           interval covers are one run of slots (a key's slot is its rank in the key set, so the
//                           sites come out in position order): +1 / -1 at the ends of the run, summed up in B3
//   B3  thread per CLUSTER: record (64 contiguous bytes per thread) and sites; the block's sites go to one run of
//                           slots taken with a single atomic, pl_compact_kernel orders the runs afterwards
// Clusters that do not fit (more than CB_CHUNK reads, T>C positions more than 64 apart, more than CB_SITES of them)
// are left to the warp-per-cluster routine above at the end of the block.
template <int NW, bool MK>
__global__ void __launch_bounds__(CB_THREADS, CB_BLOCKS_PER_SM) pl_cluster_kernel(const __grid_constant__ ClusterParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long s_wtot[CB_WARPS];
  __shared__ unsigned long long s_base;
  __shared__ uint32_t s_nfb;
  pdl_wait();      // before any path, the early returns included: the mask words are four launches back
  pdl_launch_dependents();
  if (P.stamp && threadIdx.x == 0) stamp_start(&P.st->ts[1]);
  ClusterSmem S;
  S.mask = reinterpret_cast<unsigned long long*>(smem_raw);
  S.lo = reinterpret_cast<int32_t*>(S.mask + CB_CHUNK);
  S.hi = S.lo + CB_CHUNK; S.end = S.hi + CB_CHUNK;
  S.umask = reinterpret_cast<unsigned long long*>(S.end + CB_CHUNK);
  S.scnt = reinterpret_cast<uint32_t*>(S.umask + CB_CLUSTERS);
  S.scov = S.scnt + CB_SITES * CB_CLUSTERS;
  S.skey = S.scov + CB_SITES * CB_CLUSTERS;
  S.base = reinterpret_cast<int32_t*>(S.skey + CB_SITES * CB_CLUSTERS);
  S.ovf = reinterpret_cast<uint32_t*>(S.base + CB_CLUSTERS);
  S.cid = reinterpret_cast<uint8_t*>(S.ovf + CB_CLUSTERS);
  S.first = reinterpret_cast<uint32_t*>(S.cid + CB_CHUNK);
  S.fb = S.first + CB_CLUSTERS + 1;

  const uint32_t c0 = blockIdx.x * CB_CLUSTERS;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // the block's slice of cl_first is requested before the slot count it is checked against arrives (entries past the
  // last slot are never looked at)
  static_assert(CB_CLUSTERS < CB_THREADS, "one cl_first entry per thread");
  const uint32_t f_pre = (tid <= (uint32_t)CB_CLUSTERS && (uint64_t)c0 + tid < P.cap_cl + 2) ? __ldg(P.cl_first + c0 + tid) : 0u;
  const uint32_t n_slots = P.st->n_flags + 1;          // written by the flag stage
  if (n_slots > P.cap_cl) return;                       // the host re-runs the kernels with larger arrays
  if (c0 >= n_slots) return;
  const uint32_t ncl = min((uint32_t)CB_CLUSTERS, n_slots - c0);
  const uint32_t kk = tid / CB_SPLIT, part = tid % CB_SPLIT;    // per-cluster phases: cluster inside the chunk, share
  if (tid <= ncl) S.first[tid] = f_pre;
  if (tid == 0) s_nfb = 0;
  __syncthreads();

  unsigned long long dstr = 0;
  unsigned long long blk_sites = 0;     // sites of this block's clusters (identical in every thread until the warp routine)
  ContigCache32 cc;
  uint32_t cur = 0;
  while (cur < ncl) {
    const uint32_t rs = S.first[cur];
    // clusters cur .. cur+ncomp-1 lie completely inside the chunk [rs, rs + CB_CHUNK)
    const bool complete = cur + tid < ncl && S.first[cur + tid + 1] - rs <= (uint32_t)CB_CHUNK;
    const uint32_t ncomp = (uint32_t)__syncthreads_count(complete);
    if (ncomp == 0) {           // a single cluster larger than the chunk
      if (tid == 0) S.fb[s_nfb++] = cur;
      ++cur;
      __syncthreads();
      continue;
    }
    const uint32_t re = S.first[cur + ncomp], nrd = re - rs;
    const bool mine = kk < ncomp, owner = mine && part == 0;
    // the first round's record words are requested before the pre-pass, whose own loads they overlap
    PlRaw<NW, MK> nxt = pl_load_raw<NW, MK>(P, rs + warp * 32 + lane, rs + warp * 32 + lane < re);
    // ---- pre-pass, per cluster: cluster of every read, origin of the key set -----------------------------------------
    uint32_t ra = 0, rb = 0, op_contig = 0;
    int32_t base = 0;
    if (mine) {
      const uint32_t k = cur + kk;
      ra = S.first[k] - rs; rb = S.first[k + 1] - rs;
      for (uint32_t i = ra + part; i < rb; i += CB_SPLIT) S.cid[i] = (uint8_t)kk;
      if (part == 0) {
        // sorted input: no position of a cluster lies before the start of the read that opened it, and that read is
        // the cluster's first kept one (pl_flag_kernel flags kept reads only).  Slot 0, the reads continuing the
        // preceding shard's cluster, has no opener: it is left to the warp routine
        if (c0 + k != 0) {
          const uint32_t g0 = __ldg(P.b.ref_start + S.first[k]);
          if (contig_lookup(P.ref, g0, cc)) { base = (int32_t)((uint64_t)g0 - cc.lo) + 1; op_contig = cc.idx; }
        }
        S.base[kk] = base;
        S.umask[kk] = 0;
        S.ovf[kk] = (c0 + k == 0 && rb > ra) ? 1u : 0u;
#pragma unroll
        for (int u = 0; u < CB_SITES; ++u) {
          S.scnt[u * CB_CLUSTERS + kk] = 0; S.scov[u * CB_CLUSTERS + kk] = 0; S.skey[u * CB_CLUSTERS + kk] = 0xFFFFFFFFu;
        }
      }
    }
    __syncthreads();
    // ---- A, thread per read: decode; T>C positions into the cluster's key set -------------------------------------
    for (uint32_t q = rs + warp * 32; q < re; q += CB_THREADS) {
      const uint32_t r = q + lane;
      const PlRaw<NW, MK> raw = nxt;
      // one round in flight: a second one costs registers, and the kernel gains more from 8 resident blocks per SM
      // (measured: 2 rounds at 8 / 7 / 6 blocks 0.52 / 0.31 / 0.32 ms against 0.28 ms)
      if (q + CB_THREADS < re) nxt = pl_load_raw<NW, MK>(P, r + CB_THREADS, r + CB_THREADS < re);   // in flight during this decode
      PlRead x;
      pl_decode<NW, MK>(P, q, r, r < re, raw, cc, x);
      if (r < re) {
        const uint32_t i = r - rs;
        S.mask[i] = x.mask | ((unsigned long long)x.rev << 62) | ((unsigned long long)x.kept << 63);
        S.lo[i] = x.lo; S.hi[i] = x.hi; S.end[i] = x.end;
        if (x.mask) {
          const uint32_t k = S.cid[i];
          unsigned long long bits;
          if (!t2c_positions(x.mask, x.rev, x.lo, x.hi, S.base[k], bits)) S.ovf[k] = 1u;
          else {
            // two native 32-bit atomics (a 64-bit OR on shared memory is a compare-and-swap loop)
            uint32_t* um32 = reinterpret_cast<uint32_t*>(&S.umask[k]);
            if ((uint32_t)bits) atomicOr(um32, (uint32_t)bits);
            if ((uint32_t)(bits >> 32)) atomicOr(um32 + 1, (uint32_t)(bits >> 32));
          }
        }
      }
    }
    __syncthreads();
    // ---- B0, per cluster: counters -----------------------------------------------------------------------------------
    uint32_t reads = 0, t2c = 0, minus = 0, first_rev = 0;
    int32_t end = INT32_MIN;
    unsigned long long mask = 0;
    if (mine) {
      for (uint32_t i = ra + part; i < rb; i += CB_SPLIT) {
        unsigned long long m = S.mask[i];
        if (!(m >> 63)) continue;
        ++reads; minus += (uint32_t)(m >> 62) & 1u;
        end = max(end, S.end[i]);
        m &= (1ull << 51) - 1ull;
        t2c += __popcll(m);
        mask |= m;
      }
      if (part == 0 && rb > ra) first_rev = (uint32_t)(S.mask[ra] >> 62) & 1u;     // the opening read
    }
#pragma unroll
    for (int d = 1; d < CB_SPLIT; d <<= 1) {
      reads += __shfl_xor_sync(0xFFFFFFFFu, reads, d);
      minus += __shfl_xor_sync(0xFFFFFFFFu, minus, d);
      t2c += __shfl_xor_sync(0xFFFFFFFFu, t2c, d);
      end = max(end, __shfl_xor_sync(0xFFFFFFFFu, end, d));
      mask |= __shfl_xor_sync(0xFFFFFFFFu, mask, d);
    }
    // ---- B2 -----------------------------------------------------------------------------------------------------
    for (uint32_t i = tid; i < nrd; i += CB_THREADS) {
      unsigned long long m = S.mask[i];
      if (!(m >> 63)) continue;
      const uint32_t k = S.cid[i];
      const unsigned long long um = S.umask[k];
      if (um == 0) continue;
      if (S.ovf[k] || __popcll(um) > CB_SITES) continue;
      const bool rev = (m >> 62) & 1ull;
      m &= (1ull << 51) - 1ull;
      const int32_t lo = S.lo[i] - S.base[k], hi = S.hi[i] - S.base[k];       // relative to bit 0 of the key set
      while (m) {
        const int ib = __ffsll((long long)m) - 1;
        m &= m - 1;
        const int32_t rel = rev ? hi - ib : lo + ib;
        const uint32_t slot = __popcll(um & ((1ull << rel) - 1ull));
        atomicAdd(&S.scnt[slot * CB_CLUSTERS + k], 1u);                   // mutationMap.put(pos, old + 1)
        atomicMin(&S.skey[slot * CB_CLUSTERS + k], (i << 6) | (uint32_t)ib);   // first insertion = earliest read
      }
      const int32_t l = max(lo, 0), h = min(hi, 63);                     // baseCoveredMap (:662-667) at the keys
      if (l <= h) {
        const uint32_t sa = __popcll(um & bits_below(l)), sb = __popcll(um & bits_below(h + 1));
        if (sa < sb) {
          atomicAdd(&S.scov[sa * CB_CLUSTERS + k], 1u);
          if (sb < (uint32_t)CB_SITES) atomicSub(&S.scov[sb * CB_CLUSTERS + k], 1u);
        }
      }
    }
    __syncthreads();
    // ---- B3 -----------------------------------------------------------------------------------------------------
    uint32_t ns = 0;
    bool left = false;
    unsigned long long um = 0;
    if (owner) {
      um = S.umask[kk];
      ns = __popcll(um);
      left = S.ovf[kk] != 0 || ns > (uint32_t)CB_SITES;
      if (left) { S.fb[atomicAdd(&s_nfb, 1u)] = cur + kk; ns = 0; }
    }
    unsigned long long total;
    const unsigned long long ex = block_exclusive<LbSum, CB_WARPS>((unsigned long long)ns, LbSum(), 0ull, s_wtot, total);
    blk_sites += total;
    if (tid == 0) s_base = total ? atomicAdd(&P.st->n_sites, total) : 0ull;
    __syncthreads();
    if (owner && !left) {
      const uint32_t slot = c0 + cur + kk;
      const unsigned long long sb = s_base + ex;
      const uint32_t maf = slot ? minus - first_rev : minus;   // slot 0 continues a cluster opened by the preceding shard
      ps_cluster rec;
      rec.first_read = rs + ra;
      rec.running_id = slot ? P.first_id + slot : 0;           // runningID++ then "cl_<id>_<chr>" (:355): first cluster is cl_2
      rec.contig = reads ? op_contig : 0u;
      rec.start = reads ? base : 0;
      rec.end = reads ? end : 0;
      rec.num_reads = reads;
      rec.num_t2c = t2c;
      rec.minus_after_first = maf;
      rec.first_reverse = (uint8_t)first_rev;
      rec.combined_strand = first_rev ? 1 : (maf ? 2 : 0);     // StrandOrientation state at flush (P6)
      rec.reserved = 0;
      rec.mask51 = mask;
      rec.site_begin = sb;
      rec.site_end = sb + ns;
      if (slot && !first_rev) dstr += maf;                     // doubleStranded++ (:494-498)
      const uint4* src = reinterpret_cast<const uint4*>(&rec);
      uint4* dst = reinterpret_cast<uint4*>(P.cl + slot);
#pragma unroll
      for (int w = 0; w < 4; ++w) dst[w] = src[w];
      uint32_t cov = 0;
      for (uint32_t u = 0; u < ns; ++u) {
        const int bit = __ffsll((long long)um) - 1;
        um &= um - 1;
        cov += S.scov[u * CB_CLUSTERS + kk];
        if (sb + u >= P.cap_sites) break;
        ps_site o;
        o.pos = base + bit; o.t2c = S.scnt[u * CB_CLUSTERS + kk]; o.cov = cov;
        o.reserved = 0;
        const uint32_t key = S.skey[u * CB_CLUSTERS + kk];
        o.order_key = ((unsigned long long)(rs + (key >> 6)) << 6) | (key & 63u);
        P.sites[sb + u] = o;
      }
    }
    __syncthreads();            // the next chunk overwrites the shared arrays
    cur += ncomp;
  }

  // ---- clusters left to the warp routine (tables alias the read arrays, which are free now) ---------------------------
  __syncthreads();
  {
    WarpTables* T = reinterpret_cast<WarpTables*>(smem_raw) + warp;
    WarpRing* G = reinterpret_cast<WarpRing*>(reinterpret_cast<WarpTables*>(smem_raw) + CB_WARPS) + warp;
    ps_cluster* wrec = reinterpret_cast<ps_cluster*>(reinterpret_cast<WarpRing*>(reinterpret_cast<WarpTables*>(smem_raw) + CB_WARPS) + CB_WARPS) + warp;
    const uint32_t nfb = s_nfb;
    for (uint32_t e = warp; e < nfb; e += CB_WARPS) {
      const uint32_t k = S.fb[e], slot = c0 + k;
      const uint32_t f = S.first[k], fe = S.first[k + 1];
      unsigned long long sb = 0;
      const uint32_t cnt = pl_cluster<NW, MK>(P, slot, f, fe, *T, *G, wrec, true, nullptr, 0, dstr, &sb);
      if (lane == 0 && cnt && P.tile_sites) atomicAdd(P.tile_sites + slot / COMPACT_TILE, cnt);
      __syncwarp();
      if (lane == 0) { wrec->site_begin = sb; wrec->site_end = sb + cnt; }
      __syncwarp();
      if (lane < 4) reinterpret_cast<uint4*>(P.cl + slot)[lane] = reinterpret_cast<const uint4*>(wrec)[lane];
      __syncwarp();
    }
  }
  if (tid == 0 && blk_sites && P.tile_sites) atomicAdd(P.tile_sites + c0 / COMPACT_TILE, (unsigned int)blk_sites);
  // doubleStranded of the block
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) dstr += __shfl_xor_sync(0xFFFFFFFFu, dstr, d);
  if (lane == 0 && dstr) atomicAdd(&P.st->dstr, dstr);
}

// Orders the site runs: exclusive prefix of the per-cluster site counts (look-back #3) = final site_begin; every
// cluster's sites move from the completion-ordered array to their place, so the site array ends up compact and
// sorted by (cluster, position) whatever order the blocks of pl_cluster_kernel finished in.
struct CompactParams {
  PlState* st;
  LbDesc* d_cnt;
  unsigned int epoch;
  ps_cluster* cl;
  const ps_site* src;
  ps_site* dst;
  uint64_t cap_cl, cap_sites;
  const unsigned int* tile_sites;   // sites per tile, summed up by pl_cluster_kernel: every tile adds up the entries in
                                    // front of it (no chain between the tiles); nullptr = decoupled look-back
  uint32_t stamp;                   // stamp PlState::ts
  unsigned long long* sec_ts;       // optional: stamp pair of the timed section, whose end this kernel is
};

__device__ __forceinline__ void pl_compact_body(const CompactParams& P) {
  constexpr int ITEMS = COMPACT_ITEMS;
  __shared__ unsigned long long s_wtot[PL_WARPS];
  __shared__ unsigned long long s_pre;
  __shared__ unsigned int s_tile;
  const uint32_t n_slots = P.st->n_flags + 1;
  if (n_slots > P.cap_cl || P.st->n_sites > P.cap_sites) return;
  const uint32_t n_tiles = (n_slots + PL_THREADS * ITEMS - 1) / (PL_THREADS * ITEMS);
  if (threadIdx.x == 0) s_tile = atomicAdd(&P.st->tile_ctr_compact, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  if (tile >= n_tiles) return;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t c0 = tile * PL_THREADS * ITEMS + threadIdx.x * ITEMS;
  unsigned long long from[ITEMS];
  uint32_t cnt[ITEMS];
  uint32_t mine = 0;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    from[j] = 0; cnt[j] = 0;
    if (c0 + j < n_slots) {
      const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&P.cl[c0 + j].site_begin);
      from[j] = v.x; cnt[j] = (uint32_t)(v.y - v.x);
    }
    mine += cnt[j];
  }
  unsigned long long total;
  const unsigned long long ex = block_exclusive((unsigned long long)mine, LbSum(), 0ull, s_wtot, total);
  if (P.tile_sites != nullptr) {
    unsigned long long part = 0;
    for (uint32_t t = threadIdx.x; t < tile; t += PL_THREADS) part += __ldg(P.tile_sites + t);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, d);
    if (lane == 0) s_wtot[warp] = part;      // block_exclusive is done with s_wtot
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long pre = 0;
#pragma unroll
      for (int w = 0; w < PL_WARPS; ++w) pre += s_wtot[w];
      s_pre = pre;
      if (tile == n_tiles - 1) P.st->n_sites_final = pre + total;
    }
  } else if (warp == 0) {
    unsigned long long pre = 0;
    if (tile == 0) {
      if (lane == 0) lb_publish(&P.d_cnt[0], total, 2u, P.epoch);
    } else {
      if (lane == 0) lb_publish(&P.d_cnt[tile], total, 1u, P.epoch);
      pre = lb_exclusive_prefix(P.d_cnt, (int)tile, P.epoch, LbSum(), 0ull);
      if (lane == 0) lb_publish(&P.d_cnt[tile], pre + total, 2u, P.epoch);
    }
    if (lane == 0) {
      s_pre = pre;
      if (tile == n_tiles - 1) P.st->n_sites_final = pre + total;
    }
  }
  __syncthreads();
  unsigned long long to = s_pre + ex;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    if (c0 + j >= n_slots) break;
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(P.src + from[j]);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(P.dst + to);
    if (cnt[j] <= 4) {            // the common case: every word requested before the first one is stored
      unsigned long long w[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) w[e] = (uint32_t)e < cnt[j] * 3 ? src[e] : 0ull;   // a site is 24 bytes
#pragma unroll
      for (int e = 0; e < 12; ++e)
        if ((uint32_t)e < cnt[j] * 3) dst[e] = w[e];
    } else if (cnt[j] <= 16)
      for (uint32_t e = 0; e < cnt[j] * 3; ++e) dst[e] = src[e];
    *reinterpret_cast<ulonglong2*>(&P.cl[c0 + j].site_begin) = make_ulonglong2(to, to + cnt[j]);
    if (c0 + j == 0 || c0 + j == n_slots - 1) {      // the two boundary records ride home with the run state
      ps_cluster rec = P.cl[c0 + j];
      rec.site_begin = to; rec.site_end = to + cnt[j];
      if (c0 + j == 0) P.st->head = rec;
      if (c0 + j == n_slots - 1) P.st->open = rec;
    }
    to += cnt[j];
  }
  // long site runs (deep or long clusters): the whole warp copies them
  to = s_pre + ex;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    uint32_t big = __ballot_sync(0xFFFFFFFFu, c0 + j < n_slots && cnt[j] > 16);
    while (big) {
      const int src_lane = __ffs((int)big) - 1;
      big &= big - 1;
      const unsigned long long f0 = __shfl_sync(0xFFFFFFFFu, from[j], src_lane), t0 = __shfl_sync(0xFFFFFFFFu, to, src_lane);
      const uint32_t n3 = __shfl_sync(0xFFFFFFFFu, cnt[j], src_lane) * 3u;
      const unsigned long long* src = reinterpret_cast<const unsigned long long*>(P.src + f0);
      unsigned long long* dst = reinterpret_cast<unsigned long long*>(P.dst + t0);
      for (uint32_t e = lane; e < n3; e += 32) dst[e] = src[e];
    }
    to += cnt[j];
  }
}

__global__ void __launch_bounds__(PL_THREADS) pl_compact_kernel(const __grid_constant__ CompactParams P) {
  pdl_wait();
  pdl_launch_dependents();
  if (P.stamp && threadIdx.x == 0) stamp_start(&P.st->ts[2]);
  pl_compact_body(P);
  if (P.stamp) {      // every thread is back from the body's returns
    __syncthreads();
    if (threadIdx.x == 0) {
      stamp_end(&P.st->ts[3]);
      if (P.sec_ts) stamp_end(P.sec_ts + 1);
    }
  }
}

// checkPosition interval of reads [r0, r1) (halo merge: dense coverage of a boundary cluster)
template <int NW>
__global__ void pl_interval_kernel(const __grid_constant__ ClusterParams P, uint32_t r0, uint32_t r1, int2* out) {
  ContigCache cc;
  PlRead x;
  for (uint32_t q = r0 + blockIdx.x * blockDim.x; q < r1; q += gridDim.x * blockDim.x) {
    const uint32_t qw = q + (threadIdx.x & ~31u), r = q + threadIdx.x;
    pl_decode<NW>(P, qw, r, r < r1, cc, x);
    if (r < r1) out[r - r0] = x.kept ? make_int2(x.lo, x.hi) : make_int2(1, 0);
  }
}

// run state of a call, and the per-tile site totals of the compaction (one launch instead of a kernel and a memset)
__global__ void pl_init_state(PlState* st, unsigned int* tile_sites, uint32_t n_tile_sites, unsigned long long* sec_ts) {
  pdl_wait();
  pdl_launch_dependents();
  if (sec_ts && threadIdx.x == 0) stamp_start(sec_ts);
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_tile_sites; k += gridDim.x * blockDim.x) tile_sites[k] = 0;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    st->fault = PS_FAULT_NONE; st->skipped = 0; st->dstr = 0; st->n_sites = 0; st->n_sites_final = 0; st->n_flags = 0;
    st->unsorted = 0; st->tile_ctr_flag = 0; st->tile_ctr_compact = 0; st->first_slot1 = 0xFFFFFFFFu; st->spec_failed = 0;
    st->dbg[0] = st->dbg[1] = st->dbg[2] = 0;
    st->ts[0] = st->ts[1] = st->ts[2] = st->ts[3] = 0;
  }
}

}  // namespace

struct ps_pileup {
  ps_ctx* ctx = nullptr;
  cudaStream_t stream = nullptr;
  DeviceBatch batch{};               // the records (device pointers): needed again only for the halo-merge coverage
  uint64_t stage_serial = 0;         // != 0: the batch lives in a staging slot of the context (valid for two uploads)
  uint64_t past_end = 0;             // ps_read_batch.past_end of the call: `batch` holds the reads before that record
  int nw = 0;                        // kernel flavour the batch was run with
  // device results, owned by the handle (stream-ordered allocations)
  ps_cluster* d_cl = nullptr;        // slot 0 = head partial, 1..n_flags-1 closed, n_flags = open
  ps_site* d_sites = nullptr;
  uint32_t first_slot1 = 0;          // first read of slot 1 = end of the head partial
  uint64_t n_slots = 0, n_reads = 0;
  ps_cluster head{}, open{};
  bool has_head = false;
  std::vector<uint32_t> open_cov, head_cov;
  int32_t open_cov_pos0 = 0, head_cov_pos0 = 0;
  bool cov_done = false;
  ps_pileup_counters counters{};
  ps_fault fault{};
  // call in flight (ps_pileup_submit_device ... ps_pileup_wait)
  bool pending = false;              // kernels queued, run state not looked at yet
  int rc = PS_OK;                    // what the completed call returned
  bool has_opts = false;
  ps_pileup_opts opts{};
  bool spec = false;                 // the attempt in flight used the speculative flag pass
  uint64_t cap_cl = 0, cap_sites = 0;   // capacities of the attempt in flight
  bool stamped = false;              // the attempt in flight stamps PlState::ts instead of recording pl_ev
  PlState hs_fallback{};             // landing place of the run state when the context has no page-locked scratch
  // host mode (windowed ps_pileup_bam / ps_multi_pileup_bam, tool_loops.cpp): the merged records of all windows live in
  // host vectors; nothing is resident on a device
  bool host_mode = false;
  std::vector<ps_cluster> h_cl;
  std::vector<ps_site> h_sites, h_open_sites;
};

template <typename T>
static T* scratch(ps_ctx* ctx, int slot, size_t count, cudaError_t& err, bool zero_new = false) {
  if (err != cudaSuccess) return nullptr;
  const size_t bytes = count * sizeof(T) + 64;
  const bool grow = bytes > ctx->pl_scratch[slot].cap;
  err = ctx->pl_scratch[slot].reserve(bytes);
  if (err == cudaSuccess && grow && zero_new) err = cudaMemset(ctx->pl_scratch[slot].p, 0, ctx->pl_scratch[slot].cap);
  return static_cast<T*>(ctx->pl_scratch[slot].p);
}

static bool aligned16p(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Look-back epoch of the next kernel: 30 bits ride in a descriptor's status word (lookback.cuh).  When the counter
// wraps, descriptors written 2^30 epochs ago would read as current ones: clear the three descriptor arrays (slots 2, 3,
// 8 of the scratch table) behind everything queued on the stream and start over at 1.
static unsigned int next_epoch(ps_ctx* ctx, cudaStream_t st) {
  unsigned int e = (++ctx->pl_epoch) & 0x3FFFFFFFu;
  if (e == 0) {
    for (int slot : {2, 3, 8})
      if (ctx->pl_scratch[slot].p) cudaMemsetAsync(ctx->pl_scratch[slot].p, 0, ctx->pl_scratch[slot].cap, st);
    e = (++ctx->pl_epoch) & 0x3FFFFFFFu;
  }
  return e;
}

static int flavour_of(const DeviceBatch& b) {   // 0 = generic decode, 1..4 = PAR-CLIP shape with that many 2-bit words
  const uint32_t L = b.uniform_len;
  const bool fast = L >= 1 && L <= 64 && b.uniform_ncigar == 1 && (reinterpret_cast<uintptr_t>(b.bases2) & 3u) == 0;
  return fast ? (int)((L + 15) / 16) : 0;
}

template <int NW, bool MK>
static cudaError_t launch_cluster_nw(ps_ctx* ctx, uint32_t grid, cudaStream_t st, const ClusterParams& Q) {
  auto kern = pl_cluster_kernel<NW, MK>;
  int per_sm = 0;
  cudaError_t e = fn_blocks_per_sm(ctx, reinterpret_cast<const void*>(kern), CB_THREADS, kClusterSmemBytes, &per_sm);
  if (e != cudaSuccess) return e;
  return launch_chained(ctx, kern, grid, CB_THREADS, kClusterSmemBytes, st, Q);
}
static cudaError_t launch_cluster(ps_ctx* ctx, int nw, uint32_t grid, cudaStream_t st, const ClusterParams& Q) {
  if (Q.t2c_mask != nullptr) {
    switch (nw) {
      case 1: return launch_cluster_nw<1, true>(ctx, grid, st, Q);
      case 2: return launch_cluster_nw<2, true>(ctx, grid, st, Q);
      case 3: return launch_cluster_nw<3, true>(ctx, grid, st, Q);
      case 4: return launch_cluster_nw<4, true>(ctx, grid, st, Q);
      default: break;      // no mask words exist for other shapes
    }
  }
  switch (nw) {
    case 1: return launch_cluster_nw<1, false>(ctx, grid, st, Q);
    case 2: return launch_cluster_nw<2, false>(ctx, grid, st, Q);
    case 3: return launch_cluster_nw<3, false>(ctx, grid, st, Q);
    case 4: return launch_cluster_nw<4, false>(ctx, grid, st, Q);
    default: return launch_cluster_nw<0, false>(ctx, grid, st, Q);
  }
}

constexpr uint64_t kCompactSumTiles = 4096;     // 2 M cluster slots
constexpr uint32_t kFlagSumTiles = 8192;        // 16.7 M reads on the vector path

// One attempt of the three stages on H->stream: allocations, kernels and the copy of the run state into page-locked
// memory -- nothing here waits for the device.
static int pileup_launch(ps_ctx* ctx, ps_pileup* H) {
  const DeviceBatch& b = H->batch;
  const ps_pileup_opts* opts = H->has_opts ? &H->opts : nullptr;
  cudaStream_t st = H->stream;
  const uint64_t n = b.n_reads;
  const bool vec = b.uniform_ncigar == 1 && aligned16p(b.meta) && aligned16p(b.ref_start) && aligned16p(b.cigar);
  const uint32_t tile_reads = FLAG_THREADS * (vec ? (uint32_t)PL_FLAG_ITEMS : 1u);
  const uint32_t n_tiles = (uint32_t)((n + tile_reads - 1) / tile_reads);
  const int nw = H->nw;

  cudaError_t err = cudaSuccess;
  PlState* d_state = scratch<PlState>(ctx, 0, 1, err);
  LbDesc* d_max = scratch<LbDesc>(ctx, 2, n_tiles, err, true);
  LbDesc* d_cnt = scratch<LbDesc>(ctx, 3, n_tiles, err, true);
  if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");

  unsigned long long carry_key = 0;
  if (opts && opts->carry_valid) carry_key = pileup_key(ctx->contig_rank, opts->carry_contig, opts->carry_cluster_end);

  const uint64_t cap_cl = std::min<uint64_t>(ctx->pl_cap_cl, n + 2), cap_sites = ctx->pl_cap_ev;
  H->cap_cl = cap_cl; H->cap_sites = cap_sites;
  const uint32_t c_tiles = (uint32_t)((cap_cl + CB_CLUSTERS - 1) / CB_CLUSTERS);
  LbDesc* d_sc = scratch<LbDesc>(ctx, 8, c_tiles, err, true);
  if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");
  if (H->d_cl) { cudaFreeAsync(H->d_cl, st); H->d_cl = nullptr; }
  if (H->d_sites) { cudaFreeAsync(H->d_sites, st); H->d_sites = nullptr; }
  PS_CUDA(ctx, cudaMallocAsync((void**)&H->d_cl, cap_cl * sizeof(ps_cluster), st));
  PS_CUDA(ctx, cudaMallocAsync((void**)&H->d_sites, (cap_sites + 1) * sizeof(ps_site), st));
  ps_site* d_tmp = scratch<ps_site>(ctx, 10, cap_sites + 1, err);
  uint32_t* d_first = scratch<uint32_t>(ctx, 4, cap_cl + 2, err);
  if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");

  FlagParams P;
  P.b = b; P.ref = ctx->ref; P.st = d_state; P.d_max = d_max; P.d_cnt = d_cnt; P.epoch = next_epoch(ctx, st);
  P.n_tiles = n_tiles; P.carry_key = carry_key; P.cl_first = d_first; P.cap_cl = cap_cl;
  P.carry_keys = (opts && opts->carry_keys_n) ? (const unsigned long long*)opts->carry_keys_device : nullptr;
  P.carry_keys_n = P.carry_keys ? opts->carry_keys_n : 0;
  // site totals per compaction tile, added up by the cluster kernel: up to kCompactSumTiles tiles every compaction
  // block sums the entries in front of it itself; beyond that (quadratic work) the decoupled look-back takes over
  const uint64_t n_ctiles = (cap_cl + COMPACT_TILE - 1) / COMPACT_TILE;
  unsigned int* tile_sites = nullptr;
  if (n_ctiles <= kCompactSumTiles && !ctx->pl_compact_lookback) {
    tile_sites = scratch<unsigned int>(ctx, 11, n_ctiles, err);
    if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");
  }
  // the kernels are chained (launch_chained): with that on, no event sits between them and the timers are stamps
  const bool stamp = ctx->pdl && ctx->timers_on;
  const bool ev = ctx->timers_on && !stamp;
  H->stamped = stamp;
  ctx->pl_ts_valid = false;
  const unsigned int compact_epoch = next_epoch(ctx, st);   // its occasional memset goes in front of the kernels
  timer_begin_chained(ctx, st);   // the timer pair is complete when the launch returns (a submitted call may be waited
                                  // for after other timed calls of the context)
  unsigned long long* sec_ts = ctx->cur_ts;
  PS_CUDA(ctx, launch_chained(ctx, pl_init_state, tile_sites ? (uint32_t)((n_ctiles + 255) / 256) : 1u, 256, 0, st, d_state,
                              tile_sites, tile_sites ? (uint32_t)n_ctiles : 0u, sec_ts));
  if (ev) cudaEventRecord(ctx->pl_ev[0], st);
  const bool spec = vec && !ctx->pl_exact_flags;
  H->spec = spec;
  P.tile_ein = nullptr; P.tile_agg = nullptr; P.tile_cnt = nullptr; P.flag_words = nullptr; P.scan_in_expand = 0;
  P.stamp = stamp ? 1u : 0u;
  if (spec) {
    P.tile_ein = scratch<unsigned long long>(ctx, 1, n_tiles, err);
    P.tile_agg = scratch<unsigned long long>(ctx, 7, n_tiles, err);
    P.tile_cnt = scratch<uint32_t>(ctx, 5, n_tiles, err);
    P.flag_words = scratch<uint32_t>(ctx, 6, (size_t)n_tiles * FLAG_THREADS, err);
    if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");
    // up to kFlagSumTiles tiles (16.7 M reads) the expand kernel takes the prefix over the tile table itself (every
    // block sums the counts in front of it: quadratic, but a few thousand entries); beyond that the one-block scan
    P.scan_in_expand = (n_tiles <= kFlagSumTiles && !ctx->pl_flag_scan_kernel) ? 1u : 0u;
    PS_CUDA(ctx, launch_chained(ctx, pl_flag_kernel<PL_FLAG_ITEMS, true>, n_tiles, FLAG_THREADS, 0, st, P));
    if (!P.scan_in_expand) {
      PS_CUDA(ctx, launch_chained(ctx, pl_flag_scan_kernel, 1, SCAN_THREADS, 0, st, P));
      ctx->launches += 1;
    }
    PS_CUDA(ctx, launch_chained(ctx, pl_flag_expand_kernel<PL_FLAG_ITEMS>, n_tiles, FLAG_THREADS, 0, st, P));
    ctx->launches += 1;
  } else if (vec) PS_CUDA(ctx, launch_chained(ctx, pl_flag_kernel<PL_FLAG_ITEMS, false>, n_tiles, FLAG_THREADS, 0, st, P));
  else PS_CUDA(ctx, launch_chained(ctx, pl_flag_kernel<1, false>, n_tiles, FLAG_THREADS, 0, st, P));
  if (ev) cudaEventRecord(ctx->pl_ev[1], st);
  ClusterParams Q;
  Q.b = b; Q.ref = ctx->ref; Q.st = d_state;
  Q.first_id = opts ? opts->first_running_id : 1; Q.cl_first = d_first; Q.cl = H->d_cl; Q.sites = d_tmp;
  Q.cap_cl = cap_cl; Q.cap_sites = cap_sites;
  Q.tile_sites = tile_sites;
  Q.t2c_mask = (nw > 0 && opts) ? reinterpret_cast<const unsigned long long*>(opts->t2c_masks_device) : nullptr;
  Q.stamp = P.stamp;
  PS_CUDA(ctx, launch_cluster(ctx, nw, c_tiles, st, Q));
  if (ev) cudaEventRecord(ctx->pl_ev[2], st);
  CompactParams R;
  R.st = d_state; R.d_cnt = d_sc; R.epoch = compact_epoch; R.cl = H->d_cl; R.src = d_tmp; R.dst = H->d_sites;
  R.cap_cl = cap_cl; R.cap_sites = cap_sites; R.tile_sites = Q.tile_sites;
  R.stamp = P.stamp; R.sec_ts = sec_ts;
  PS_CUDA(ctx, launch_chained(ctx, pl_compact_kernel, (uint32_t)n_ctiles, PL_THREADS, 0, st, R));
  if (ev) { cudaEventRecord(ctx->pl_ev[3], st); ctx->pl_ev_valid = true; }
  if (stamp) ctx->pl_ev_valid = false;
  ctx->launches += 4;
  PlState* hsp = ctx->h_pinned ? static_cast<PlState*>(ctx->h_pinned) : &H->hs_fallback;
  PS_CUDA(ctx, cudaMemcpyAsync(hsp, d_state, sizeof(PlState), cudaMemcpyDeviceToHost, st));
  timer_end(ctx, st);
  return PS_OK;
}

// Waits for the attempt in flight; repeats it with the exact flag kernel or larger arrays where the run state asks for
// that; fills the handle's counters.  Returns what the synchronous call returns.
static int pileup_finish(ps_ctx* ctx, ps_pileup* H) {
  if (!H->pending) return H->rc;
  H->pending = false;
  if (ctx->pl_pending == H) ctx->pl_pending = nullptr;
  auto done = [&](int rc) { H->rc = rc; return rc; };
  auto past_end = [&]() {
    H->fault.code = PS_FAULT_PAST_END;
    H->fault.read_ordinal = H->past_end - 1;
    return done(set_error(ctx, PS_ERR_UNSUPPORTED, "pileup: a record with no reference span starts past its contig's end"));
  };
  cudaStream_t st = H->stream;
  const uint64_t n = H->n_reads;
  if (n == 0) return past_end();        // only a call whose first record is past its contig's end waits here unlaunched
  PlState hs{};
  for (int attempt = 0;; ++attempt) {
    const PlState* hsp = ctx->h_pinned ? static_cast<const PlState*>(ctx->h_pinned) : &H->hs_fallback;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "pileup"));
    hs = *hsp;
    bool again = false;
    if (H->spec && hs.spec_failed) {     // a record reaches over the halo: this context keeps to the exact kernel from now on
      ctx->pl_exact_flags = true;
      --attempt;
      again = true;
    } else {
      const uint64_t need_cl = (uint64_t)hs.n_flags + 1, need_sites = hs.n_sites;
      if (need_cl > H->cap_cl || need_sites > H->cap_sites) {
        if (attempt >= 2) return done(set_error(ctx, PS_ERR_CUDA, "pileup: capacity retry failed"));
        // the totals do not depend on the capacities (dropped writes only); the site total is only known once the
        // cluster slots fit, so a batch may need two more passes the first time a context sees its shape
        ctx->pl_cap_cl = std::max(ctx->pl_cap_cl, need_cl + need_cl / 16 + 2);
        ctx->pl_cap_ev = std::max(ctx->pl_cap_ev, need_sites + need_sites / 16);
        again = true;
      }
    }
    if (!again) break;
    const int rc = pileup_launch(ctx, H);
    if (rc != PS_OK) return done(rc);
  }
  if (H->stamped) {
    for (int i = 0; i < 4; ++i) ctx->pl_ts[i] = hs.ts[i];
    ctx->pl_ts_valid = true;
  }
  H->counters.skipped_due_indel = hs.skipped;
  if (hs.fault != PS_FAULT_NONE) {
    H->fault.code = (int32_t)(hs.fault & 0xFF);
    H->fault.read_ordinal = hs.fault >> 8;
    if (H->fault.code == PS_FAULT_CIGAR_OPS)
      return done(set_error(ctx, PS_ERR_UNSUPPORTED, "pileup: a record of this batch has more than 255 CIGAR operations"));
    return done(set_error(ctx, PS_ERR_REFERENCE_WOULD_THROW, "pileup: the JVM would die on a record of this batch"));
  }
  if (H->past_end) return past_end();
  if (hs.unsorted) return done(set_error(ctx, PS_ERR_UNSORTED, ps_strerror(PS_ERR_UNSORTED)));

  const uint64_t n_slots = (uint64_t)hs.n_flags + 1;
  H->n_slots = n_slots;
  // summary: head partial (slot 0), open cluster (last slot)
  if (getenv("PARASUITE_B200_DEBUG"))
    fprintf(stderr, "[ps_pileup] warp-routine site passes %llu, sweep give-ups %llu, window passes %llu\n", hs.dbg[0], hs.dbg[1], hs.dbg[2]);
  H->head = hs.head;
  if (hs.n_flags) H->open = hs.open;
  H->first_slot1 = hs.first_slot1 == 0xFFFFFFFFu ? (uint32_t)n : hs.first_slot1;
  H->has_head = H->head.num_reads != 0;
  H->counters.has_open_cluster = hs.n_flags ? 1 : 0;
  H->counters.double_stranded = hs.dstr;
  H->counters.n_clusters = hs.n_flags ? hs.n_flags - 1 : 0;
  const uint64_t sites_before_open = hs.n_flags ? H->open.site_begin : hs.n_sites_final;
  H->counters.n_sites = sites_before_open - H->head.site_end;
  return done(PS_OK);
}

// Creates the handle and queues the first attempt.  wait == false: returns right behind the launches (ps_pileup_wait
// completes the call); one submitted call per context at a time (run state and scratch belong to the context).
static int run_pileup(ps_ctx* ctx, const DeviceBatch& b, const ps_pileup_opts* opts, cudaStream_t st, ps_pileup** out,
                      bool wait = true) {
  if (ctx->pl_pending) return set_error(ctx, PS_ERR_STATE, "a submitted pileup call of this context has not been waited for");
  if (opts && opts->carry_valid && opts->carry_contig >= ctx->ref.n_contigs)
    return set_error(ctx, PS_ERR_INVALID_ARG, "carry_contig is not a contig of the reference");
  // A batch that sits in a staging slot of this context (ps_batch_upload / ps_pileup_batch): the pileup never reads
  // qualities, so it may start as soon as the other streams of the records have arrived (event staged_core), while the
  // quality bytes (more than half of the upload) are still on their way.  Asked to run on the context's own stream --
  // behind the whole upload -- it goes to the auxiliary stream instead; on a caller's stream it waits for the event.
  for (int slot = 0; slot < 2; ++slot)
    if (b.n_reads && b.meta == ctx->staged[slot].view.meta && ctx->staged_core[slot]) {
      if (st == ctx->stream && ctx->stream2) st = ctx->stream2;
      if (st != ctx->stream) cudaStreamWaitEvent(st, ctx->staged_core[slot], 0);
    }
  ps_pileup* H = new ps_pileup();
  *out = H;
  H->ctx = ctx;
  H->stream = st;
  H->batch = b;
  if (b.past_end && b.past_end <= b.n_reads) {
    // a record past its contig's end (pileup_finish answers PS_FAULT_PAST_END for it): the reads before it decide whether
    // an earlier record faults first, and none of the kernels sees the record
    H->past_end = b.past_end;
    H->batch.n_reads = b.past_end - 1;
  }
  H->batch.past_end = 0;
  H->has_opts = opts != nullptr;
  if (opts) H->opts = *opts;
  const uint64_t n = H->batch.n_reads;
  H->n_reads = n;
  H->counters.num_reads_processed = b.n_reads;
  if (n == 0) {
    if (!H->past_end) return PS_OK;
    H->pending = true;
    ctx->pl_pending = H;
    return wait ? pileup_finish(ctx, H) : PS_OK;
  }
  if (n >= 0xFFFFFFFFull) return set_error(ctx, PS_ERR_UNSUPPORTED, "pileup batch of >= 2^32 reads");
  H->nw = flavour_of(b);
  if (ctx->pl_cap_cl < 1024) ctx->pl_cap_cl = std::max<uint64_t>(1024, n / 8);
  if (ctx->pl_cap_ev < 1024) ctx->pl_cap_ev = std::max<uint64_t>(1024, n / 4);   // site capacity
  const int rc = pileup_launch(ctx, H);
  if (rc != PS_OK) { H->rc = rc; return rc; }
  H->pending = true;
  ctx->pl_pending = H;
  return wait ? pileup_finish(ctx, H) : PS_OK;
}

static void free_handle(ps_pileup* h) {
  if (!h) return;
  if (h->host_mode) { delete h; return; }
  if (h->ctx) cudaSetDevice(h->ctx->device);
  if (h->pending && h->ctx) pileup_finish(h->ctx, h);     // the kernels in flight use the handle's arrays
  if (h->ctx && h->ctx->pl_pending == h) h->ctx->pl_pending = nullptr;
  if (h->d_cl) cudaFreeAsync(h->d_cl, h->stream);
  if (h->d_sites) cudaFreeAsync(h->d_sites, h->stream);
  delete h;
}

// dense baseCoveredMap of the two boundary clusters, from the read intervals (needed only by the halo merge)
static int boundary_coverage(ps_pileup* h) {
  if (h->cov_done) return PS_OK;
  ps_ctx* ctx = h->ctx;
  if (!ctx || h->n_reads == 0) { h->cov_done = true; return PS_OK; }
  if (h->stage_serial && ctx->stage_serial - h->stage_serial >= 2)
    return set_error(ctx, PS_ERR_STATE, "boundary coverage must be read before the second-next upload on this context");
  cudaSetDevice(ctx->device);
  ClusterParams Q{};
  Q.b = h->batch; Q.ref = ctx->ref; Q.st = (PlState*)ctx->pl_scratch[0].p;
  auto dense = [&](uint64_t r0, uint64_t r1, std::vector<uint32_t>& cov, int32_t& pos0) -> int {
    if (r1 <= r0) return PS_OK;
    int2* d_iv = nullptr;
    PS_CUDA(ctx, cudaMallocAsync((void**)&d_iv, (r1 - r0) * sizeof(int2), h->stream));
    const uint32_t grid = (uint32_t)std::min<uint64_t>((r1 - r0 + 255) / 256, 1024);
    switch (h->nw) {
      case 1: pl_interval_kernel<1><<<grid, 256, 0, h->stream>>>(Q, (uint32_t)r0, (uint32_t)r1, d_iv); break;
      case 2: pl_interval_kernel<2><<<grid, 256, 0, h->stream>>>(Q, (uint32_t)r0, (uint32_t)r1, d_iv); break;
      case 3: pl_interval_kernel<3><<<grid, 256, 0, h->stream>>>(Q, (uint32_t)r0, (uint32_t)r1, d_iv); break;
      case 4: pl_interval_kernel<4><<<grid, 256, 0, h->stream>>>(Q, (uint32_t)r0, (uint32_t)r1, d_iv); break;
      default: pl_interval_kernel<0><<<grid, 256, 0, h->stream>>>(Q, (uint32_t)r0, (uint32_t)r1, d_iv); break;
    }
    ctx->launches++;
    std::vector<int2> v(r1 - r0);
    PS_CUDA(ctx, cudaMemcpyAsync(v.data(), d_iv, (r1 - r0) * sizeof(int2), cudaMemcpyDeviceToHost, h->stream));
    PS_CUDA(ctx, cudaStreamSynchronize(h->stream));
    cudaFreeAsync(d_iv, h->stream);
    int32_t mn = INT32_MAX, mx = INT32_MIN;
    for (const int2& x : v)
      if (x.x <= x.y) { mn = std::min(mn, x.x); mx = std::max(mx, x.y); }
    if (mn > mx) return PS_OK;
    pos0 = mn;
    cov.assign((size_t)(mx - mn + 1), 0);
    for (const int2& x : v)
      for (int32_t p = x.x; p <= x.y; ++p) cov[p - mn]++;
    return PS_OK;
  };
  const uint64_t n_flags = h->n_slots - 1;
  if (h->has_head) {
    const uint32_t r1 = n_flags ? h->first_slot1 : (uint32_t)h->n_reads;
    int rc = dense(0, r1, h->head_cov, h->head_cov_pos0);
    if (rc) return rc;
  }
  if (h->counters.has_open_cluster) {
    int rc = dense(h->open.first_read, h->n_reads, h->open_cov, h->open_cov_pos0);
    if (rc) return rc;
  }
  h->cov_done = true;
  return PS_OK;
}

// Handle over records that already sit on the host: closed clusters (site_begin / site_end index `sites`), the open
// cluster with its sites (site range [0, n)) and its dense coverage, the run's counters.
ps_pileup* pileup_host_handle(ps_ctx* ctx, std::vector<ps_cluster>&& clusters, std::vector<ps_site>&& sites, bool has_open,
                              const ps_cluster& open, std::vector<ps_site>&& open_sites, int32_t open_cov_pos0,
                              std::vector<uint32_t>&& open_cov, const ps_pileup_counters& counters) {
  ps_pileup* H = new ps_pileup();
  H->ctx = ctx;
  H->host_mode = true;
  H->h_cl = std::move(clusters);
  H->h_sites = std::move(sites);
  H->h_open_sites = std::move(open_sites);
  H->open = open;
  H->open_cov = std::move(open_cov);
  H->open_cov_pos0 = open_cov_pos0;
  H->cov_done = true;
  H->counters = counters;
  H->counters.n_clusters = H->h_cl.size();
  H->counters.n_sites = H->h_sites.size();
  H->counters.has_open_cluster = has_open ? 1 : 0;
  H->n_reads = counters.num_reads_processed;
  return H;
}

void pileup_set_fault(ps_pileup* h, const ps_fault& f) { h->fault = f; }

extern "C" {

int ps_pileup_batch_device(ps_ctx* ctx, const ps_read_batch* b, const ps_pileup_opts* opts, void* stream,
                           ps_pileup** out) {
  if (!ctx || !b || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc = run_pileup(ctx, view_of(b), opts, st, out);
  if (rc != PS_OK && !(*out && (*out)->fault.code)) { free_handle(*out); *out = nullptr; }   // a fault stays readable
  return rc;
}

int ps_pileup_submit_device(ps_ctx* ctx, const ps_read_batch* b, const ps_pileup_opts* opts, void* stream,
                            ps_pileup** out) {
  if (!ctx || !b || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc = run_pileup(ctx, view_of(b), opts, st, out, /*wait=*/false);
  if (rc != PS_OK) { free_handle(*out); *out = nullptr; }
  return rc;
}
int ps_pileup_wait(ps_pileup* h) {
  if (!h) return PS_ERR_INVALID_ARG;
  if (!h->ctx) return PS_OK;
  cudaSetDevice(h->ctx->device);
  return pileup_finish(h->ctx, h);
}
int ps_pileup_batch(ps_ctx* ctx, const ps_read_batch* hb, const ps_pileup_opts* opts, ps_pileup** out) {
  if (!ctx || !hb || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  if (hb->n_reads == 0) { *out = new ps_pileup(); (*out)->ctx = ctx; return PS_OK; }
  StagedBatch* sb = nullptr;
  int rc = stage_batch(ctx, hb, /*with_qual=*/false, &sb);
  if (rc) return rc;
  ps_pileup_opts o{};
  if (opts) o = *opts;
  o.t2c_masks_device = nullptr;      // mask words belong to a device-resident batch the caller ran the profile on
  rc = run_pileup(ctx, sb->view, opts ? &o : nullptr, ctx->stream, out);
  if (*out) (*out)->stage_serial = ctx->stage_serial;
  if (rc != PS_OK && !(*out && (*out)->fault.code)) { free_handle(*out); *out = nullptr; }   // a fault stays readable
  return rc;
}

int ps_pileup_max_key_device(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream, uint64_t** dev_key) {
  if (!ctx || !dev_batch || !dev_key) return PS_ERR_INVALID_ARG;
  if (!ctx->ref_loaded) return set_error(ctx, PS_ERR_STATE, "no reference loaded");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  // a batch in a staging slot of this context, keyed on a caller's stream: meta / ref_start / cigar have arrived once
  // the slot's core event has fired (the key kernel reads nothing else)
  for (int slot = 0; slot < 2; ++slot)
    if (st != ctx->stream && dev_batch->n_reads && dev_batch->meta == ctx->staged[slot].view.meta && ctx->staged_core[slot])
      cudaStreamWaitEvent(st, ctx->staged_core[slot], 0);
  cudaError_t err = cudaSuccess;
  unsigned long long* d_key = scratch<unsigned long long>(ctx, 9, 1, err);
  if (err != cudaSuccess) return cuda_fail(ctx, err, "pileup scratch");
  *dev_key = reinterpret_cast<uint64_t*>(d_key);
  PS_CUDA(ctx, cudaMemsetAsync(d_key, 0, 8, st));
  if (dev_batch->n_reads == 0) return PS_OK;
  FlagParams P{};
  P.b = view_of(dev_batch); P.ref = ctx->ref;
  const uint32_t grid = (uint32_t)std::min<uint64_t>((dev_batch->n_reads + PL_THREADS - 1) / PL_THREADS, (uint64_t)ctx->sm_count * 8);
  pl_maxkey_kernel<<<grid, PL_THREADS, 0, st>>>(P, d_key);
  ctx->launches++;
  PS_CUDA(ctx, cudaGetLastError());
  return PS_OK;
}

int ps_pileup_max_key(ps_ctx* ctx, const ps_read_batch* dev_batch, void* stream, uint32_t* valid, uint32_t* contig,
                      int32_t* end) {
  if (!ctx || !dev_batch || !valid || !contig || !end) return PS_ERR_INVALID_ARG;
  *valid = 0; *contig = 0; *end = 0;
  uint64_t* d_key = nullptr;
  const int rc = ps_pileup_max_key_device(ctx, dev_batch, stream, &d_key);
  if (rc != PS_OK) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  unsigned long long* hk = ctx->h_pinned ? reinterpret_cast<unsigned long long*>(static_cast<char*>(ctx->h_pinned) + 1024) : nullptr;
  unsigned long long tmp = 0;
  PS_CUDA(ctx, cudaMemcpyAsync(hk ? hk : &tmp, d_key, 8, cudaMemcpyDeviceToHost, st));
  PS_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned long long k = hk ? *hk : tmp;
  if (k) { *valid = 1; pileup_key_decode(ctx->contig_by_rank, k, contig, end); }
  return PS_OK;
}

int ps_pileup_counters_get(const ps_pileup* h, ps_pileup_counters* out) {
  if (!h || !out) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  *out = h->counters;
  return PS_OK;
}

int64_t ps_pileup_next(ps_pileup* h, uint64_t first, ps_cluster* clusters, uint64_t max_clusters, ps_site* sites,
                       uint64_t max_sites) {
  if (!h || !clusters || (!sites && max_sites)) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  const uint64_t n_closed = h->counters.n_clusters;
  if (first >= n_closed || max_clusters == 0) return 0;
  if (h->host_mode) {
    const uint64_t cnt0 = std::min<uint64_t>(max_clusters, n_closed - first);
    const uint64_t sb = h->h_cl[first].site_begin;
    uint64_t m = 0;
    while (m < cnt0 && h->h_cl[first + m].site_end - sb <= max_sites) ++m;
    if (m == 0) return 0;
    std::memcpy(clusters, h->h_cl.data() + first, m * sizeof(ps_cluster));
    const uint64_t ns = h->h_cl[first + m - 1].site_end - sb;
    if (ns) std::memcpy(sites, h->h_sites.data() + sb, ns * sizeof(ps_site));
    for (uint64_t k = 0; k < m; ++k) { clusters[k].site_begin -= sb; clusters[k].site_end -= sb; }
    return (int64_t)m;
  }
  ps_ctx* ctx = h->ctx;
  cudaSetDevice(ctx->device);
  uint64_t cnt = std::min<uint64_t>(max_clusters, n_closed - first);
  // closed clusters are slots 1 .. n_flags-1; their sites are contiguous and in slot order
  if (first == 0 && cnt == n_closed && h->counters.n_sites <= max_sites) {
    // everything at once (the common call): the site range is known from the boundary records, so both copies are
    // queued back to back and the host waits once
    const uint64_t sb = h->head.site_end, ns = h->counters.n_sites;
    PS_CUDA(ctx, cudaMemcpyAsync(clusters, h->d_cl + 1, cnt * sizeof(ps_cluster), cudaMemcpyDeviceToHost, h->stream));
    if (ns) PS_CUDA(ctx, cudaMemcpyAsync(sites, h->d_sites + sb, ns * sizeof(ps_site), cudaMemcpyDeviceToHost, h->stream));
    PS_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (sb)
      for (uint64_t k = 0; k < cnt; ++k) { clusters[k].site_begin -= sb; clusters[k].site_end -= sb; }
    return (int64_t)cnt;
  }
  PS_CUDA(ctx, cudaMemcpyAsync(clusters, h->d_cl + 1 + first, cnt * sizeof(ps_cluster), cudaMemcpyDeviceToHost, h->stream));
  PS_CUDA(ctx, cudaStreamSynchronize(h->stream));
  const uint64_t sb = clusters[0].site_begin;
  uint64_t m = 0;
  while (m < cnt && clusters[m].site_end - sb <= max_sites) ++m;
  if (m == 0) return 0;
  const uint64_t ns = clusters[m - 1].site_end - sb;
  if (ns) {
    PS_CUDA(ctx, cudaMemcpyAsync(sites, h->d_sites + sb, ns * sizeof(ps_site), cudaMemcpyDeviceToHost, h->stream));
    PS_CUDA(ctx, cudaStreamSynchronize(h->stream));
  }
  if (sb)
    for (uint64_t k = 0; k < m; ++k) { clusters[k].site_begin -= sb; clusters[k].site_end -= sb; }
  return (int64_t)m;
}

static int copy_boundary(ps_pileup* h, const ps_cluster& src, ps_cluster* cluster, ps_site* sites, uint64_t max_sites) {
  const uint64_t ns = src.site_end - src.site_begin;
  if (ns > max_sites) return PS_ERR_INVALID_ARG;
  *cluster = src;
  cluster->site_begin = 0;
  cluster->site_end = ns;
  if (ns) {
    if (!sites) return PS_ERR_INVALID_ARG;
    ps_ctx* ctx = h->ctx;
    cudaSetDevice(ctx->device);
    PS_CUDA(ctx, cudaMemcpyAsync(sites, h->d_sites + src.site_begin, ns * sizeof(ps_site), cudaMemcpyDeviceToHost, h->stream));
    PS_CUDA(ctx, cudaStreamSynchronize(h->stream));
  }
  return 1;
}

int ps_pileup_open_cluster(ps_pileup* h, ps_cluster* cluster, ps_site* sites, uint64_t max_sites) {
  if (!h || !cluster) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  if (!h->counters.has_open_cluster) return 0;
  if (h->host_mode) {
    if (h->h_open_sites.size() > max_sites) return PS_ERR_INVALID_ARG;
    *cluster = h->open;
    cluster->site_begin = 0;
    cluster->site_end = h->h_open_sites.size();
    if (!h->h_open_sites.empty()) {
      if (!sites) return PS_ERR_INVALID_ARG;
      std::memcpy(sites, h->h_open_sites.data(), h->h_open_sites.size() * sizeof(ps_site));
    }
    return 1;
  }
  return copy_boundary(h, h->open, cluster, sites, max_sites);
}

int ps_pileup_head_partial(ps_pileup* h, ps_cluster* cluster, ps_site* sites, uint64_t max_sites) {
  if (!h || !cluster) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  if (!h->has_head) return 0;
  return copy_boundary(h, h->head, cluster, sites, max_sites);
}

int64_t ps_pileup_boundary_coverage(ps_pileup* h, int which, int32_t* first_pos, uint32_t* cov, uint64_t max) {
  if (!h || !first_pos) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  int rc = boundary_coverage(h);
  if (rc) return rc;
  const std::vector<uint32_t>& v = which ? h->open_cov : h->head_cov;
  *first_pos = which ? h->open_cov_pos0 : h->head_cov_pos0;
  if (!cov) return (int64_t)v.size();
  if (v.size() > max) return PS_ERR_INVALID_ARG;
  if (!v.empty()) std::memcpy(cov, v.data(), v.size() * 4);
  return (int64_t)v.size();
}

int ps_pileup_fault(const ps_pileup* h, ps_fault* out) {
  if (!h || !out) return PS_ERR_INVALID_ARG;
  if (h->pending) return PS_ERR_STATE;
  *out = h->fault;
  return PS_OK;
}

void ps_pileup_close(ps_pileup* h) { free_handle(h); }

}  // extern "C"
