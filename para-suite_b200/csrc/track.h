// Host side of the track (track.cu), shared with the windowed file tool (tool_loops.cpp).
#pragma once
#include <vector>

#include "internal.h"

// Positions [key0, key0 + len) of one contig, keys (rank + 1) << 32 | 1-based position (ps_ctx::contig_rank);
// v = cov+, cov-, t2c+, t2c-, len entries each; with base counts ten more: the event counters A, C, G, T, N of the plus
// strand, then of the minus strand (TrackBases); with indel counts four more at the end: del+, del-, ins+, ins-.
struct TrackDense {
  unsigned long long key0 = 0;
  uint32_t len = 0;
  std::vector<uint32_t> v;
};

// The base-count option of a call (ps_track_opts), thresholds and mask normalised: on == false is the plain track.
struct TrackBases {
  bool on = false;
  uint32_t min_cov = 1, min_ev = 1;
  uint32_t mask = 0;           // the twelve substitution bits that count, diagonal cleared
};
// ps_track_opts -> TrackBases; PS_ERR_INVALID_ARG for bits above 15
int track_bases_of(const ps_track_opts* o, TrackBases* out);
// The row of one position and strand (device selection and host pending region alike): ev[0..4] are its event counters
// (read bases A C G T other than the reference base a, and N calls; strand orientation), n[0..4] receives the row.  The
// reference base's own count is what the coverage leaves.  false: no row under `sel`.
__host__ __device__ inline bool track_base_row(const TrackBases& sel, uint32_t a, uint32_t cov, const uint32_t* ev, uint32_t* n) {
  uint32_t picked = 0, other = 0;
  for (uint32_t b = 0; b < 4; ++b) {
    if (b == a) continue;
    other += ev[b];
    if ((sel.mask >> (4 * a + b)) & 1u) picked += ev[b];
  }
  if (cov < sel.min_cov || picked < sel.min_ev) return false;
  for (uint32_t b = 0; b < 4; ++b) n[b] = b == a ? cov - other - ev[4] : ev[b];
  n[4] = ev[4];
  return true;
}

// The indel option of a call (ps_track_indel_opts), thresholds normalised: on == false counts no indels.  With it on,
// TrackDense::v gains four arrays after the others: del+, del-, ins+, ins-.
struct TrackIndels {
  bool on = false;
  uint32_t min_depth = 1, min_ev = 1;
};
// ps_track_indel_opts -> TrackIndels; PS_ERR_INVALID_ARG for reserved != 0
int track_indels_of(const ps_track_indel_opts* o, TrackIndels* out);
// The indel row rule of one position and strand (device selection and host pending region alike): cov is that strand's
// coverage, del / ins its deletions and anchored insertions.
__host__ __device__ inline bool track_indel_row(const TrackIndels& sel, uint32_t cov, uint32_t del, uint32_t ins) {
  return (uint64_t)del + ins >= sel.min_ev && (uint64_t)cov + del >= sel.min_depth;
}

// The read and base filters of a call (ps_track_filter_opts), validated: on == false is the unfiltered track.
// records: a flag or MAPQ test is set (tr_read_kernel<true>); min_bq > 0: the base filter (tr_accum_kernel<.., true>).
struct TrackFilter {
  bool on = false, records = false;
  uint32_t min_mapq = 0, require = 0, exclude = 0, min_bq = 0;
};
// ps_track_filter_opts -> TrackFilter; PS_ERR_INVALID_ARG as the header says (aux may be NULL)
int track_filter_of(const ps_track_filter_opts* o, const ps_read_aux* aux, TrackFilter* out);
// The record filter (device and host alike): 0 kept, 1 dropped by a flag test, 2 dropped for its MAPQ
__host__ __device__ inline int track_filtered(const TrackFilter& f, uint32_t sam_flags, uint32_t mapq) {
  if ((sam_flags & f.exclude) || (sam_flags & f.require) != f.require) return 1;
  return mapq < f.min_mapq ? 2 : 0;
}

// One track call.  Runs and sites are final for the positions reported; keys as in TrackDense.
struct TrackOut {
  std::vector<ps_track_run> runs[2];
  std::vector<ps_track_site> sites;
  ps_track_counters ctr{};
  ps_fault fault{};
  unsigned long long first_key = 0, last_key = 0, max_end_key = 0;   // first / last kept start, maximum end; 0: no kept read
  TrackDense head, tail;     // windowed only
  bool bases_on = false;
  std::vector<ps_track_base_row> base_rows;
  ps_track_base_totals totals{};
  bool indels_on = false;
  std::vector<ps_track_indel_row> indel_rows;
  ps_track_indel_totals indel_totals{};
  bool filter_on = false;
  ps_track_filter_counters fctr{};
};

// windowed == false: the batch is the whole input, every position is reported.
// windowed == true (one window of a sorted file): positions up to prev_end (the maximum end key of the windows before,
// 0 if none) come back dense in `head`, positions from the last kept start on dense in `tail`; the runs and sites cover
// the positions in between.  Waits for the device.
// `bases`, `indels`: the base-count and indel options (rows for the reported positions, totals over every kept read).
// `filter`, `aux`: the read and base filters and the device aux arrays they read (b.qual for the base filter).
int track_run(ps_ctx* ctx, const DeviceBatch& b, cudaStream_t st, bool windowed, uint64_t prev_end, TrackOut* out,
              const TrackBases& bases = TrackBases(), const TrackIndels& indels = TrackIndels(),
              const TrackFilter& filter = TrackFilter(), const ps_read_aux& aux = ps_read_aux{});
// Copies the host aux arrays the filter reads into the staging slot `sb` (ctx->stream); *dev: their device pointers
int track_stage_aux(ps_ctx* ctx, StagedBatch* sb, uint64_t n, const ps_read_aux* aux, const TrackFilter& filter,
                    ps_read_aux* dev);
