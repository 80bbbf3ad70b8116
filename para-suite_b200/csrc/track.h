// Host side of the track (track.cu), shared with the windowed file tool (tool_loops.cpp).
#pragma once
#include <vector>

#include "internal.h"

// Positions [key0, key0 + len) of one contig, keys (rank + 1) << 32 | 1-based position (ps_ctx::contig_rank);
// v = cov+, cov-, t2c+, t2c-, len entries each.
struct TrackDense {
  unsigned long long key0 = 0;
  uint32_t len = 0;
  std::vector<uint32_t> v;
};

// One track call.  Runs and sites are final for the positions reported; keys as in TrackDense.
struct TrackOut {
  std::vector<ps_track_run> runs[2];
  std::vector<ps_track_site> sites;
  ps_track_counters ctr{};
  ps_fault fault{};
  unsigned long long first_key = 0, last_key = 0, max_end_key = 0;   // first / last kept start, maximum end; 0: no kept read
  TrackDense head, tail;     // windowed only
};

// windowed == false: the batch is the whole input, every position is reported.
// windowed == true (one window of a sorted file): positions up to prev_end (the maximum end key of the windows before,
// 0 if none) come back dense in `head`, positions from the last kept start on dense in `tail`; the runs and sites cover
// the positions in between.  Waits for the device.
int track_run(ps_ctx* ctx, const DeviceBatch& b, cudaStream_t st, bool windowed, uint64_t prev_end, TrackOut* out);
