// TEST INFRASTRUCTURE ONLY.
//
// CPU restatement (C++17, no dependencies) of the track's per-position deletion and insertion counts: the contract in
// the header comment next to ps_track_batch_ex2 (include/parasuite_b200.h), fed the same SoA read batches and packed
// reference as the CUDA path.  The runs, sites, counters and faults are those of the track restatement in
// oracle/track_oracle.cpp, compiled into this library; the indel counts come from a walk of their own, per position
// (no difference arrays).  Pinned against the Python restatement in track_indels_oracle.py
// (tests/test_track_indels_cpu.py).  Built and loaded by track_indels_oracle.py.
#include "../oracle/track_oracle.cpp"

namespace {

struct or_track_indels {
  or_track_result* track = nullptr;
  std::vector<ps_track_indel_row> rows;
  ps_track_indel_totals totals{};
};

// per contig: coverage, deletions and anchored insertions by strand and position
struct IndelContig {
  int64_t contig = -1;
  uint64_t lo = 0;                       // global offset of the contig's first base
  std::vector<uint32_t> cov[2], del[2], ins[2];
  void flush(or_track_indels* R, const ps_reference* ref, uint32_t min_depth, uint32_t min_ev) {
    if (contig < 0) return;
    for (size_t p = 0; p < cov[0].size(); ++p)
      for (uint32_t s = 0; s < 2; ++s) {
        const uint64_t d = del[s][p], i = ins[s][p], c = cov[s][p];
        if (d + i < min_ev || c + d < min_depth) continue;
        const uint64_t g = lo + p;
        ps_track_indel_row x{};
        x.contig = (uint32_t)contig; x.pos = (int32_t)p + 1; x.strand = (uint8_t)s;
        x.ref = ((ref->inv[g >> 5] >> (g & 31)) & 1u) ? 4 : (uint8_t)(((ref->seq2[g >> 4] >> (2 * (g & 15))) & 3u) ^ (s ? 3u : 0u));
        x.cov = (uint32_t)c; x.del = (uint32_t)d; x.ins = (uint32_t)i;
        R->rows.push_back(x);
      }
    contig = -1;
  }
};

}  // namespace

extern "C" {

or_track_indels* or_track_run_indels(const ps_reference* ref, const ps_read_batch* b, const ps_track_indel_opts* o) {
  auto* R = new or_track_indels();
  R->track = or_track_run(ref, b);
  if (R->track->status != PS_OK) return R;         // a faulting or unsorted batch has no indel rows
  const uint32_t min_depth = std::max<uint32_t>(1, o->min_depth), min_ev = std::max<uint32_t>(1, o->min_events);
  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  IndelContig T;
  for (uint64_t ord = 0; ord < b->n_reads; ++ord, cur.advance()) {
    cur.get(v);
    if (v.flags & PS_RF_UNMAPPED) continue;
    bool hasI = false, hasD = false, hasN = false;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15;
      hasI |= op == 1; hasD |= op == 2; hasN |= op == 3;
    }
    if ((hasI || hasD) && hasN) continue;
    const int64_t contig = contig_of(ref, v.ref_start);
    const uint64_t c_lo = ref->contig_off[contig], c_hi = ref->contig_off[contig + 1];
    if (contig != T.contig) {
      T.flush(R, ref, min_depth, min_ev);
      T.contig = contig;
      T.lo = c_lo;
      for (int s = 0; s < 2; ++s) {
        T.cov[s].assign((size_t)(c_hi - c_lo), 0u);
        T.del[s].assign((size_t)(c_hi - c_lo), 0u);
        T.ins[s].assign((size_t)(c_hi - c_lo), 0u);
      }
    }
    const uint32_t s = (v.flags & PS_RF_REVERSE) ? 1 : 0;
    uint64_t g = v.ref_start;                      // the next reference position (global offset)
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15, n = v.cigar[e] >> 4;
      if (op == 0 || op == 7 || op == 8) {
        for (uint32_t k = 0; k < n; ++k) T.cov[s][g + k - c_lo]++;
      } else if (op == 2 && n) {
        R->totals.deletion_ops[s]++;
        for (uint32_t k = 0; k < n; ++k)
          if (g + k < c_hi) { T.del[s][g + k - c_lo]++; R->totals.deleted_bases[s]++; }
      } else if (op == 1 && n) {
        R->totals.insertion_ops[s]++;
        R->totals.inserted_bases[s] += n;
        if (g > v.ref_start && g - 1 < c_hi) T.ins[s][g - 1 - c_lo]++;
        else R->totals.unanchored_insertions[s]++;
      }
      if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) g += n;
    }
  }
  T.flush(R, ref, min_depth, min_ev);
  R->totals.n_rows = R->rows.size();
  return R;
}

int or_track_indels_status(const or_track_indels* r, ps_track_counters* ctr, ps_fault* fault) {
  return or_track_status(r->track, ctr, fault);
}
// which = 0 / 1: runs of that strand, 2: sites, 3: indel rows
int64_t or_track_indels_copy(const or_track_indels* r, int which, void* out, uint64_t max) {
  if (which < 3) return or_track_copy(r->track, which, out, max);
  const uint64_t n = std::min<uint64_t>(max, r->rows.size());
  if (n) std::memcpy(out, r->rows.data(), n * sizeof(ps_track_indel_row));
  return (int64_t)n;
}
void or_track_indel_totals(const or_track_indels* r, ps_track_indel_totals* out) { *out = r->totals; }
void or_track_free_indels(or_track_indels* r) {
  or_track_free(r->track);
  delete r;
}

}  // extern "C"
