// TEST INFRASTRUCTURE ONLY.
//
// CPU restatement (C++17, no dependencies) of the track's per-position base counts: the contract in the header comment
// next to ps_track_batch_ex (include/parasuite_b200.h), fed the same SoA read batches and packed reference as the CUDA
// path.  The runs, sites, counters and faults are those of the track restatement in oracle/track_oracle.cpp, compiled
// into this library; the base counts come from a walk of their own.  Pinned against the Python restatement in
// track_bases_oracle.py (tests/test_track_bases_cpu.py).  Built and loaded by track_bases_oracle.py.
#include "../oracle/track_oracle.cpp"

namespace {

struct or_track_ex {
  or_track_result* track = nullptr;
  std::vector<ps_track_base_row> rows;
  ps_track_base_totals totals{};
};

// per contig: [strand][A C G T N][position], the plus-strand reference code of every ACGT position (4: none)
struct BasesContig {
  int64_t contig = -1;
  std::vector<uint32_t> n[2][5];
  std::vector<uint8_t> ref;
  void flush(or_track_ex* R, uint32_t mask, uint32_t min_cov, uint32_t min_ev) {
    if (contig < 0) return;
    for (size_t p = 0; p < ref.size(); ++p) {
      if (ref[p] > 3) continue;
      for (uint32_t s = 0; s < 2; ++s) {
        ps_track_base_row x{};
        for (int b = 0; b < 5; ++b) { x.n[b] = n[s][b][p]; x.cov += x.n[b]; }
        if (!x.cov) continue;
        const uint32_t a = ref[p] ^ (s ? 3u : 0u);
        uint32_t picked = 0;
        for (uint32_t b = 0; b < 4; ++b)
          if (b != a && ((mask >> (4 * a + b)) & 1u)) picked += x.n[b];
        if (x.cov < min_cov || picked < min_ev) continue;
        x.contig = (uint32_t)contig; x.pos = (int32_t)p + 1; x.strand = (uint8_t)s; x.ref = (uint8_t)a;
        R->rows.push_back(x);
      }
    }
    contig = -1;
  }
};

}  // namespace

extern "C" {

or_track_ex* or_track_run_ex(const ps_reference* ref, const ps_read_batch* b, const ps_track_opts* o) {
  auto* R = new or_track_ex();
  R->track = or_track_run(ref, b);
  if (R->track->status != PS_OK) return R;         // a faulting or unsorted batch has no base rows
  const uint32_t mask = (o->substitutions ? o->substitutions : 0xFFFFu) & ~0x8421u;
  const uint32_t min_cov = std::max<uint32_t>(1, o->min_coverage), min_ev = std::max<uint32_t>(1, o->min_events);
  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  std::vector<uint8_t> bases;
  BasesContig T;
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
      T.flush(R, mask, min_cov, min_ev);
      T.contig = contig;
      for (auto& s : T.n)
        for (auto& a : s) a.assign((size_t)(c_hi - c_lo), 0u);
      T.ref.assign((size_t)(c_hi - c_lo), 4);
    }
    const uint32_t s = (v.flags & PS_RF_REVERSE) ? 1 : 0, flip = s ? 3u : 0u;
    read_ascii(v, bases);
    uint64_t rd = 0, rf = 0;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15, n = v.cigar[e] >> 4;
      if (op == 1 || op == 4) rd += n;
      else if (op == 2 || op == 3) rf += n;
      else if (op == 0 || op == 7 || op == 8) {
        for (uint32_t k = 0; k < n; ++k) {
          const uint64_t g = v.ref_start + rf + k, p = g - c_lo;
          if ((ref->inv[g >> 5] >> (g & 31)) & 1u) continue;
          const uint32_t a = (ref->seq2[g >> 4] >> (2 * (g & 15))) & 3u;
          T.ref[p] = (uint8_t)a;
          const char* hit = (const char*)memchr(kBase, bases[rd + k], 4);
          const uint32_t col = hit ? (uint32_t)(hit - kBase) ^ flip : 4u;
          T.n[s][col][p]++;
          R->totals.bases[s][a ^ flip][col]++;
        }
        rd += n; rf += n;
      }
    }
  }
  T.flush(R, mask, min_cov, min_ev);
  R->totals.n_rows = R->rows.size();
  return R;
}

int or_track_ex_status(const or_track_ex* r, ps_track_counters* ctr, ps_fault* fault) {
  return or_track_status(r->track, ctr, fault);
}
// which = 0 / 1: runs of that strand, 2: sites, 3: base rows
int64_t or_track_ex_copy(const or_track_ex* r, int which, void* out, uint64_t max) {
  if (which < 3) return or_track_copy(r->track, which, out, max);
  const uint64_t n = std::min<uint64_t>(max, r->rows.size());
  if (n) std::memcpy(out, r->rows.data(), n * sizeof(ps_track_base_row));
  return (int64_t)n;
}
void or_track_base_totals(const or_track_ex* r, ps_track_base_totals* out) { *out = r->totals; }
void or_track_free_ex(or_track_ex* r) {
  or_track_free(r->track);
  delete r;
}

}  // extern "C"
