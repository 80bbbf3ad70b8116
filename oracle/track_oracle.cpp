// TEST INFRASTRUCTURE ONLY.
//
// CPU restatement (C++17, no dependencies) of the per-position T>C conversion and coverage track (tool `track`, no Java
// counterpart): the contract in the header comment of ps_track_batch (include/parasuite_b200.h), fed the same SoA read
// batches and packed reference as the CUDA path.  Pinned against the independent Python restatement in track_oracle.py
// (tests/test_track_cpu.py).  Built and loaded by track_oracle.py.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../include/parasuite_b200.h"

namespace {

const char kBase[4] = {'A', 'C', 'G', 'T'};

struct ReadView {
  uint32_t flags, L, ncig;
  uint64_t ref_start;
  const uint32_t* cigar;
  const uint8_t* bases2;
  std::vector<uint32_t> invalid_pos;  // exceptions of this read
};

// walks the tile structure of a batch sequentially
struct BatchCursor {
  const ps_read_batch* b;
  uint64_t r = 0;
  uint64_t boff = 0, coff = 0;
  explicit BatchCursor(const ps_read_batch* bb) : b(bb) {}
  void enter_tile(uint64_t t) {
    boff = b->uniform_len ? r * ((b->uniform_len + 3) / 4) : b->tile_base_off[t];
    coff = b->uniform_ncigar ? r * (uint64_t)b->uniform_ncigar : b->tile_cigar_off[t];
  }
  void get(ReadView& v) {
    const uint32_t m = b->meta[r];
    v.flags = PS_META_FLAGS(m);
    v.L = PS_META_LEN(m);
    v.ncig = PS_META_NCIGAR(m);
    v.ref_start = b->ref_start[r];
    v.cigar = b->cigar + coff;
    v.bases2 = b->bases2 + boff;
    v.invalid_pos.clear();
    if ((v.flags & PS_RF_HAS_INVALID) && b->tile_exc_off) {
      const uint64_t t = r / PS_TILE_READS;
      const uint32_t rit = (uint32_t)(r % PS_TILE_READS);
      for (uint32_t e = b->tile_exc_off[t]; e < b->tile_exc_off[t + 1]; ++e)
        if ((b->exc[e] >> 16) == rit) v.invalid_pos.push_back(b->exc[e] & 0xFFFFu);
    }
  }
  void advance() {
    const uint32_t m = b->meta[r];
    boff += (PS_META_LEN(m) + 3) / 4;
    coff += PS_META_NCIGAR(m);
    ++r;
    if (r % PS_TILE_READS == 0 && r < b->n_reads) enter_tile(r / PS_TILE_READS);
  }
};

// the read's bases as ASCII, 'N' where the batch lists an invalid base
void read_ascii(const ReadView& v, std::vector<uint8_t>& out) {
  out.resize(v.L);
  for (uint32_t p = 0; p < v.L; ++p) out[p] = kBase[(v.bases2[p >> 2] >> (2 * (p & 3))) & 3];
  for (uint32_t p : v.invalid_pos)
    if (p < v.L) out[p] = 'N';
}

inline uint32_t contig_of(const ps_reference* ref, uint64_t g) {
  const uint64_t* lo = ref->contig_off;
  const uint64_t* it = std::upper_bound(lo, lo + ref->n_contigs + 1, g);
  return (uint32_t)(it - lo) - 1;
}

}  // namespace

// arrays (one contig at a time: the records are sorted), rows in (contig, position) order.  Contigs in FASTA order.
namespace {

struct or_track_result {
  std::vector<ps_track_run> runs[2];
  std::vector<ps_track_site> sites;
  ps_track_counters ctr{};
  ps_fault fault{};
  int status = PS_OK;
};

struct TrackContig {
  int64_t contig = -1;
  std::vector<uint32_t> v[4];          // cov+, cov-, t2c+, t2c-
  void flush(or_track_result* R) {
    if (contig < 0) return;
    const uint32_t c = (uint32_t)contig;
    for (int s = 0; s < 2; ++s) {
      const std::vector<uint32_t>& a = v[s];
      for (size_t p = 0; p < a.size();) {
        if (!a[p]) { ++p; continue; }
        size_t q = p;
        while (q < a.size() && a[q] == a[p]) ++q;
        R->runs[s].push_back(ps_track_run{c, (uint32_t)p, (uint32_t)q, a[p]});
        p = q;
      }
    }
    for (size_t p = 0; p < v[0].size(); ++p)
      for (int s = 0; s < 2; ++s)
        if (v[2 + s][p]) R->sites.push_back(ps_track_site{c, (int32_t)p + 1, (uint32_t)s, v[2 + s][p], v[s][p]});
    contig = -1;
    for (auto& a : v) std::vector<uint32_t>().swap(a);
  }
};

}  // namespace

extern "C" {

or_track_result* or_track_run(const ps_reference* ref, const ps_read_batch* b) {
  auto* R = new or_track_result();
  R->ctr.num_reads_processed = b->n_reads;
  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  std::vector<uint8_t> bases;
  TrackContig T;
  int64_t prev_contig = -1, prev_start = 0;
  bool unsorted = false;
  auto fault = [&](int32_t code, uint64_t ord) { R->fault.code = code; R->fault.read_ordinal = ord; };
  for (uint64_t ord = 0; ord < b->n_reads; ++ord, cur.advance()) {
    cur.get(v);
    if (v.flags & PS_RF_UNMAPPED) { R->ctr.unmapped++; continue; }
    if (v.flags & PS_RF_CIGAR_OVERFLOW) { fault(PS_FAULT_CIGAR_OPS, ord); break; }
    bool hasI = false, hasD = false, hasN = false;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15;
      hasI |= op == 1; hasD |= op == 2; hasN |= op == 3;
    }
    if ((hasI || hasD) && hasN) { R->ctr.skipped_due_indel++; continue; }
    if ((v.flags & PS_RF_POS_ZERO) || v.ref_start >= ref->n_bases) { fault(PS_THROW_REF_RANGE, ord); break; }
    const int64_t contig = contig_of(ref, v.ref_start);
    const uint64_t c_lo = ref->contig_off[contig], c_hi = ref->contig_off[contig + 1];
    // every block is fetched before a base is looked at
    int32_t bad = 0;
    uint64_t rd = 0, rf = 0;
    for (uint32_t e = 0; e < v.ncig && !bad; ++e) {
      const uint32_t op = v.cigar[e] & 15, n = v.cigar[e] >> 4;
      if (op == 1 || op == 4) rd += n;
      else if (op == 2 || op == 3) rf += n;
      else if (op == 0 || op == 7 || op == 8) {
        if (rd + n > v.L) bad = PS_THROW_BLOCK_RANGE;
        else if ((v.flags & PS_RF_REF_RANGE) || v.ref_start + rf + n > c_hi) bad = PS_THROW_REF_RANGE;
        rd += n; rf += n;
      }
    }
    if (bad) { fault(bad, ord); break; }
    const int64_t start = (int64_t)(v.ref_start - c_lo) + 1;
    if (prev_contig >= 0 && (contig < prev_contig || (contig == prev_contig && start < prev_start))) unsorted = true;
    prev_contig = contig; prev_start = start;
    if (contig != T.contig) {
      T.flush(R);
      T.contig = contig;
      for (auto& a : T.v) a.assign((size_t)(c_hi - c_lo), 0u);
    }
    R->ctr.reads_counted++;
    const int s = (v.flags & PS_RF_REVERSE) ? 1 : 0;
    read_ascii(v, bases);
    rd = 0; rf = 0;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15, n = v.cigar[e] >> 4;
      if (op == 1 || op == 4) rd += n;
      else if (op == 2 || op == 3) rf += n;
      else if (op == 0 || op == 7 || op == 8) {
        for (uint32_t k = 0; k < n; ++k) {
          const uint64_t g = v.ref_start + rf + k, p = g - c_lo;
          T.v[s][p]++;
          R->ctr.aligned_bases[s]++;
          if ((ref->inv[g >> 5] >> (g & 31)) & 1u) continue;
          const char a = kBase[(ref->seq2[g >> 4] >> (2 * (g & 15))) & 3], r = (char)bases[rd + k];
          if (s == 0 ? (a == 'T' && r == 'C') : (a == 'A' && r == 'G')) { T.v[2 + s][p]++; R->ctr.t2c_events[s]++; }
        }
        rd += n; rf += n;
      }
    }
  }
  T.flush(R);
  if (R->fault.code) R->status = R->fault.code == PS_FAULT_CIGAR_OPS ? PS_ERR_UNSUPPORTED : PS_ERR_REFERENCE_WOULD_THROW;
  else if (unsorted) R->status = PS_ERR_UNSORTED;
  R->ctr.n_runs[0] = R->runs[0].size();
  R->ctr.n_runs[1] = R->runs[1].size();
  R->ctr.n_sites = R->sites.size();
  return R;
}

// status of the call (PS_OK, PS_ERR_REFERENCE_WOULD_THROW / PS_ERR_UNSUPPORTED with *fault, PS_ERR_UNSORTED)
int or_track_status(const or_track_result* r, ps_track_counters* ctr, ps_fault* fault) {
  *ctr = r->ctr;
  *fault = r->fault;
  return r->status;
}
// which = 0 / 1: runs of that strand, 2: sites
int64_t or_track_copy(const or_track_result* r, int which, void* out, uint64_t max) {
  if (which < 2) {
    const uint64_t n = std::min<uint64_t>(max, r->runs[which].size());
    if (n) std::memcpy(out, r->runs[which].data(), n * sizeof(ps_track_run));
    return (int64_t)n;
  }
  const uint64_t n = std::min<uint64_t>(max, r->sites.size());
  if (n) std::memcpy(out, r->sites.data(), n * sizeof(ps_track_site));
  return (int64_t)n;
}
void or_track_free(or_track_result* r) { delete r; }

}  // extern "C"
