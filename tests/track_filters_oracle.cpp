// TEST INFRASTRUCTURE ONLY.
//
// CPU restatement (C++17, no dependencies) of the track's read and base filters: the contract in the header comment next
// to ps_track_batch_ex3 (include/parasuite_b200.h), fed the same SoA read batches, aux arrays and packed reference as the
// CUDA path.  One call gives the runs, sites, counters and faults of the track, and optionally its base counts and
// indel counts, all under the filters.  The batch walk (ReadView, BatchCursor, TrackContig) is the track restatement's
// in oracle/track_oracle.cpp, compiled into this library; the filters, the quality offsets and the three walks are
// restated here.  Pinned against the Python restatement in track_filters_oracle.py (tests/test_track_filters_cpu.py).
// Built and loaded by track_filters_oracle.py.
#include "../oracle/track_oracle.cpp"

namespace {

struct or_track_filtered {
  or_track_result track;
  ps_track_filter_counters fctr{};
  std::vector<ps_track_base_row> base_rows;
  ps_track_base_totals base_totals{};
  std::vector<ps_track_indel_row> indel_rows;
  ps_track_indel_totals indel_totals{};
};

// 0: kept, 1: dropped by a flag test, 2: for its MAPQ (f == NULL: no filter)
int filtered(const ps_track_filter_opts* f, const ps_read_aux* aux, uint64_t r) {
  if (!f) return 0;
  const uint32_t flag = (aux && aux->sam_flags) ? aux->sam_flags[r] : 0u, mapq = (aux && aux->mapq) ? aux->mapq[r] : 255u;
  if ((flag & f->exclude_flags) || (flag & f->require_flags) != f->require_flags) return 1;
  return mapq < f->min_mapq ? 2 : 0;
}

// byte offset of every read's qualities
std::vector<uint64_t> qual_offsets(const ps_read_batch* b) {
  std::vector<uint64_t> q(b->n_reads);
  uint64_t cur = 0;
  for (uint64_t r = 0; r < b->n_reads; ++r) {
    if (r % PS_TILE_READS == 0) cur = b->uniform_len ? r * b->uniform_len : b->tile_qual_off[r / PS_TILE_READS];
    q[r] = cur;
    cur += PS_META_LEN(b->meta[r]);
  }
  return q;
}

// read base p of read r is below min_base_quality (a read without qualities has none)
bool low_quality(const ps_track_filter_opts* f, const ps_read_batch* b, const std::vector<uint64_t>& qoff, uint64_t r,
                 uint32_t flags, uint32_t p) {
  return f && f->min_base_quality && !(flags & PS_RF_QUAL_MISSING) && b->qual[qoff[r] + p] < f->min_base_quality;
}

bool skipped(const ReadView& v) {
  bool hasI = false, hasD = false, hasN = false;
  for (uint32_t e = 0; e < v.ncig; ++e) {
    const uint32_t op = v.cigar[e] & 15;
    hasI |= op == 1; hasD |= op == 2; hasN |= op == 3;
  }
  return (hasI || hasD) && hasN;
}

// the track: or_track_run with the filters
void run_track(or_track_filtered* F, const ps_reference* ref, const ps_read_batch* b, const ps_read_aux* aux,
               const ps_track_filter_opts* filter, const std::vector<uint64_t>& qoff) {
  or_track_result* R = &F->track;
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
    if (const int why = filtered(filter, aux, ord)) {
      // absent, except that the batch's one past-end record is refused even so
      if (b->past_end && ord == b->past_end - 1) { fault(PS_FAULT_PAST_END, ord); break; }
      (why == 1 ? F->fctr.filtered_flags : F->fctr.filtered_mapq)++;
      continue;
    }
    if (v.flags & PS_RF_UNMAPPED) { R->ctr.unmapped++; continue; }
    if (v.flags & PS_RF_CIGAR_OVERFLOW) { fault(PS_FAULT_CIGAR_OPS, ord); break; }
    if (skipped(v)) { R->ctr.skipped_due_indel++; continue; }
    if (b->past_end && ord == b->past_end - 1) { fault(PS_FAULT_PAST_END, ord); break; }
    if ((v.flags & PS_RF_POS_ZERO) || v.ref_start >= ref->n_bases) { fault(PS_THROW_REF_RANGE, ord); break; }
    const int64_t contig = contig_of(ref, v.ref_start);
    const uint64_t c_lo = ref->contig_off[contig], c_hi = ref->contig_off[contig + 1];
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
          if (low_quality(filter, b, qoff, ord, v.flags, (uint32_t)(rd + k))) { F->fctr.low_quality_bases[s]++; continue; }
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
  if (R->fault.code) R->status = (R->fault.code == PS_FAULT_CIGAR_OPS || R->fault.code == PS_FAULT_PAST_END) ? PS_ERR_UNSUPPORTED : PS_ERR_REFERENCE_WOULD_THROW;
  else if (unsorted) R->status = PS_ERR_UNSORTED;
  R->ctr.n_runs[0] = R->runs[0].size();
  R->ctr.n_runs[1] = R->runs[1].size();
  R->ctr.n_sites = R->sites.size();
}

// the kept records of a clean batch, in order: (view, ordinal, contig, contig start, contig end)
template <typename Fn>
void for_kept(const ps_reference* ref, const ps_read_batch* b, const ps_read_aux* aux, const ps_track_filter_opts* filter,
              Fn&& fn) {
  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  for (uint64_t ord = 0; ord < b->n_reads; ++ord, cur.advance()) {
    cur.get(v);
    if (filtered(filter, aux, ord) || (v.flags & PS_RF_UNMAPPED) || skipped(v)) continue;
    const int64_t contig = contig_of(ref, v.ref_start);
    fn(v, ord, contig, ref->contig_off[contig], ref->contig_off[contig + 1]);
  }
}

// base counts under the filters (the rows and totals of ps_track_opts)
void run_bases(or_track_filtered* F, const ps_reference* ref, const ps_read_batch* b, const ps_read_aux* aux,
               const ps_track_filter_opts* filter, const std::vector<uint64_t>& qoff, const ps_track_opts* o) {
  const uint32_t mask = (o->substitutions ? o->substitutions : 0xFFFFu) & ~0x8421u;
  const uint32_t min_cov = std::max<uint32_t>(1, o->min_coverage), min_ev = std::max<uint32_t>(1, o->min_events);
  int64_t cur_contig = -1;
  std::vector<uint32_t> n[2][5];
  std::vector<uint8_t> refc;
  auto flush = [&]() {
    if (cur_contig < 0) return;
    for (size_t p = 0; p < refc.size(); ++p) {
      if (refc[p] > 3) continue;
      for (uint32_t s = 0; s < 2; ++s) {
        ps_track_base_row x{};
        for (int c = 0; c < 5; ++c) { x.n[c] = n[s][c][p]; x.cov += x.n[c]; }
        if (!x.cov) continue;
        const uint32_t a = refc[p] ^ (s ? 3u : 0u);
        uint32_t picked = 0;
        for (uint32_t c = 0; c < 4; ++c)
          if (c != a && ((mask >> (4 * a + c)) & 1u)) picked += x.n[c];
        if (x.cov < min_cov || picked < min_ev) continue;
        x.contig = (uint32_t)cur_contig; x.pos = (int32_t)p + 1; x.strand = (uint8_t)s; x.ref = (uint8_t)a;
        F->base_rows.push_back(x);
      }
    }
  };
  std::vector<uint8_t> bases;
  for_kept(ref, b, aux, filter, [&](const ReadView& v, uint64_t ord, int64_t contig, uint64_t c_lo, uint64_t c_hi) {
    if (contig != cur_contig) {
      flush();
      cur_contig = contig;
      for (auto& s : n)
        for (auto& a : s) a.assign((size_t)(c_hi - c_lo), 0u);
      refc.assign((size_t)(c_hi - c_lo), 4);
    }
    const uint32_t s = (v.flags & PS_RF_REVERSE) ? 1 : 0, flip = s ? 3u : 0u;
    read_ascii(v, bases);
    uint64_t rd = 0, rf = 0;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15, len = v.cigar[e] >> 4;
      if (op == 1 || op == 4) rd += len;
      else if (op == 2 || op == 3) rf += len;
      else if (op == 0 || op == 7 || op == 8) {
        for (uint32_t k = 0; k < len; ++k) {
          const uint64_t g = v.ref_start + rf + k, p = g - c_lo;
          if (low_quality(filter, b, qoff, ord, v.flags, (uint32_t)(rd + k))) continue;
          if ((ref->inv[g >> 5] >> (g & 31)) & 1u) continue;
          const uint32_t a = (ref->seq2[g >> 4] >> (2 * (g & 15))) & 3u;
          refc[p] = (uint8_t)a;
          const char* hit = (const char*)memchr(kBase, bases[rd + k], 4);
          const uint32_t col = hit ? (uint32_t)(hit - kBase) ^ flip : 4u;
          n[s][col][p]++;
          F->base_totals.bases[s][a ^ flip][col]++;
        }
        rd += len; rf += len;
      }
    }
  });
  flush();
  F->base_totals.n_rows = F->base_rows.size();
}

// indel counts under the filters: the indels are not filtered by base quality, the coverage of the row rule is
void run_indels(or_track_filtered* F, const ps_reference* ref, const ps_read_batch* b, const ps_read_aux* aux,
                const ps_track_filter_opts* filter, const std::vector<uint64_t>& qoff, const ps_track_indel_opts* o) {
  const uint32_t min_depth = std::max<uint32_t>(1, o->min_depth), min_ev = std::max<uint32_t>(1, o->min_events);
  ps_track_indel_totals& tot = F->indel_totals;
  int64_t cur_contig = -1;
  uint64_t lo = 0;
  std::vector<uint32_t> cov[2], del[2], ins[2];
  auto flush = [&]() {
    if (cur_contig < 0) return;
    for (size_t p = 0; p < cov[0].size(); ++p)
      for (uint32_t s = 0; s < 2; ++s) {
        const uint64_t d = del[s][p], i = ins[s][p], c = cov[s][p];
        if (d + i < min_ev || c + d < min_depth) continue;
        const uint64_t g = lo + p;
        ps_track_indel_row x{};
        x.contig = (uint32_t)cur_contig; x.pos = (int32_t)p + 1; x.strand = (uint8_t)s;
        x.ref = ((ref->inv[g >> 5] >> (g & 31)) & 1u) ? 4 : (uint8_t)(((ref->seq2[g >> 4] >> (2 * (g & 15))) & 3u) ^ (s ? 3u : 0u));
        x.cov = (uint32_t)c; x.del = (uint32_t)d; x.ins = (uint32_t)i;
        F->indel_rows.push_back(x);
      }
  };
  for_kept(ref, b, aux, filter, [&](const ReadView& v, uint64_t ord, int64_t contig, uint64_t c_lo, uint64_t c_hi) {
    if (contig != cur_contig) {
      flush();
      cur_contig = contig;
      lo = c_lo;
      for (int s = 0; s < 2; ++s) {
        cov[s].assign((size_t)(c_hi - c_lo), 0u);
        del[s].assign((size_t)(c_hi - c_lo), 0u);
        ins[s].assign((size_t)(c_hi - c_lo), 0u);
      }
    }
    const uint32_t s = (v.flags & PS_RF_REVERSE) ? 1 : 0;
    uint64_t g = v.ref_start;                      // the next reference position (global offset)
    uint32_t rd = 0;                               // the next read position
    for (uint32_t e = 0; e < v.ncig; ++e) {
      const uint32_t op = v.cigar[e] & 15, n = v.cigar[e] >> 4;
      if (op == 0 || op == 7 || op == 8) {
        for (uint32_t k = 0; k < n; ++k)
          if (!low_quality(filter, b, qoff, ord, v.flags, rd + k)) cov[s][g + k - c_lo]++;
      } else if (op == 2 && n) {
        tot.deletion_ops[s]++;
        for (uint32_t k = 0; k < n; ++k)
          if (g + k < c_hi) { del[s][g + k - c_lo]++; tot.deleted_bases[s]++; }
      } else if (op == 1 && n) {
        tot.insertion_ops[s]++;
        tot.inserted_bases[s] += n;
        if (g > v.ref_start && g - 1 < c_hi) ins[s][g - 1 - c_lo]++;
        else tot.unanchored_insertions[s]++;
      }
      if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) g += n;
      if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) rd += n;
    }
  });
  flush();
  tot.n_rows = F->indel_rows.size();
}

}  // namespace

extern "C" {

// aux / filter may be NULL (no filter); bases / indels: NULL leaves that option out.  A faulting or unsorted batch has
// no base or indel rows.
or_track_filtered* or_track_run_filtered(const ps_reference* ref, const ps_read_batch* b, const ps_read_aux* aux,
                                         const ps_track_filter_opts* filter, const ps_track_opts* bases,
                                         const ps_track_indel_opts* indels) {
  auto* F = new or_track_filtered();
  const std::vector<uint64_t> qoff = qual_offsets(b);
  run_track(F, ref, b, aux, filter, qoff);
  if (F->track.status != PS_OK) return F;
  if (bases) run_bases(F, ref, b, aux, filter, qoff, bases);
  if (indels) run_indels(F, ref, b, aux, filter, qoff, indels);
  return F;
}

int or_track_filtered_status(const or_track_filtered* r, ps_track_counters* ctr, ps_fault* fault,
                             ps_track_filter_counters* fctr, ps_track_base_totals* bt, ps_track_indel_totals* it) {
  *fctr = r->fctr;
  *bt = r->base_totals;
  *it = r->indel_totals;
  return or_track_status(&r->track, ctr, fault);
}
// which = 0 / 1: runs of that strand, 2: sites, 3: base rows, 4: indel rows
int64_t or_track_filtered_copy(const or_track_filtered* r, int which, void* out, uint64_t max) {
  if (which < 3) return or_track_copy(&r->track, which, out, max);
  if (which == 3) {
    const uint64_t n = std::min<uint64_t>(max, r->base_rows.size());
    if (n) std::memcpy(out, r->base_rows.data(), n * sizeof(ps_track_base_row));
    return (int64_t)n;
  }
  const uint64_t n = std::min<uint64_t>(max, r->indel_rows.size());
  if (n) std::memcpy(out, r->indel_rows.data(), n * sizeof(ps_track_indel_row));
  return (int64_t)n;
}
void or_track_filtered_free(or_track_filtered* r) { delete r; }

}  // extern "C"
