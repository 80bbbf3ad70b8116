// The two tool loops over FILES, streaming and across several GPUs of one process (the entry points a JVM binds when
// it replaces ErrorProfiling.inferErrorProfile and PileupClusters.calculateReadPileups: Main.java:595-597, :634-636).
//
//   error profile : batches of records go round-robin to the contexts, every context accumulates its share, the int64
//                   accumulator vectors (< 10 KB) are summed on the host at the end (all outputs are commutative integer
//                   sums, SURVEY Q12; Java's int wrap-around is applied after the sum).
//   T>C pileup    : the file is taken in WINDOWS of records (PileupClusters.java:137 streams; a window is a shard in
//                   time).  The carry-in of a window -- Java's (tempClusterChr, tempClusterEnd) at its first record -- is
//                   the maximum (contig, end) over all earlier windows, known on the host from the decoded records before
//                   the window is launched, so windows go to the contexts round-robin and run while the next one is
//                   being decoded.  The reads at the head of a window that continue the cluster left open by the window
//                   before come back as a "head partial" and are folded into that cluster here (halo merge: counts,
//                   masks, strand state, T>C sites by position with their first-insertion keys, coverage re-read from the
//                   summed dense coverage of the boundary cluster).
//   clust files   : the merged closed clusters of every window go, with the window's records, through the flush
//                   arithmetic and the native writers (flush.cpp, clust_writer.cpp).
//   track         : windows round-robin over the contexts, each on a thread of its own while the next window decodes.
//                   A window reports final runs and sites for the positions after the maximum end of the windows before
//                   it and before its own last kept start; its head (up to that maximum end) and its tail (from its last
//                   kept start on) come back as dense arrays, added on the host into one pending region -- in a sorted
//                   file no later record reaches a position before the last kept start, so the region is bounded by the
//                   longest reference span of a record.
// No compute happens on the host: boundaries, masks, counts and sites all come from the kernels.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "internal.h"
#include "track.h"

extern "C" int open_for_ctx(ps_ctx* ctx, const char* bam_path, uint64_t max_batch, ps_bam** B);
int stage_batch(ps_ctx* ctx, const ps_read_batch* hb, bool with_qual, StagedBatch** out);

struct ps_multi {
  std::vector<ps_ctx*> ctx;
  bool owns = true;
  ps_packed_fasta* fasta = nullptr;
  std::string err;
  std::mutex err_mu;          // the window loop's sink thread reports errors too
};

static int multi_fail(ps_multi* m, int st, const std::string& msg) {
  if (m) {
    std::lock_guard<std::mutex> g(m->err_mu);
    m->err = msg;
  }
  return st;
}

namespace {

// max over the kept records of a host batch of their pileup keys (what pl_maxkey_kernel computes); rank: the context's
// contig order (ps_ctx::contig_rank)
uint64_t host_max_key(const ps_read_batch& b, const std::vector<uint64_t>& contig_off, const std::vector<uint32_t>& rank) {
  uint64_t best = 0, coff = (!b.uniform_ncigar && b.tile_cigar_off) ? b.tile_cigar_off[0] : 0;
  size_t ci = 0;
  for (uint64_t r = 0; r < b.n_reads; ++r) {
    const uint32_t meta = b.meta[r], flags = PS_META_FLAGS(meta), ncig = PS_META_NCIGAR(meta);
    const uint32_t* cig = b.cigar + coff;
    coff += ncig;
    if (flags & (PS_RF_UNMAPPED | PS_RF_POS_ZERO | PS_RF_CIGAR_OVERFLOW)) continue;
    bool hasI = false, hasD = false, hasN = false;
    uint64_t R = 0;
    for (uint32_t e = 0; e < ncig; ++e) {
      const uint32_t op = cig[e] & 15u;
      hasI |= op == 1u; hasD |= op == 2u; hasN |= op == 3u;
      if ((0x18Du >> op) & 1u) R += cig[e] >> 4;
    }
    if ((hasI || hasD) && hasN) continue;
    const uint64_t g = b.ref_start[r];
    if (g >= contig_off.back()) continue;
    if (!(g >= contig_off[ci] && g < contig_off[ci + 1]))
      ci = (size_t)(std::upper_bound(contig_off.begin(), contig_off.end(), g) - contig_off.begin()) - 1;
    const uint64_t end = g - contig_off[ci] + R;          // start + R - 1 with start = g - off + 1
    best = std::max(best, pileup_key(rank, (uint32_t)ci, (int32_t)(uint32_t)end));
  }
  return best;
}

struct OpenCluster {            // the cluster left open behind the windows taken so far
  bool have = false;
  ps_cluster c{};
  std::vector<ps_site> sites;
  int32_t cov_pos0 = 0;
  std::vector<uint32_t> cov;    // dense baseCoveredMap: cov[k] = coverage at cov_pos0 + k
};

// halo merge: the head partial of the next window (counts of the reads that continue the open cluster) into it
void merge_head(OpenCluster& o, const ps_cluster& hp, const std::vector<ps_site>& hs, int32_t hp_pos0,
                const std::vector<uint32_t>& hcov, uint64_t& double_stranded) {
  o.c.num_reads += hp.num_reads;
  o.c.num_t2c += hp.num_t2c;
  o.c.end = std::max(o.c.end, hp.end);
  o.c.mask51 |= hp.mask51;
  o.c.minus_after_first += hp.minus_after_first;
  if (!o.c.first_reverse) double_stranded += hp.minus_after_first;      // doubleStranded++ per minus member (:494-498)
  o.c.combined_strand = o.c.first_reverse ? 1 : (o.c.minus_after_first ? 2 : 0);
  // coverage: a site seen on one side of the cut is also covered by the other side's reads
  if (!hcov.empty()) {
    if (o.cov.empty()) { o.cov = hcov; o.cov_pos0 = hp_pos0; }
    else {
      const int64_t lo = std::min<int64_t>(o.cov_pos0, hp_pos0);
      const int64_t hi = std::max<int64_t>((int64_t)o.cov_pos0 + (int64_t)o.cov.size(), (int64_t)hp_pos0 + (int64_t)hcov.size());
      std::vector<uint32_t> sum((size_t)(hi - lo), 0);
      for (size_t k = 0; k < o.cov.size(); ++k) sum[(size_t)(o.cov_pos0 - lo) + k] += o.cov[k];
      for (size_t k = 0; k < hcov.size(); ++k) sum[(size_t)(hp_pos0 - lo) + k] += hcov[k];
      o.cov.swap(sum);
      o.cov_pos0 = (int32_t)lo;
    }
  }
  // sites: union by position; counts add, the first-insertion key is the smaller one
  std::vector<ps_site> all = o.sites;
  all.insert(all.end(), hs.begin(), hs.end());
  std::stable_sort(all.begin(), all.end(), [](const ps_site& a, const ps_site& b) { return a.pos < b.pos; });
  std::vector<ps_site> merged;
  for (const ps_site& s : all) {
    if (!merged.empty() && merged.back().pos == s.pos) {
      merged.back().t2c += s.t2c;
      merged.back().order_key = std::min(merged.back().order_key, s.order_key);
    } else merged.push_back(s);
  }
  for (ps_site& s : merged) {
    const int64_t k = (int64_t)s.pos - o.cov_pos0;
    s.cov = (k >= 0 && k < (int64_t)o.cov.size()) ? o.cov[(size_t)k] : 0u;
  }
  o.sites.swap(merged);
}

// what one window hands to its consumer: the clusters that closed with it (site_begin / site_end index `sites`), and the
// first read of the cluster still open behind it
struct WindowOut {
  ps_read_batch host{};        // copy of the window's batch descriptor (the arrays live in the batcher's slab)
  const ps_read_batch* batch;
  uint64_t first_ordinal;
  std::vector<ps_cluster> closed;
  std::vector<ps_site> sites;
  bool has_open;
  uint64_t open_first_read;
};
using WindowSink = std::function<int(const WindowOut&)>;

struct InFlight {
  ps_ctx* ctx = nullptr;
  ps_pileup* h = nullptr;
  ps_read_batch host{};       // the window's records (slab of the batcher: valid until the third-next ps_bam_next)
  uint64_t offset = 0;
  bool live = false;
};

int sync_fail(ps_multi* m, ps_ctx* c, int st) { return multi_fail(m, st, ps_last_error(c)); }

// The windowed pileup over an open file, every context keyed in the file's contig order.  counters / open: the run's
// totals and the cluster left open at the end.
int pileup_windows_run(ps_multi* m, ps_bam* B, const ps_pileup_opts* opts, const WindowSink& sink, ps_pileup_counters* counters,
                       OpenCluster* open_out, ps_fault* fault) {
  ps_ctx* c0 = m->ctx[0];
  int st = PS_OK;
  const std::vector<uint64_t>& contig_off = c0->contig_off;
  const uint32_t first_id = opts ? opts->first_running_id : 1u;
  uint64_t carry_key = 0;
  if (opts && opts->carry_valid) carry_key = pileup_key(c0->contig_rank, opts->carry_contig, opts->carry_cluster_end);
  memset(counters, 0, sizeof *counters);
  OpenCluster open;
  uint64_t created = 0, offset = 0, window = 0;
  InFlight fl[2];
  // The sink (the host writer of `clust`: cluster sequences, rows, files) runs on a thread of its own, one window at a
  // time and in file order, while this thread decodes the next window: the batcher keeps three slabs, so the records
  // of the window in the sink's hands stay valid until its successor has been handed over (which joins it first).
  std::thread sink_thread;
  int sink_rc = PS_OK;
  auto join_sink = [&]() -> int {
    if (sink_thread.joinable()) sink_thread.join();
    const int rc = sink_rc;
    sink_rc = PS_OK;
    return rc;
  };

  // completes window `f`: fetches its records, merges the boundary, hands the closed clusters to the sink
  auto complete = [&](InFlight& f) -> int {
    f.live = false;
    ps_ctx* c = f.ctx;
    int rc = ps_pileup_wait(f.h);
    if (rc != PS_OK) {
      if (rc == PS_ERR_REFERENCE_WOULD_THROW || rc == PS_ERR_UNSUPPORTED) {
        ps_pileup_fault(f.h, fault);
        fault->read_ordinal += f.offset;
      }
      multi_fail(m, rc, ps_last_error(c));
      ps_pileup_close(f.h);
      return rc;
    }
    ps_pileup_counters ctr;
    ps_pileup_counters_get(f.h, &ctr);
    counters->num_reads_processed += ctr.num_reads_processed;
    counters->skipped_due_indel += ctr.skipped_due_indel;
    counters->double_stranded += ctr.double_stranded;
    auto out_p = std::make_shared<WindowOut>();
    WindowOut& out = *out_p;
    out.host = f.host;
    out.batch = &out.host;
    out.first_ordinal = f.offset;
    // head partial -> the open cluster
    {
      ps_cluster hp;
      std::vector<ps_site> hs(1 << 12);
      int k = ps_pileup_head_partial(f.h, &hp, hs.data(), hs.size());
      if (k == PS_ERR_INVALID_ARG) { hs.resize(1 << 20); k = ps_pileup_head_partial(f.h, &hp, hs.data(), hs.size()); }
      if (k < 0) { ps_pileup_close(f.h); return multi_fail(m, k, "head partial"); }
      if (k > 0) {
        if (!open.have) { ps_pileup_close(f.h); return multi_fail(m, PS_ERR_STATE, "head partial without an open cluster"); }
        hs.resize(hp.site_end);
        for (ps_site& s : hs) s.order_key += f.offset << 6;
        int32_t p0 = 0;
        const int64_t ln = ps_pileup_boundary_coverage(f.h, 0, &p0, nullptr, 0);
        std::vector<uint32_t> cov((size_t)std::max<int64_t>(ln, 0));
        if (ln > 0) ps_pileup_boundary_coverage(f.h, 0, &p0, cov.data(), cov.size());
        merge_head(open, hp, hs, p0, cov, counters->double_stranded);
      }
    }
    const uint64_t n_closed = ctr.n_clusters, n_new = n_closed + (ctr.has_open_cluster ? 1 : 0);
    if (n_new && open.have) {            // the open cluster closes with this window's first new cluster
      ps_cluster c2 = open.c;
      c2.site_begin = 0;
      c2.site_end = open.sites.size();
      out.closed.push_back(c2);
      out.sites = open.sites;
      open = OpenCluster();
    }
    if (n_closed) {
      const size_t c_at = out.closed.size(), s_at = out.sites.size();
      out.closed.resize(c_at + n_closed);
      out.sites.resize(s_at + ctr.n_sites);
      const int64_t got = ps_pileup_next(f.h, 0, out.closed.data() + c_at, n_closed, out.sites.data() + s_at, ctr.n_sites);
      if (got != (int64_t)n_closed) { ps_pileup_close(f.h); return multi_fail(m, got < 0 ? (int)got : PS_ERR_STATE, "ps_pileup_next"); }
      for (size_t k = c_at; k < out.closed.size(); ++k) {
        out.closed[k].running_id += (uint32_t)created;
        out.closed[k].first_read += f.offset;
        out.closed[k].site_begin += s_at;
        out.closed[k].site_end += s_at;
      }
      for (size_t k = s_at; k < out.sites.size(); ++k) out.sites[k].order_key += f.offset << 6;
    }
    if (ctr.has_open_cluster) {
      std::vector<ps_site> os(1 << 12);
      int k = ps_pileup_open_cluster(f.h, &open.c, os.data(), os.size());
      if (k == PS_ERR_INVALID_ARG) { os.resize(1 << 20); k = ps_pileup_open_cluster(f.h, &open.c, os.data(), os.size()); }
      if (k <= 0) { ps_pileup_close(f.h); return multi_fail(m, k < 0 ? k : PS_ERR_STATE, "open cluster"); }
      os.resize(open.c.site_end);
      for (ps_site& s : os) s.order_key += f.offset << 6;
      open.sites.swap(os);
      open.c.first_read += f.offset;
      open.c.running_id += (uint32_t)created;
      int32_t p0 = 0;
      const int64_t ln = ps_pileup_boundary_coverage(f.h, 1, &p0, nullptr, 0);
      open.cov.assign((size_t)std::max<int64_t>(ln, 0), 0);
      if (ln > 0) ps_pileup_boundary_coverage(f.h, 1, &p0, open.cov.data(), open.cov.size());
      open.cov_pos0 = p0;
      open.have = true;
    }
    ps_pileup_close(f.h);
    created += n_new;
    out.has_open = open.have;
    out.open_first_read = open.have ? open.c.first_read : 0;
    counters->n_clusters += out.closed.size();
    counters->n_sites += out.sites.size();
    const int prev_rc = join_sink();                       // the window before this one has been written
    if (prev_rc != PS_OK) return prev_rc;
    sink_thread = std::thread([&sink, &sink_rc, out_p] { sink_rc = sink(*out_p); });
    return PS_OK;
  };

  for (;; ++window) {
    InFlight& f = fl[window & 1];
    // two windows in flight at most: the slab ps_bam_next is about to fill belongs to the window before last, whose
    // records the sink still needs -- complete it first (windows complete in file order)
    if (f.live) { st = complete(f); if (st) break; }
    ps_read_batch hb;
    const int k = ps_bam_next(B, &hb);
    if (k < 0) { st = multi_fail(m, k, ps_bam_error(B)); break; }
    if (k == 0) break;
    ps_ctx* c = m->ctx[window % m->ctx.size()];
    // a context takes one submitted call at a time (its scratch belongs to it): with a single context the window before
    // -- whose kernels ran while this one was being decoded -- completes before this one is launched
    InFlight& prev = fl[(window & 1) ^ 1];
    if (prev.live && prev.ctx == c) { st = complete(prev); if (st) break; }
    cudaSetDevice(c->device);
    // cluster ids are numbered from the window's own first cluster; the clusters opened by earlier windows are added
    // when the window completes (they are not known yet: those windows may still be running)
    ps_pileup_opts o{};
    o.first_running_id = first_id;
    if (carry_key) { o.carry_valid = 1; pileup_key_decode(c0->contig_by_rank, carry_key, &o.carry_contig, &o.carry_cluster_end); }
    f.ctx = c; f.host = hb; f.offset = offset;
    // upload without the quality bytes (the pileup never reads them: more than half of the records' bytes)
    StagedBatch* sb = nullptr;
    st = stage_batch(c, &hb, /*with_qual=*/false, &sb);
    if (st == PS_OK) {
      ps_read_batch view = hb;
      const DeviceBatch& v = sb->view;
      view.meta = v.meta; view.ref_start = v.ref_start; view.bases2 = v.bases2; view.qual = v.qual; view.cigar = v.cigar;
      view.tile_base_off = v.tile_base_off; view.tile_qual_off = v.tile_qual_off; view.tile_cigar_off = v.tile_cigar_off;
      view.tile_exc_off = v.tile_exc_off; view.exc = v.exc;
      st = ps_pileup_submit_device(c, &view, &o, nullptr, &f.h);
    }
    if (st != PS_OK) { sync_fail(m, c, st); break; }
    f.live = true;
    carry_key = std::max(carry_key, host_max_key(hb, contig_off, c0->contig_rank));
    offset += hb.n_reads;
  }
  for (int i = 0; i < 2 && st == PS_OK; ++i) {
    InFlight& f = fl[(window + i) & 1];
    if (f.live) st = complete(f);
  }
  {
    const int rc = join_sink();
    if (st == PS_OK) st = rc;
  }
  for (InFlight& f : fl)
    if (f.live) { ps_pileup_close(f.h); f.live = false; }
  if (st != PS_OK) return st;
  counters->has_open_cluster = open.have ? 1 : 0;
  if (open_out) *open_out = std::move(open);
  return PS_OK;
}

// Opens a file for a windowed tool.  The records follow the contig order of the file's header, which need not be the
// FASTA's: every context takes that order for the call (window carries and keys follow it) and has the caller's own order
// back afterwards, whatever the outcome.
int with_file_order(ps_multi* m, const char* bam_path, uint64_t window_reads, const std::function<int(ps_bam*)>& run) {
  ps_ctx* c0 = m->ctx[0];
  ps_bam* B = nullptr;
  int st = open_for_ctx(c0, bam_path, window_reads, &B);
  if (st) return sync_fail(m, c0, st);
  std::vector<uint32_t> file_order((size_t)std::max<int64_t>(ps_bam_contig_order(B, nullptr, 0), 0));
  ps_bam_contig_order(B, file_order.data(), file_order.size());
  std::vector<std::vector<uint32_t>> saved;
  for (ps_ctx* c : m->ctx) {
    if (!c->ref_loaded) { st = multi_fail(m, PS_ERR_STATE, "no reference loaded"); break; }
    saved.push_back(c->contig_by_rank);
    st = set_contig_order(c, file_order.data(), (uint32_t)file_order.size());
    if (st != PS_OK) { sync_fail(m, c, st); break; }
  }
  if (st == PS_OK) st = run(B);
  ps_bam_close(B);
  for (size_t i = 0; i < saved.size(); ++i) {
    const int rc = set_contig_order(m->ctx[i], saved[i].data(), (uint32_t)saved[i].size());
    if (rc != PS_OK && st == PS_OK) st = sync_fail(m, m->ctx[i], rc);
  }
  return st;
}

// The windowed pileup over a file.
int pileup_windows(ps_multi* m, const char* bam_path, const ps_pileup_opts* opts, uint64_t window_reads, const WindowSink& sink,
                   ps_pileup_counters* counters, OpenCluster* open_out, ps_fault* fault) {
  if (m->ctx.empty()) return multi_fail(m, PS_ERR_STATE, "no context");
  for (ps_ctx* c : m->ctx)
    if (c->pl_pending) return multi_fail(m, PS_ERR_STATE, "a submitted pileup call of a context has not been waited for");
  ps_ctx* c0 = m->ctx[0];
  if (opts && opts->carry_valid && opts->carry_contig >= c0->ref.n_contigs)
    return multi_fail(m, PS_ERR_INVALID_ARG, "carry_contig is not a contig of the reference");
  return with_file_order(m, bam_path, window_reads, [&](ps_bam* B) {
    return pileup_windows_run(m, B, opts, sink, counters, open_out, fault);
  });
}


// ---- track files -------------------------------------------------------------------------------------------------------
// The three files of the track tool.  Runs that touch with equal coverage are merged, so a run cut by a window boundary
// is one row.
struct TrackWriter {
  FILE* f[3] = {nullptr, nullptr, nullptr};      // plus bedGraph, minus bedGraph, t2c tsv
  std::vector<std::string> names;
  ps_track_run last[2]{};
  bool have[2] = {false, false};
  uint64_t rows[3] = {0, 0, 0};
  uint64_t merged[2] = {0, 0};                  // runs joined to the one before
  std::string buf[3];
  int open(const std::string& prefix) {
    const char* ext[3] = {".plus.bedGraph", ".minus.bedGraph", ".t2c.tsv"};
    for (int k = 0; k < 3; ++k) {
      f[k] = fopen((prefix + ext[k]).c_str(), "wb");
      if (!f[k]) return PS_ERR_IO;
    }
    buf[2] = "chrom\tpos\tstrand\tt2c\tcoverage\n";
    return PS_OK;
  }
  static void num(std::string& b, uint64_t v) {
    char t[24];
    int n = 0;
    do { t[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) b.push_back(t[--n]);
  }
  int drain(int k, bool force) {
    if (buf[k].size() < (1u << 20) && !force) return PS_OK;
    if (!buf[k].empty() && fwrite(buf[k].data(), 1, buf[k].size(), f[k]) != buf[k].size()) return PS_ERR_IO;
    buf[k].clear();
    return PS_OK;
  }
  int flush_run(int s) {
    if (!have[s]) return PS_OK;
    std::string& b = buf[s];
    b += names[last[s].contig]; b.push_back('\t');
    num(b, last[s].start0); b.push_back('\t');
    num(b, last[s].end0); b.push_back('\t');
    num(b, last[s].cov); b.push_back('\n');
    ++rows[s];
    have[s] = false;
    return drain(s, false);
  }
  int run(int s, const ps_track_run& r) {
    if (have[s] && last[s].contig == r.contig && last[s].end0 == r.start0 && last[s].cov == r.cov) {
      last[s].end0 = r.end0;
      ++merged[s];
      return PS_OK;
    }
    const int rc = flush_run(s);
    last[s] = r;
    have[s] = true;
    return rc;
  }
  int site(const ps_track_site& x) {
    std::string& b = buf[2];
    b += names[x.contig]; b.push_back('\t');
    num(b, (uint32_t)x.pos); b.push_back('\t');
    b.push_back(x.strand ? '-' : '+'); b.push_back('\t');
    num(b, x.t2c); b.push_back('\t');
    num(b, x.cov); b.push_back('\n');
    ++rows[2];
    return drain(2, false);
  }
  int finish() {
    int rc = PS_OK;
    for (int s = 0; s < 2; ++s) if (rc == PS_OK) rc = flush_run(s);
    for (int k = 0; k < 3; ++k) if (rc == PS_OK) rc = drain(k, true);
    return rc;
  }
  ~TrackWriter() { for (FILE* x : f) if (x) fclose(x); }
};

// what a window hands to the writer: final runs and sites, in file order
struct TrackRows {
  std::vector<ps_track_run> runs[2];
  std::vector<ps_track_site> sites;
};

// positions not final yet: [key0, key0 + len) of one contig, cov+, cov-, t2c+, t2c-
struct TrackPending {
  unsigned long long key0 = 0;
  std::vector<uint32_t> v[4];
  size_t len() const { return v[0].size(); }
  // rows of the positions before `upto` (keys), which leave the region
  void emit_before(unsigned long long upto, const std::vector<uint32_t>& by_rank, TrackRows& out) {
    const size_t n = len();
    size_t k_end = 0;
    if (upto > key0) k_end = (size_t)std::min<unsigned long long>(n, upto - key0);
    if ((upto >> 32) != (key0 >> 32)) k_end = upto > key0 ? n : 0;
    if (!k_end) return;
    const uint32_t contig = by_rank[(uint32_t)(key0 >> 32) - 1];
    const uint32_t p0 = (uint32_t)key0 - 1;         // 0-based position of entry 0
    for (int s = 0; s < 2; ++s)
      for (size_t k = 0; k < k_end; ++k) {
        const uint32_t c = v[s][k];
        if (!c) continue;
        std::vector<ps_track_run>& r = out.runs[s];
        if (!r.empty() && r.back().contig == contig && r.back().end0 == p0 + k && r.back().cov == c) r.back().end0++;
        else r.push_back(ps_track_run{contig, p0 + (uint32_t)k, p0 + (uint32_t)k + 1, c});
      }
    for (size_t k = 0; k < k_end; ++k)
      for (int s = 0; s < 2; ++s)
        if (v[2 + s][k]) out.sites.push_back(ps_track_site{contig, (int32_t)(p0 + k + 1), (uint32_t)s, v[2 + s][k], v[s][k]});
    for (auto& a : v) a.erase(a.begin(), a.begin() + (ptrdiff_t)k_end);
    key0 += k_end;
  }
};

struct TrackFlight {
  ps_ctx* ctx = nullptr;
  std::thread th;
  TrackOut out;
  int rc = PS_OK;
  std::string err;
  uint64_t offset = 0;
  bool live = false;
};

// The windowed track over an open file (contexts keyed in the file's contig order)
int track_windows_run(ps_multi* m, ps_bam* B, TrackWriter& W, ps_track_counters* ctr, ps_fault* fault) {
  ps_ctx* c0 = m->ctx[0];
  const std::vector<uint64_t>& contig_off = c0->contig_off;
  const std::vector<uint32_t>& by_rank = c0->contig_by_rank;
  memset(ctr, 0, sizeof *ctr);
  TrackPending P;
  unsigned long long last_start = 0, max_end = 0;     // over the windows launched so far / completed so far
  uint64_t offset = 0, window = 0;
  TrackFlight fl[2];
  std::thread sink_thread;
  int sink_rc = PS_OK;
  auto join_sink = [&]() -> int {
    if (sink_thread.joinable()) sink_thread.join();
    const int rc = sink_rc;
    sink_rc = PS_OK;
    return rc;
  };
  // PARASUITE_B200_DEBUG: per window, the kept records, the pending positions it made final and the pending length after it
  const bool dbg = getenv("PARASUITE_B200_DEBUG") != nullptr;
  auto print_window = [&](const TrackOut& o, size_t emitted) {
    if (dbg)
      fprintf(stderr, "[ps_track_window] kept %llu, emitted %zu, pending %zu\n", (unsigned long long)o.ctr.reads_counted,
              emitted, P.len());
  };
  auto complete = [&](TrackFlight& f) -> int {
    f.live = false;
    f.th.join();
    const TrackOut& o = f.out;
    if (f.rc != PS_OK) {
      if (o.fault.code && !fault->code) { *fault = o.fault; fault->read_ordinal += f.offset; }
      return multi_fail(m, f.rc, f.err);
    }
    ctr->num_reads_processed += o.ctr.num_reads_processed;
    ctr->unmapped += o.ctr.unmapped;
    ctr->skipped_due_indel += o.ctr.skipped_due_indel;
    ctr->reads_counted += o.ctr.reads_counted;
    ctr->fast_path_reads += o.ctr.fast_path_reads;
    for (int s = 0; s < 2; ++s) { ctr->aligned_bases[s] += o.ctr.aligned_bases[s]; ctr->t2c_events[s] += o.ctr.t2c_events[s]; }
    if (!o.first_key) { print_window(o, 0); return PS_OK; }      // no kept record: nothing changes
    if (o.first_key < last_start) return multi_fail(m, PS_ERR_UNSORTED, ps_strerror(PS_ERR_UNSORTED));
    if (o.head.len) {
      if (o.head.key0 < P.key0 || o.head.key0 + o.head.len > P.key0 + P.len())
        return multi_fail(m, PS_ERR_STATE, "track: window head outside the pending region");
      const size_t at = (size_t)(o.head.key0 - P.key0);
      for (int j = 0; j < 4; ++j)
        for (uint32_t k = 0; k < o.head.len; ++k) P.v[j][at + k] += o.head.v[(size_t)j * o.head.len + k];
    }
    auto rows = std::make_shared<TrackRows>();
    const size_t pending_before = P.len();
    P.emit_before(o.last_key, by_rank, *rows);
    const size_t emitted = pending_before - P.len();
    for (int s = 0; s < 2; ++s) rows->runs[s].insert(rows->runs[s].end(), o.runs[s].begin(), o.runs[s].end());
    rows->sites.insert(rows->sites.end(), o.sites.begin(), o.sites.end());
    if (o.tail.len) {
      if (P.len() && P.key0 + P.len() != o.tail.key0) return multi_fail(m, PS_ERR_STATE, "track: window tail not next to the pending region");
      if (!P.len()) P.key0 = o.tail.key0;
      for (int j = 0; j < 4; ++j) P.v[j].insert(P.v[j].end(), o.tail.v.begin() + (ptrdiff_t)j * o.tail.len, o.tail.v.begin() + (ptrdiff_t)(j + 1) * o.tail.len);
    }
    last_start = o.last_key;
    print_window(o, emitted);
    const int prev_rc = join_sink();
    if (prev_rc != PS_OK) return prev_rc;
    sink_thread = std::thread([&W, &sink_rc, rows] {
      int rc = PS_OK;
      for (int s = 0; s < 2 && rc == PS_OK; ++s)
        for (const ps_track_run& r : rows->runs[s]) if ((rc = W.run(s, r)) != PS_OK) break;
      for (const ps_track_site& x : rows->sites) if (rc != PS_OK || (rc = W.site(x)) != PS_OK) break;
      sink_rc = rc;
    });
    return PS_OK;
  };
  int st = PS_OK;
  for (;; ++window) {
    TrackFlight& f = fl[window & 1];
    if (f.live) { st = complete(f); if (st) break; }
    ps_read_batch hb;
    const int k = ps_bam_next(B, &hb);
    if (k < 0) { st = multi_fail(m, k, ps_bam_error(B)); break; }
    if (k == 0) break;
    ps_ctx* c = m->ctx[window % m->ctx.size()];
    TrackFlight& prev = fl[(window & 1) ^ 1];
    if (prev.live && prev.ctx == c) { st = complete(prev); if (st) break; }
    cudaSetDevice(c->device);
    StagedBatch* sb = nullptr;
    st = stage_batch(c, &hb, /*with_qual=*/false, &sb);     // the track reads no qualities
    if (st != PS_OK) { sync_fail(m, c, st); break; }
    f.ctx = c; f.offset = offset; f.rc = PS_OK; f.live = true;
    const DeviceBatch view = sb->view;
    const uint64_t prev_end = max_end;
    f.th = std::thread([&f, c, view, prev_end] {
      cudaSetDevice(c->device);
      f.rc = track_run(c, view, c->stream, true, prev_end, &f.out);
      if (f.rc != PS_OK) f.err = c->err;
    });
    max_end = std::max<unsigned long long>(max_end, host_max_key(hb, contig_off, c0->contig_rank));
    offset += hb.n_reads;
  }
  for (int i = 0; i < 2; ++i) {            // in file order; after an error only the threads are joined
    TrackFlight& f = fl[(window + i) & 1];
    if (!f.live) continue;
    if (st == PS_OK) st = complete(f);
    else { f.live = false; f.th.join(); }
  }
  {
    const int rc = join_sink();
    if (st == PS_OK) st = rc;
  }
  if (st != PS_OK) return st;
  TrackRows rest;
  P.emit_before(~0ull, by_rank, rest);
  for (int s = 0; s < 2 && st == PS_OK; ++s)
    for (const ps_track_run& r : rest.runs[s]) if ((st = W.run(s, r)) != PS_OK) break;
  for (const ps_track_site& x : rest.sites) if (st != PS_OK || (st = W.site(x)) != PS_OK) break;
  if (st == PS_OK) st = W.finish();
  if (st != PS_OK) return multi_fail(m, st, "track: writing the output files failed");
  ctr->n_runs[0] = W.rows[0];
  ctr->n_runs[1] = W.rows[1];
  ctr->n_sites = W.rows[2];
  if (dbg)
    fprintf(stderr, "[ps_track_files] runs %llu %llu, merged %llu %llu, sites %llu\n", (unsigned long long)W.rows[0],
            (unsigned long long)W.rows[1], (unsigned long long)W.merged[0], (unsigned long long)W.merged[1],
            (unsigned long long)W.rows[2]);
  return PS_OK;
}

}  // namespace

extern "C" {

// ---- several devices behind one handle --------------------------------------------------------------------------------
int ps_create_multi(ps_multi** out, const int* devices, int n) {
  if (!out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  std::vector<int> dev;
  if (devices && n > 0) dev.assign(devices, devices + n);
  else if (const char* e = getenv("PARASUITE_B200_DEVICES")) {      // "0,1,2"
    for (const char* p = e; *p;) {
      char* q = nullptr;
      const long v = strtol(p, &q, 10);
      if (q == p) break;
      dev.push_back((int)v);
      p = (*q == ',') ? q + 1 : q;
    }
  }
  if (dev.empty()) dev.push_back(0);
  ps_multi* m = new ps_multi();
  for (int d : dev) {
    ps_ctx* c = nullptr;
    const int st = ps_create(&c, d);
    if (st != PS_OK) {
      for (ps_ctx* x : m->ctx) ps_destroy(x);
      delete m;
      return st;
    }
    m->ctx.push_back(c);
  }
  *out = m;
  return PS_OK;
}

void ps_destroy_multi(ps_multi* m) {
  if (!m) return;
  if (m->owns)
    for (ps_ctx* c : m->ctx) ps_destroy(c);
  if (m->fasta) ps_fasta_free(m->fasta);
  delete m;
}

int ps_multi_device_count(const ps_multi* m) { return m ? (int)m->ctx.size() : 0; }
ps_ctx* ps_multi_context(ps_multi* m, int i) { return (m && i >= 0 && i < (int)m->ctx.size()) ? m->ctx[(size_t)i] : nullptr; }
const char* ps_multi_last_error(const ps_multi* m) { return m ? m->err.c_str() : "no object"; }

// FASTA (+ .fai) packed once on the host, resident in the HBM of every device
int ps_multi_load_fasta(ps_multi* m, const char* fasta_path) {
  if (!m || !fasta_path) return PS_ERR_INVALID_ARG;
  ps_packed_fasta* F = nullptr;
  int st = ps_fasta_pack(fasta_path, &F);
  if (st != PS_OK) {
    multi_fail(m, st, F ? ps_fasta_error(F) : "FASTA pack failed");
    ps_fasta_free(F);
    return st;
  }
  for (ps_ctx* c : m->ctx) {
    st = ps_reference_upload(c, ps_fasta_reference(F));
    if (st != PS_OK) { sync_fail(m, c, st); ps_fasta_free(F); return st; }
    if (c->fasta && !c->fasta_shared) ps_fasta_free(c->fasta);
    c->fasta = F;
    c->fasta_shared = true;
    c->fasta_path = fasta_path;
  }
  if (m->fasta) ps_fasta_free(m->fasta);
  m->fasta = F;
  return PS_OK;
}

// ErrorProfiling.inferErrorProfile's record loop (:104-409): batches round-robin over the devices, one host sum at the end
int ps_multi_profile_bam(ps_multi* m, const char* bam_path, const ps_profile_opts* opts, ps_profile_result* out) {
  if (!m || !bam_path || !opts || !out) return PS_ERR_INVALID_ARG;
  if (m->ctx.empty()) return multi_fail(m, PS_ERR_STATE, "no context");
  ps_bam* B = nullptr;
  uint64_t batch_reads = 1ull << 22;
  if (const char* e = getenv("PARASUITE_B200_BATCH_READS")) { const long long v = atoll(e); if (v > 0) batch_reads = (uint64_t)v; }
  int st = open_for_ctx(m->ctx[0], bam_path, batch_reads, &B);
  if (st) return sync_fail(m, m->ctx[0], st);
  ps_profile_opts o = *opts;
  o.emit_t2c_masks = 0;
  for (ps_ctx* c : m->ctx) {
    st = ps_profile_begin(c, &o);
    if (st) { sync_fail(m, c, st); break; }
  }
  uint64_t ordinal = 0, batch = 0;
  cudaEvent_t pending[2] = {nullptr, nullptr};        // upload of the batch that owns the slab about to be reused
  int pending_dev[2] = {0, 0};
  ps_read_batch hb;
  while (st == PS_OK) {
    if (pending[batch & 1]) { cudaSetDevice(pending_dev[batch & 1]); cudaEventSynchronize(pending[batch & 1]); pending[batch & 1] = nullptr; }
    const int k = ps_bam_next(B, &hb);
    if (k < 0) { st = multi_fail(m, k, ps_bam_error(B)); break; }
    if (k == 0) break;
    ps_ctx* c = m->ctx[batch % m->ctx.size()];
    c->reads_seen = ordinal;                           // fault ordinals are positions in the file, not in the context's share
    const int slot = c->staged_next;
    st = ps_profile_batch(c, &hb);
    if (st) { sync_fail(m, c, st); break; }
    pending[batch & 1] = c->staged_done[slot];
    pending_dev[batch & 1] = c->device;
    ordinal += hb.n_reads;
    ++batch;
  }
  // every context's accumulator, summed; the earliest fault wins
  const size_t n_acc = ps_profile_acc_len(o.max_read_length, o.infer_qualities);
  std::vector<int64_t> sum(n_acc, 0), part(n_acc);
  ps_fault first_fault{};
  int first_fault_st = PS_OK;
  std::string first_fault_msg;
  for (ps_ctx* c : m->ctx) {
    if (!c->profile_open) continue;
    ps_profile_result r;
    memset(&r, 0, sizeof r);
    r.wide = part.data();
    const int e = ps_profile_end(c, &r);
    if (e == PS_ERR_REFERENCE_WOULD_THROW || e == PS_ERR_UNSUPPORTED) {
      if (first_fault_st == PS_OK || r.fault.read_ordinal < first_fault.read_ordinal) {
        first_fault = r.fault; first_fault_st = e; first_fault_msg = ps_last_error(c);
      }
    } else if (e != PS_OK && st == PS_OK) st = sync_fail(m, c, e);
    else if (e == PS_OK)
      for (size_t k = 0; k < n_acc; ++k) sum[k] += part[k];
  }
  ps_bam_close(B);
  if (st != PS_OK) return st;
  out->fault.code = 0;
  out->fault.read_ordinal = 0;
  if (first_fault_st != PS_OK) {
    out->fault = first_fault;
    return multi_fail(m, first_fault_st, first_fault_msg);
  }
  profile_fill_result(make_layout(o.max_read_length, o.infer_qualities ? 1 : 0), sum.data(), out);
  return PS_OK;
}

static uint64_t window_reads_default() {
  uint64_t w = 1ull << 23;
  if (const char* e = getenv("PARASUITE_B200_WINDOW_READS")) { const long long v = atoll(e); if (v > 0) w = (uint64_t)v; }
  return std::min<uint64_t>(w, 0xFFFFFF00ull);
}

// PileupClusters.calculateReadPileups' record loop (:62-500), streaming: the handle holds the merged records of all
// windows on the host (ps_pileup_next / ps_pileup_open_cluster / ps_pileup_counters_get as usual)
int ps_multi_pileup_bam(ps_multi* m, const char* bam_path, const ps_pileup_opts* opts, ps_pileup** out) {
  if (!m || !bam_path || !out) return PS_ERR_INVALID_ARG;
  *out = nullptr;
  std::vector<ps_cluster> clusters;
  std::vector<ps_site> sites;
  ps_pileup_counters ctr;
  OpenCluster open;
  ps_fault fault{};
  const int st = pileup_windows(m, bam_path, opts, window_reads_default(), [&](const WindowOut& w) {
    const size_t s_at = sites.size();
    for (ps_cluster c : w.closed) { c.site_begin += s_at; c.site_end += s_at; clusters.push_back(c); }
    sites.insert(sites.end(), w.sites.begin(), w.sites.end());
    return PS_OK;
  }, &ctr, &open, &fault);
  if (st != PS_OK) {
    if (st == PS_ERR_REFERENCE_WOULD_THROW || st == PS_ERR_UNSUPPORTED) {      // a handle that only carries the fault
      ps_pileup_counters none{};
      ps_pileup* H = pileup_host_handle(m->ctx[0], {}, {}, false, ps_cluster{}, {}, 0, {}, none);
      *out = H;
      pileup_set_fault(H, fault);
    }
    return st;
  }
  if (open.have) { open.c.site_begin = 0; open.c.site_end = open.sites.size(); }
  *out = pileup_host_handle(m->ctx[0], std::move(clusters), std::move(sites), open.have, open.c, std::move(open.sites),
                            open.cov_pos0, std::move(open.cov), ctr);
  return PS_OK;
}

// The whole `clust` tool from files (PileupClusters.calculateReadPileups :62-584): <out>, <out>.ccr.fasta, <out>.ccr.tsv,
// <out>.report, <bam>.sitefrequency.tsv, <bam>.sitepositions.tsv.  snp_vcf may be NULL (no SNP filter).
int ps_multi_clust_bam(ps_multi* m, const char* bam_path, const char* out_path, const char* snp_vcf, uint32_t min_read_coverage,
                       ps_pileup_counters* counters_out, ps_fault* fault_out) {
  if (!m || !bam_path || !out_path) return PS_ERR_INVALID_ARG;
  if (m->ctx.empty() || !m->ctx[0]->fasta) return multi_fail(m, PS_ERR_STATE, "load the reference first (ps_multi_load_fasta)");
  ps_ctx* c0 = m->ctx[0];
  std::vector<const char*> names;
  for (uint32_t i = 0; i < c0->ref.n_contigs; ++i) names.push_back(ps_fasta_contig_name(c0->fasta, i));
  ps_flush* fl = nullptr;
  int st = ps_flush_create(&fl, min_read_coverage, (uint32_t)names.size(), names.data());
  if (st != PS_OK) return multi_fail(m, st, "ps_flush_create");
  if (snp_vcf && *snp_vcf) {
    st = ps_flush_load_vcf(fl, snp_vcf);
    if (st != PS_OK) { multi_fail(m, st, ps_flush_error(fl)); ps_flush_destroy(fl); return st; }
  }
  ps_clust_writer* w = nullptr;
  st = ps_clust_writer_open(&w, fl, c0->fasta_path.c_str(), out_path, bam_path);
  if (st != PS_OK) { multi_fail(m, st, ps_clust_writer_error(w)); ps_clust_writer_close(w); ps_flush_destroy(fl); return st; }
  ps_pileup_counters ctr;
  ps_fault fault{};
  st = pileup_windows(m, bam_path, nullptr, window_reads_default(), [&](const WindowOut& o) {
    const int rc = ps_clust_writer_feed(w, o.batch, o.first_ordinal, o.closed.data(), o.closed.size(), o.sites.data(),
                                        o.has_open ? 1 : 0, o.open_first_read);
    if (rc != PS_OK) {
      multi_fail(m, rc, ps_clust_writer_error(w));
      if (rc == PS_ERR_REFERENCE_WOULD_THROW) ps_clust_writer_fault(w, &fault);
    }
    return rc;
  }, &ctr, nullptr, &fault);
  if (st == PS_OK) {
    st = ps_clust_writer_finish(w, &ctr);
    if (st != PS_OK) multi_fail(m, st, ps_clust_writer_error(w));
  }
  if (counters_out) *counters_out = ctr;
  if (fault_out) *fault_out = fault;
  ps_clust_writer_close(w);
  ps_flush_destroy(fl);
  return st;
}

// ---- the single-context forms ------------------------------------------------------------------------------------------
static void borrow(ps_multi& m, ps_ctx* ctx) { m.ctx.assign(1, ctx); m.owns = false; }

int ps_pileup_bam(ps_ctx* ctx, const char* bam_path, const ps_pileup_opts* opts, ps_pileup** out) {
  if (!ctx || !bam_path || !out) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_multi m;
  borrow(m, ctx);
  const int st = ps_multi_pileup_bam(&m, bam_path, opts, out);
  if (st != PS_OK && !m.err.empty()) set_error(ctx, st, m.err);
  return st;
}

// The whole `error` tool from files (ErrorProfiling.inferErrorProfile, :96-621 without the plot): record loop on the
// GPU(s), the six output files natively.
int ps_multi_error_bam(ps_multi* m, const char* bam_path, const ps_profile_opts* opts, int32_t* counters_out, ps_fault* fault_out) {
  if (!m || !bam_path || !opts) return PS_ERR_INVALID_ARG;
  const uint32_t ml = opts->max_read_length;
  std::vector<int32_t> pc((size_t)ml * 16), qpm(16), qpmc(16), ctr(PS_PC_COUNT);
  std::vector<double> ins(ml), del(ml);
  std::vector<int64_t> qh(opts->infer_qualities ? (size_t)ml * 256 : 0);
  ps_profile_result r{};
  r.position_conversions = pc.data(); r.quality_per_mismatch = qpm.data(); r.quality_per_mismatch_counts = qpmc.data();
  r.insertions_per_pos = ins.data(); r.deletions_per_pos = del.data(); r.counters = ctr.data();
  r.quality_hist = opts->infer_qualities ? qh.data() : nullptr;
  int st = ps_multi_profile_bam(m, bam_path, opts, &r);
  if (fault_out) *fault_out = r.fault;
  if (st != PS_OK) return st;
  char err[512];
  st = ps_profile_write_files(&r, ml, opts->infer_qualities, bam_path, nullptr, err, sizeof err);
  if (st != PS_OK) return multi_fail(m, st, err);
  if (counters_out) memcpy(counters_out, ctr.data(), sizeof(int32_t) * PS_PC_COUNT);
  return PS_OK;
}

int ps_error_bam(ps_ctx* ctx, const char* bam_path, const ps_profile_opts* opts, int32_t* counters_out, ps_fault* fault_out) {
  if (!ctx || !bam_path || !opts) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_multi m;
  borrow(m, ctx);
  const int st = ps_multi_error_bam(&m, bam_path, opts, counters_out, fault_out);
  if (st != PS_OK && !m.err.empty()) set_error(ctx, st, m.err);
  return st;
}

int ps_clust_bam(ps_ctx* ctx, const char* bam_path, const char* out_path, const char* snp_vcf, uint32_t min_read_coverage,
                 ps_pileup_counters* counters_out, ps_fault* fault_out) {
  if (!ctx || !bam_path || !out_path) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_multi m;
  borrow(m, ctx);
  const int st = ps_multi_clust_bam(&m, bam_path, out_path, snp_vcf, min_read_coverage, counters_out, fault_out);
  if (st != PS_OK && !m.err.empty()) set_error(ctx, st, m.err);
  return st;
}

// The track tool from files: <out_prefix>.plus.bedGraph, .minus.bedGraph, .t2c.tsv
int ps_multi_track_bam(ps_multi* m, const char* bam_path, const char* out_prefix, ps_track_counters* counters_out,
                       ps_fault* fault_out) {
  if (!m || !bam_path || !out_prefix) return PS_ERR_INVALID_ARG;
  if (m->ctx.empty() || !m->ctx[0]->fasta) return multi_fail(m, PS_ERR_STATE, "load the reference first (ps_multi_load_fasta)");
  ps_ctx* c0 = m->ctx[0];
  TrackWriter W;
  for (uint32_t i = 0; i < c0->ref.n_contigs; ++i) W.names.push_back(ps_fasta_contig_name(c0->fasta, i));
  int st = W.open(out_prefix);
  if (st != PS_OK) return multi_fail(m, st, std::string("cannot write ") + out_prefix + ".*");
  ps_track_counters ctr{};
  ps_fault fault{};
  st = with_file_order(m, bam_path, window_reads_default(), [&](ps_bam* B) { return track_windows_run(m, B, W, &ctr, &fault); });
  if (counters_out) *counters_out = ctr;
  if (fault_out) *fault_out = fault;
  return st;
}

int ps_track_bam(ps_ctx* ctx, const char* bam_path, const char* out_prefix, ps_track_counters* counters_out,
                 ps_fault* fault_out) {
  if (!ctx || !bam_path || !out_prefix) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_multi m;
  borrow(m, ctx);
  const int st = ps_multi_track_bam(&m, bam_path, out_prefix, counters_out, fault_out);
  if (st != PS_OK && !m.err.empty()) set_error(ctx, st, m.err);
  return st;
}

}  // extern "C"
