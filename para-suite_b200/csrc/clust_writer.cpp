// Output files of the `clust` tool, natively: what PileupClusters.java does with every closed cluster AFTER the
// arithmetic of the flush (flush.cpp) -- the cluster sequence it assembles read by read (:367-414 initial, :421-487
// extension, mergeByteArrays / mergeByteSubArrays :723-748), the cluster row (:317-343), the CCR FASTA / TSV rows
// (:262-315) -- and the end-of-run files (.report :502-514, sitefrequency / sitepositions :529-545).
// (reference: /root/reference/src/src/utils/pileupclusters/PileupClusters.java)
//
// Host code, no GPU needed.  The record loop itself stays on the GPU: this writer is FED with the SoA batches the
// kernels saw (for the CIGARs the sequence assembly walks) and with the closed cluster records they produced; it never
// decides a cluster boundary itself -- a read opens a cluster iff its ordinal is the first_read of the next record.
// The sequence quirks are kept: only M and D elements fetch reference bytes, every non-I element (S, H, N, P, =, X too)
// advances the fetch cursor, an element that starts behind the cluster end is PREPENDED, raw FASTA case is kept,
// the strand of the first read reverse-complements the sequence at flush.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <deque>
#include <string>
#include <thread>
#include <vector>

#include "parasuite_b200.h"
#include "java_double.h"
#include "record.h"

namespace {

struct RawFasta {      // IndexedFastaSequenceFile: raw bytes (case kept) by contig and 1-based inclusive range
  struct Entry { std::string name; uint64_t len, offset, linebases, linewidth; };
  std::vector<Entry> e;
  std::vector<uint64_t> off;     // cumulative lengths = the global coordinate space of the packed reference
  const uint8_t* p = nullptr;
  size_t n = 0;
  int fd = -1;
  ~RawFasta() {
    if (p) munmap((void*)p, n);
    if (fd >= 0) close(fd);
  }
  bool open(const char* path, std::string& err) {
    const std::string fp = std::string(path) + ".fai";
    FILE* f = fopen(fp.c_str(), "r");
    if (!f) { err = "cannot open " + fp; return false; }
    char line[4096];
    while (fgets(line, sizeof line, f)) {
      char name[2048];
      unsigned long long a, b, c, d;
      if (sscanf(line, "%2047[^\t]\t%llu\t%llu\t%llu\t%llu", name, &a, &b, &c, &d) != 5) continue;
      if (c == 0 || d < c) { fclose(f); err = "malformed .fai line"; return false; }
      e.push_back({name, a, b, c, d});
    }
    fclose(f);
    if (e.empty()) { err = "empty FASTA index"; return false; }
    fd = ::open(path, O_RDONLY);
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0) { err = std::string("cannot open ") + path; return false; }
    n = (size_t)st.st_size;
    void* m = n ? mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0) : nullptr;
    if (n && m == MAP_FAILED) { err = std::string("cannot map ") + path; return false; }
    p = (const uint8_t*)m;
    off.assign(1, 0);
    for (auto& x : e) off.push_back(off.back() + x.len);
    return true;
  }
  // 0: ok; 1: SAMException (start > stop + 1, stop past the contig, unknown contig); 2: start < 1 -- htsjdk then reads
  // file bytes in front of the contig (or dies on a negative file position), which is not emulated
  int fetch(int64_t contig, int64_t start, int64_t stop, std::string& out) const {
    out.clear();
    if (contig < 0 || contig >= (int64_t)e.size()) return 1;
    if (start > stop + 1) return 1;
    const Entry& x = e[(size_t)contig];
    if (stop > (int64_t)x.len) return 1;
    if (start < 1) return 2;
    const size_t len = (size_t)(stop - start + 1);
    out.resize(len);
    // one division for the first base, then whole line segments (a division per base was most of the writer's time)
    const uint64_t b0 = (uint64_t)(start - 1);
    uint64_t col = x.linebases ? b0 % x.linebases : 0;
    uint64_t at = x.offset + (x.linebases ? b0 / x.linebases * x.linewidth : 0) + col;
    size_t k = 0;
    while (k < len) {
      const size_t run = x.linebases ? (size_t)std::min<uint64_t>(len - k, x.linebases - col) : len - k;
      if (at + run <= n) memcpy(&out[k], p + at, run);
      else
        for (size_t j = 0; j < run; ++j) out[k + j] = at + j < n ? (char)p[at + j] : 'N';
      k += run;
      at += run + (x.linewidth - x.linebases);
      col = 0;
    }
    return 0;
  }
};

struct CompTable {     // htsjdk SequenceUtil.reverseComplement: only ACGTacgt are mapped
  unsigned char t[256];
  CompTable() {
    for (int c = 0; c < 256; ++c) t[c] = (unsigned char)c;
    const char* from = "ACGTacgt"; const char* to = "TGCAtgca";
    for (int k = 0; k < 8; ++k) t[(unsigned char)from[k]] = (unsigned char)to[k];
  }
};
const CompTable kComp;

void reverse_complement(char* s, size_t n) {
  for (size_t i = 0; i < n / 2; ++i) {
    const char a = (char)kComp.t[(unsigned char)s[i]], b = (char)kComp.t[(unsigned char)s[n - 1 - i]];
    s[i] = b; s[n - 1 - i] = a;
  }
  if (n & 1) s[n / 2] = (char)kComp.t[(unsigned char)s[n / 2]];
}

const char* kStrand[3] = {"+", "-", "+/-"};

}  // namespace

// Row text is put together by hand (raw appends into one growing buffer per file, written out a megabyte at a time):
// the rows are the writer's whole cost -- three fprintf calls with a dozen conversions each were 4 us per cluster, and
// std::string appends with their capacity checks and temporaries were still 2.5.
struct RowBuf {
  char* d = nullptr;
  size_t n = 0, cap = 0;
  RowBuf() = default;
  RowBuf(const RowBuf&) = delete;
  RowBuf& operator=(const RowBuf&) = delete;
  RowBuf(RowBuf&& o) noexcept : d(o.d), n(o.n), cap(o.cap) { o.d = nullptr; o.n = o.cap = 0; }
  ~RowBuf() { free(d); }
  char* room(size_t need) {               // a cursor with `need` bytes behind it; took() says how far it got
    if (n + need > cap) {
      cap = std::max<size_t>((n + need) * 2, (size_t)1 << 16);
      d = (char*)realloc(d, cap);
      if (!d) abort();
    }
    return d + n;
  }
  void took(char* end) { n = (size_t)(end - d); }
  void append(const RowBuf& o) { if (o.n) { char* p = room(o.n); memcpy(p, o.d, o.n); n += o.n; } }
  void flush_to(FILE* f, bool force) {
    if (n >= ((size_t)1 << 20) || (force && n)) { fwrite(d, 1, n, f); n = 0; }
  }
};
static inline char* put_s(char* p, const char* s, size_t n) { memcpy(p, s, n); return p + n; }
static inline char* put_s(char* p, const std::string& s) { return put_s(p, s.data(), s.size()); }
static inline char* put_i(char* p, long long v) { return std::to_chars(p, p + 24, v).ptr; }
static inline char* put_u(char* p, unsigned long long v) { return std::to_chars(p, p + 24, v).ptr; }

struct ps_clust_writer {
  ps_flush* flush = nullptr;
  RawFasta fa;
  FILE *f_pileup = nullptr, *f_ccr_fa = nullptr, *f_ccr_tsv = nullptr, *f_report = nullptr, *f_sitefreq = nullptr,
       *f_sitepos = nullptr;
  std::string err;
  ps_fault fault{};
  // the cluster being assembled (Java: tempClusterBytes, tempClusterEnd)
  bool have = false;
  std::string bytes;
  RowBuf b_pileup, b_ccr_fa, b_ccr_tsv;      // rows not yet written
  struct Job { ps_cluster c; ps_flush_row row; std::string bytes; };
  std::vector<Job> jobs;                     // closed clusters of the feed in progress, rows still to be formatted
  int64_t cluster_end = 0;
  uint64_t cluster_first = 0;
  // closed records waiting for their cluster to end in the read stream
  struct Pending { ps_cluster c; ps_flush_row row; };
  std::deque<Pending> pending;
  std::deque<uint64_t> starts;        // first_read ordinals of clusters that have not begun yet
  uint64_t reads_fed = 0, rows_written = 0, ccr_written = 0, ccr_start_before_contig = 0;
};

static int cw_fail(ps_clust_writer* w, int st, const std::string& m) { w->err = m; return st; }

static void cw_close_files(ps_clust_writer* w) {
  if (w->f_pileup) w->b_pileup.flush_to(w->f_pileup, true);
  if (w->f_ccr_fa) w->b_ccr_fa.flush_to(w->f_ccr_fa, true);
  if (w->f_ccr_tsv) w->b_ccr_tsv.flush_to(w->f_ccr_tsv, true);
  for (FILE** f : {&w->f_pileup, &w->f_ccr_fa, &w->f_ccr_tsv, &w->f_report, &w->f_sitefreq, &w->f_sitepos})
    if (*f) { fclose(*f); *f = nullptr; }
}

// rows of one closed cluster (PileupClusters.java:262-343)
struct RowOut { RowBuf pileup, ccr_fa, ccr_tsv; uint64_t rows = 0, ccr = 0, ccr_before = 0; };

static void cw_format_cluster(const ps_clust_writer* w, const ps_cluster& c, const ps_flush_row& row, const std::string& bytes,
                              RowOut& O) {
  if (!row.emitted) return;                                            // numReadsPerCluster < minReadCoverage (:180)
  static const std::string unknown("?");
  const std::string& chr = c.contig < w->fa.e.size() ? w->fa.e[c.contig].name : unknown;
  char id[64 + 2048];                                                  // "cl_" + running id + "_" + chromosome (:356)
  size_t id_n;
  {
    char* p = put_s(id, "cl_", 3);
    p = put_u(p, c.running_id);
    *p++ = '_';
    p = put_s(p, chr.data(), std::min<size_t>(chr.size(), 2047));      // (.fai names are read with %2047[^\t])
    id_n = (size_t)(p - id);
  }
  const char* comb = kStrand[c.combined_strand < 3 ? c.combined_strand : 2];
  const size_t comb_n = strlen(comb);
  char fraction[40];
  const size_t fraction_n = (size_t)(java_double_to(fraction, row.fraction) - fraction);
  const size_t fixed = id_n + chr.size() + 512;                        // everything in a row but the sequences
  if (row.has_ccr) {                                                         // tempBestMutationPos > 0 (:262)
    thread_local std::string ccr;
    const int rc = w->fa.fetch(c.contig, (int64_t)row.best_pos - 20, (int64_t)row.best_pos + 20, ccr);
    if (rc == 2) O.ccr_before++;
    if (rc != 0) ccr.clear();                                                // catch (SAMException) -> new byte[0] (:278)
    else if (c.combined_strand == 1) reverse_complement(&ccr[0], ccr.size());   // getStrandOrientation().equals("-") (:271)
    for (char& ch : ccr) ch = (char)(ch - ((ch >= 'a' && ch <= 'z') ? 32 : 0));   // :283-288
    {
      char* p = O.ccr_fa.room(fixed + ccr.size());
      *p++ = '>'; p = put_s(p, id, id_n); p = put_s(p, " 20-anchor-20 ", 14); p = put_s(p, chr); *p++ = ':';
      p = put_s(p, comb, comb_n); *p++ = ':'; p = put_i(p, row.best_pos - 20); *p++ = '-'; p = put_i(p, row.best_pos + 20);
      *p++ = '\n'; p = put_s(p, ccr); *p++ = '\n';
      O.ccr_fa.took(p);
    }
    {
      char* p = O.ccr_tsv.room(fixed + ccr.size());
      p = put_s(p, "Gene\t", 5); p = put_s(p, id, id_n); *p++ = '\t'; p = put_s(p, comb, comb_n); *p++ = '\t';
      p = put_s(p, chr); *p++ = '\t'; p = put_i(p, c.start); *p++ = '\t'; p = put_i(p, c.end); *p++ = '\t';
      p = put_i(p, row.best_pos - 20); *p++ = '\t'; p = put_i(p, row.best_pos + 20); *p++ = '\t'; p = put_s(p, ccr); *p++ = '\t';
      p = put_i(p, row.best_pos); *p++ = '\t'; p = put_u(p, c.num_reads); *p++ = '\t'; p = put_u(p, row.num_t2c_sites);
      *p++ = '\t'; p = put_u(p, row.best_count); *p++ = '\t'; p = java_double_to(p, row.best_value); *p++ = '\t';
      p = put_u(p, c.num_t2c); *p++ = '\t'; p = put_s(p, fraction, fraction_n); *p++ = '\n';
      O.ccr_tsv.took(p);
    }
    O.ccr++;
  }
  {
    char* p = O.pileup.room(fixed + bytes.size());
    p = put_s(p, id, id_n); *p++ = '\t'; p = put_s(p, chr); *p++ = '\t'; p = put_i(p, c.start); *p++ = '\t'; p = put_i(p, c.end);
    *p++ = '\t'; *p++ = c.first_reverse ? '-' : '+'; *p++ = '\t'; p = put_u(p, c.num_reads); *p++ = '\t'; p = put_u(p, c.num_t2c);
    *p++ = '\t'; p = put_u(p, row.num_t2c_sites); *p++ = '\t'; p = put_s(p, fraction, fraction_n); *p++ = '\t';
    char* seq = p;
    p = put_s(p, bytes);
    if (c.first_reverse) reverse_complement(seq, bytes.size());               // :318-321, in place in the row
    *p++ = '\t'; p = put_s(p, comb, comb_n); *p++ = '\t'; p = put_u(p, bytes.size()); *p++ = '\n';
    O.pileup.took(p);
  }
  O.rows++;
}

// Formats the rows of the queued clusters on all host threads (the clusters are independent once the flush arithmetic
// has run; every thread takes a contiguous range) and appends them to the files in cluster order.
static void cw_write_jobs(ps_clust_writer* w) {
  const size_t n = w->jobs.size();
  if (n == 0) return;
  const unsigned hw = std::thread::hardware_concurrency();
  const size_t T = std::max<size_t>(1, std::min<size_t>({(size_t)(hw ? hw : 1), (size_t)16, n / 256 + 1}));
  std::vector<RowOut> outs(T);
  auto work = [&](size_t t) {
    for (size_t k = n * t / T; k < n * (t + 1) / T; ++k) cw_format_cluster(w, w->jobs[k].c, w->jobs[k].row, w->jobs[k].bytes, outs[t]);
  };
  if (T == 1) work(0);
  else {
    std::vector<std::thread> pool;
    for (size_t t = 0; t < T; ++t) pool.emplace_back(work, t);
    for (auto& th : pool) th.join();
  }
  // every file takes its pieces in cluster order; the three files are written side by side
  auto put_all = [&](RowBuf& held, RowBuf RowOut::*which, FILE* f) {
    for (size_t t = 0; t < T; ++t) {
      RowBuf& fresh = outs[t].*which;
      if (fresh.n >= ((size_t)1 << 16)) { held.flush_to(f, true); fwrite(fresh.d, 1, fresh.n, f); }   // a large piece goes out as it is
      else { held.append(fresh); held.flush_to(f, false); }
    }
  };
  if (n >= 4096) {
    std::thread a([&] { put_all(w->b_ccr_fa, &RowOut::ccr_fa, w->f_ccr_fa); }), b([&] { put_all(w->b_ccr_tsv, &RowOut::ccr_tsv, w->f_ccr_tsv); });
    put_all(w->b_pileup, &RowOut::pileup, w->f_pileup);
    a.join(); b.join();
  } else {
    put_all(w->b_pileup, &RowOut::pileup, w->f_pileup); put_all(w->b_ccr_fa, &RowOut::ccr_fa, w->f_ccr_fa); put_all(w->b_ccr_tsv, &RowOut::ccr_tsv, w->f_ccr_tsv);
  }
  for (size_t t = 0; t < T; ++t) { w->rows_written += outs[t].rows; w->ccr_written += outs[t].ccr; w->ccr_start_before_contig += outs[t].ccr_before; }
  w->jobs.clear();
}

// ---- cluster sequence, read by read (PileupClusters.java:146-157, :347-480) ------------------------------------------------
// The sequence of a cluster depends on the reads from its first one on and on nothing in front of it, and the first reads
// are known before the loop starts (the kernels found them), so the records of a feed are walked in ranges that begin
// at a cluster start, one range per host thread; the first range continues the cluster the previous feed left open.
struct SeqState { bool have = false; uint64_t cluster_first = 0; int64_t cluster_end = 0; std::string bytes; };
struct RangeOut {
  std::vector<std::pair<uint64_t, std::string>> done;      // clusters that ended inside the range: first read, sequence
  SeqState st;                                             // the cluster open at the end of the range
  size_t starts_used = 0;
  int status = PS_OK;
  uint64_t fault_ordinal = 0;
  const char* msg = nullptr;
};
static const char* const kDisagree = "cluster records and read stream disagree (records must be fed in order)";
static const char* const kFetchPast = "cluster sequence: FASTA fetch past the contig (the JVM would die here)";

static void cw_walk_range(const ps_clust_writer* w, const ps_read_batch* hb, uint64_t first_ordinal, uint64_t r_lo, uint64_t r_hi,
                          uint64_t coff, const uint64_t* starts, size_t n_starts, RangeOut& O) {
  SeqState& st = O.st;
  std::string piece;
  size_t sc = 0;
  auto stop = [&](int status, const char* msg, uint64_t ordinal) { O.status = status; O.msg = msg; O.fault_ordinal = ordinal; O.starts_used = sc; };
  for (uint64_t r = r_lo; r < r_hi; ++r) {
    const uint32_t meta = hb->meta[r], flags = PS_META_FLAGS(meta), ncig = PS_META_NCIGAR(meta);
    const uint32_t* cig = hb->cigar + coff;
    coff += ncig;
    const uint64_t ordinal = first_ordinal + r;
    const CigarShape<int64_t> shape = cigar_shape<int64_t>(cig, ncig);
    if ((flags & PS_RF_UNMAPPED) || shape.skip) {                              // :146, :152-157
      if (sc < n_starts && starts[sc] == ordinal) return stop(PS_ERR_STATE, kDisagree, ordinal);   // a cluster cannot begin here
      continue;
    }
    // contig and 1-based start from the global offset (same coordinate space as the packed reference)
    const uint64_t g = hb->ref_start[r];
    size_t ci = 0;
    {
      size_t lo = 0, hi = w->fa.e.size();
      while (hi - lo > 1) { const size_t mid = (lo + hi) / 2; if (w->fa.off[mid] <= g) lo = mid; else hi = mid; }
      ci = lo;
    }
    const int64_t start = (int64_t)(g - w->fa.off[ci]) + 1, end = start + shape.ref_span - 1;
    if (sc < n_starts && starts[sc] == ordinal) {
      ++sc;
      if (st.have) O.done.emplace_back(st.cluster_first, std::move(st.bytes));   // the previous cluster is flushed (:178)
      st.have = true;
      st.cluster_first = ordinal;
      st.cluster_end = end;                                                 // :347
      st.bytes.clear();                                                     // :367
      int64_t cur = start;
      for (uint32_t e = 0; e < ncig; ++e) {
        const uint32_t op = cig[e] & 15u;
        const int64_t len = cig[e] >> 4;
        if (op == 2u || op == 0u) {                                         // D or M only (:383-386)
          if (w->fa.fetch((int64_t)ci, cur, cur + len - 1, piece) != 0)     // SAMException outside any try block: the JVM dies here
            return stop(PS_ERR_REFERENCE_WOULD_THROW, kFetchPast, ordinal);
          st.bytes += piece;
        }
        if (op != 1u) cur += len;                                           // every non-I element advances (:402-404)
      }
    } else {
      if (!st.have) return stop(PS_ERR_STATE, "a kept read in front of the first cluster start", ordinal);
      if (end > st.cluster_end) {                                           // :421
        int64_t cur = start;
        for (uint32_t e = 0; e < ncig; ++e) {
          const uint32_t op = cig[e] & 15u;
          const int64_t len = cig[e] >> 4;
          if (cur + len - 1 < st.cluster_end) {                             // :429-436
            if (op != 1u) cur += len;
            continue;
          }
          if (op == 2u || op == 0u) {
            if (w->fa.fetch((int64_t)ci, cur, cur + len - 1, piece) != 0) return stop(PS_ERR_REFERENCE_WOULD_THROW, kFetchPast, ordinal);
            const int64_t overhang = st.cluster_end - cur + 1;              // :449
            if (overhang > 0) st.bytes.append(piece, (size_t)overhang, std::string::npos);   // mergeByteSubArrays (:453-457)
            else st.bytes.insert(0, piece);                                 // mergeByteArrays(additionalNucs, tempClusterBytes) (:462)
          }
          st.cluster_end = end;                                             // :480, inside the element loop
          if (op != 1u) cur += len;
        }
      }
    }
  }
  O.starts_used = sc;
}

extern "C" {

int ps_clust_writer_open(ps_clust_writer** out, ps_flush* flush, const char* fasta_path, const char* out_path,
                         const char* bam_path) {
  if (!out) return PS_ERR_INVALID_ARG;
  ps_clust_writer* w = new ps_clust_writer();
  *out = w;                       // returned even on failure so the caller can read the message
  if (!flush || !fasta_path || !out_path || !bam_path) return cw_fail(w, PS_ERR_INVALID_ARG, "NULL argument");
  w->flush = flush;
  if (!w->fa.open(fasta_path, w->err)) return PS_ERR_IO;
  const std::string o = out_path, b = bam_path;
  struct { FILE** f; std::string path; } files[] = {
      {&w->f_pileup, o}, {&w->f_sitefreq, b + ".sitefrequency.tsv"}, {&w->f_ccr_fa, o + ".ccr.fasta"},
      {&w->f_ccr_tsv, o + ".ccr.tsv"}, {&w->f_sitepos, b + ".sitepositions.tsv"}, {&w->f_report, o + ".report"}};   // :73-83
  for (auto& f : files) {
    *f.f = fopen(f.path.c_str(), "w");
    if (!*f.f) { cw_close_files(w); return cw_fail(w, PS_ERR_IO, "cannot create " + f.path); }
  }
  fputs("ClusterID\tChr\tStart\tEnd\tStrand\t#reads\t#T2C\t#T2C sites\tT2C Fraction\tSeqenece\tCombStrand\tSeqLength\n",
        w->f_pileup);                                                                                                  // :94-96
  fputs("Protein_Group\tCluster ID\tStrand\tChromosome\tCluster_Begin\tCluster_End\tAnchor_FlankSeq_Begin\tAnchor_FlankSeq_End"
        "\tAnchor_FlankSeq\tAnchor_Position\tCluster_Clone_Count\tNumber_of_T2C_Positions\tT2C_Freq_at_Anchor_Position"
        "\tT2C_Fract_at_Anchor_Position\tT2C_Freq_Whole_Cluster\tT2C_Fract_Whole_Cluster\n", w->f_ccr_tsv);            // :98-104
  return PS_OK;
}

const char* ps_clust_writer_error(const ps_clust_writer* w) { return w ? w->err.c_str() : "no object"; }

int ps_clust_writer_fault(const ps_clust_writer* w, ps_fault* out) {
  if (!w || !out) return PS_ERR_INVALID_ARG;
  *out = w->fault;
  return PS_OK;
}

// One batch of records in file order (host SoA, ordinals first_ordinal ...), the clusters that closed with it -- in
// order, flushed here through ps_flush_clusters -- and the first read of the cluster still open behind it.
int ps_clust_writer_feed(ps_clust_writer* w, const ps_read_batch* hb, uint64_t first_ordinal, const ps_cluster* closed,
                         uint64_t n_closed, const ps_site* sites, int has_open, uint64_t open_first_read) {
  if (!w || !hb || (n_closed && !closed)) return PS_ERR_INVALID_ARG;
  if (!w->f_pileup) return cw_fail(w, PS_ERR_STATE, "writer is closed");
  if (hb->n_reads && (!hb->meta || !hb->cigar || !hb->ref_start || !hb->bases2 || !hb->qual))
    return cw_fail(w, PS_ERR_INVALID_ARG, "the writer reads the records on the host: the compact upload form (flags8 / uniform_cigar) is not accepted here");
  // a record whose cluster begins in this batch announces a start; so does the cluster still open behind the batch.  (A
  // record of a cluster that began in an earlier batch was announced then, as that batch's open cluster.)
  std::vector<uint64_t> starts(w->starts.begin(), w->starts.end());
  w->starts.clear();
  for (uint64_t k = 0; k < n_closed; ++k)
    if (closed[k].first_read >= first_ordinal) starts.push_back(closed[k].first_read);
  if (has_open && open_first_read >= first_ordinal) starts.push_back(open_first_read);
  const uint64_t n = hb->n_reads;
  // ---- ranges of records, each beginning at a cluster start --------------------------------------------------------------
  const unsigned hw = std::thread::hardware_concurrency();
  size_t T = std::max<size_t>(1, std::min<size_t>({(size_t)(hw ? hw : 1), (size_t)16, (size_t)(n / 32768 + 1)}));
  if (const char* e = getenv("PARASUITE_B200_WRITER_THREADS")) T = std::max(1, atoi(e));
  bool ordered = true;                   // the starts the kernels return are ascending ordinals inside the batch
  for (size_t k = 0; k < starts.size() && ordered; ++k)
    ordered = starts[k] >= first_ordinal && starts[k] - first_ordinal < n && (k == 0 || starts[k - 1] < starts[k]);
  if (!ordered) T = 1;                   // (anything else is walked as one range, which reports it)
  std::vector<size_t> cut{0};            // range t takes starts [cut[t], cut[t + 1])
  for (size_t t = 1; t < T; ++t) {
    const size_t k = (size_t)(std::lower_bound(starts.begin(), starts.end(), first_ordinal + n * t / T) - starts.begin());
    if (k > cut.back() && k < starts.size()) cut.push_back(k);
  }
  T = cut.size();
  cut.push_back(starts.size());
  std::vector<uint64_t> r_lo(T + 1, 0), coff0(T, 0);
  for (size_t t = 1; t < T; ++t) r_lo[t] = starts[cut[t]] - first_ordinal;
  r_lo[T] = n;
  coff0[0] = (!hb->uniform_ncigar && hb->tile_cigar_off) ? hb->tile_cigar_off[0] : 0;
  if (T > 1) {                           // cigar offset of every range's first record
    uint64_t c = coff0[0];
    size_t t = 1;
    for (uint64_t r = 0; r < n && t < T; ++r) {
      if (r == r_lo[t]) coff0[t++] = c;
      c += PS_META_NCIGAR(hb->meta[r]);
    }
  }
  std::vector<RangeOut> outs(T);
  outs[0].st.have = w->have;
  outs[0].st.cluster_first = w->cluster_first;
  outs[0].st.cluster_end = w->cluster_end;
  outs[0].st.bytes = std::move(w->bytes);
  w->bytes.clear();
  std::vector<std::thread> pool;
  for (size_t t = 1; t < T; ++t)
    pool.emplace_back([&, t] { cw_walk_range(w, hb, first_ordinal, r_lo[t], r_lo[t + 1], coff0[t], starts.data() + cut[t], cut[t + 1] - cut[t], outs[t]); });
  std::thread first;
  if (T > 1) first = std::thread([&] { cw_walk_range(w, hb, first_ordinal, r_lo[0], r_lo[1], coff0[0], starts.data(), cut[1], outs[0]); });
  // ---- meanwhile: arithmetic of the flush for the new records, in order (running state lives in the flush object) --------
  std::vector<ps_flush_row> rows(n_closed);
  const int flush_st = n_closed ? ps_flush_clusters(w->flush, closed, n_closed, sites, rows.data()) : PS_OK;
  if (T == 1) cw_walk_range(w, hb, first_ordinal, 0, n, coff0[0], starts.data(), starts.size(), outs[0]);
  else first.join();
  for (auto& th : pool) th.join();
  if (flush_st != PS_OK) return cw_fail(w, flush_st, ps_flush_error(w->flush));
  for (uint64_t k = 0; k < n_closed; ++k) w->pending.push_back({closed[k], rows[k]});
  // ---- the ranges in order: a cluster that ended pairs up with the oldest closed record still waiting -------------------
  auto close_cluster = [&](uint64_t first_read, std::string&& bytes) {
    if (w->pending.empty() || w->pending.front().c.first_read != first_read) return false;
    w->jobs.push_back({w->pending.front().c, w->pending.front().row, std::move(bytes)});
    w->pending.pop_front();
    return true;
  };
  SeqState carry;
  carry.have = false;
  for (size_t t = 0; t < T; ++t) {
    RangeOut& O = outs[t];
    bool ok = true;
    if (t > 0) {
      // range t begins with the first read of a cluster: the one open at the end of range t - 1 ended there -- unless
      // range t stopped before it took that read
      if (O.starts_used == 0 && O.status != PS_OK) ok = true;
      else if (carry.have) ok = close_cluster(carry.cluster_first, std::move(carry.bytes));
    }
    for (size_t k = 0; ok && k < O.done.size(); ++k) ok = close_cluster(O.done[k].first, std::move(O.done[k].second));
    if (ok && O.status == PS_OK && O.starts_used != cut[t + 1] - cut[t] && T > 1) { ok = false; }
    if (!ok || O.status != PS_OK) {
      cw_write_jobs(w);
      if (!ok) return cw_fail(w, PS_ERR_STATE, kDisagree);
      if (O.status == PS_ERR_REFERENCE_WOULD_THROW) { w->fault.code = PS_THROW_REF_RANGE; w->fault.read_ordinal = O.fault_ordinal; }
      return cw_fail(w, O.status, O.msg);
    }
    carry = std::move(O.st);
  }
  for (size_t k = outs[T - 1].starts_used + cut[T - 1]; k < starts.size(); ++k) w->starts.push_back(starts[k]);
  w->have = carry.have;
  w->cluster_first = carry.cluster_first;
  w->cluster_end = carry.cluster_end;
  w->bytes = std::move(carry.bytes);
  w->reads_fed += n;
  cw_write_jobs(w);
  return PS_OK;
}

// End of the run (PileupClusters.java:502-545): the last cluster is never flushed; .report, sitefrequency and
// sitepositions are written, every file is closed.
int ps_clust_writer_finish(ps_clust_writer* w, const ps_pileup_counters* totals) {
  if (!w || !totals) return PS_ERR_INVALID_ARG;
  if (!w->f_pileup) return cw_fail(w, PS_ERR_STATE, "writer is closed");
  ps_flush_totals t;
  ps_flush_totals_get(w->flush, &t, nullptr, 0);
  std::vector<double> afi(t.n_allele_frequency);
  ps_flush_totals_get(w->flush, &t, afi.data(), afi.size());
  fprintf(w->f_report, "Double stranded clusters found: %llu\n", (unsigned long long)totals->double_stranded);
  fprintf(w->f_report, "Loci found that are SNPs: 0\n");                                  // `SNPs` is never incremented (:135)
  fprintf(w->f_report, "%llu insertion or deletion skipped\n", (unsigned long long)totals->skipped_due_indel);
  fprintf(w->f_report, "T-C mutations identified as SNPs: %llu\n", (unsigned long long)t.snp_hit);
  fprintf(w->f_report, "T-C mutations identified as SNVs (100%% T-C in 1 site): %llu\n", (unsigned long long)t.high_frequent_error);
  for (double v : afi) fprintf(w->f_sitefreq, "%s\n", java_double(v / (double)t.num_crosslinked_clusters).c_str());   // :531-536
  for (int j = 0; j < 51; ++j)
    fprintf(w->f_sitepos, "%s\n", java_double((double)t.allele_positions[j] / (double)t.num_allele_positions).c_str());   // :538-543
  cw_close_files(w);
  return PS_OK;
}

void ps_clust_writer_stats(const ps_clust_writer* w, uint64_t* rows, uint64_t* ccr_rows, uint64_t* ccr_start_before_contig) {
  if (!w) return;
  if (rows) *rows = w->rows_written;
  if (ccr_rows) *ccr_rows = w->ccr_written;
  if (ccr_start_before_contig) *ccr_start_before_contig = w->ccr_start_before_contig;
}

void ps_clust_writer_close(ps_clust_writer* w) {
  if (!w) return;
  cw_close_files(w);
  delete w;
}

}  // extern "C"
