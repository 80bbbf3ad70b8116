// Host batcher: FASTA(+.fai) -> packed reference, BGZF/BAM -> SoA read batches in page-locked memory.
//
// Stands in for what htsjdk does for the two Java loops (reference: /root/reference/src/src/utils/errorprofile/
// ErrorProfiling.java:104-110 opens the BAM with SamReaderFactory and the FASTA with IndexedFastaSequenceFile; the
// loops then see SAMRecord objects in file order).  The record view presented to the kernels is the one SURVEY.md 8(b)
// lists: POS+1 (0 when POS = -1), flags 0x4 / 0x10 / 0x400, cigar ops 0..8 = MIDNSHP=X, bases from 4-bit nibbles via
// "=ACMGRSVTWYHKDBN" (only A, C, G, T are countable), raw phred bytes (first byte 0xFF = missing), header sort order.
//
// BGZF blocks are independent deflate streams: the block table is scanned once (sequential, 18 bytes per block), the
// blocks of a window are inflated by a pool of threads straight into their place of one contiguous buffer, records are
// located with a cheap sequential hop over block_size fields, and the SoA arrays are filled by the same pool
// (thread ranges are multiples of the 256-read tile so the per-tile offset tables fall out of one prefix sum).
#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "internal.h"

namespace {

struct MappedFile {
  const uint8_t* p = nullptr;
  size_t n = 0;
  int fd = -1;
  bool open(const char* path) {
    fd = ::open(path, O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0) { ::close(fd); fd = -1; return false; }
    n = (size_t)st.st_size;
    if (n == 0) { p = nullptr; return true; }
    void* m = mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) { ::close(fd); fd = -1; return false; }
    p = static_cast<const uint8_t*>(m);
    return true;
  }
  ~MappedFile() {
    if (p) munmap(const_cast<uint8_t*>(p), n);
    if (fd >= 0) ::close(fd);
  }
};

template <typename F>
void parallel_for(int threads, uint64_t n, F f) {   // f(thread, lo, hi) over [0, n) in contiguous ranges
  if (threads < 1) threads = 1;
  if ((uint64_t)threads > n) threads = n ? (int)n : 1;
  if (threads == 1) { f(0, (uint64_t)0, n); return; }
  std::vector<std::thread> pool;
  for (int t = 0; t < threads; ++t) {
    const uint64_t lo = n * t / threads, hi = n * (t + 1) / threads;
    pool.emplace_back([=] { f(t, lo, hi); });
  }
  for (auto& th : pool) th.join();
}

inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline uint16_t rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// FASTA
// ---------------------------------------------------------------------------------------------------------
struct ps_packed_fasta {
  std::vector<std::string> names;
  std::vector<uint64_t> off;          // [n+1]
  std::vector<uint32_t> seq2, inv;
  std::vector<const char*> name_ptrs;
  ps_reference view{};
  std::string err;
};

static int fasta_pack(const char* path, ps_packed_fasta* F, int threads) {
  struct Fai { std::string name; uint64_t len, offset, linebases, linewidth; };
  std::vector<Fai> fai;
  {
    const std::string fp = std::string(path) + ".fai";
    FILE* f = fopen(fp.c_str(), "r");
    if (!f) { F->err = "cannot open " + fp + " (the FASTA index is required, as for htsjdk's IndexedFastaSequenceFile)"; return PS_ERR_IO; }
    char line[4096];
    while (fgets(line, sizeof line, f)) {
      char name[2048];
      unsigned long long a, b, c, d;
      if (sscanf(line, "%2047[^\t]\t%llu\t%llu\t%llu\t%llu", name, &a, &b, &c, &d) != 5) continue;
      if (c == 0 || d < c) { fclose(f); F->err = "malformed .fai line"; return PS_ERR_FORMAT; }
      fai.push_back({name, a, b, c, d});
    }
    fclose(f);
  }
  if (fai.empty()) { F->err = "empty FASTA index"; return PS_ERR_FORMAT; }
  MappedFile mf;
  if (!mf.open(path)) { F->err = std::string("cannot open ") + path; return PS_ERR_IO; }
  F->off.assign(1, 0);
  for (auto& e : fai) { F->names.push_back(e.name); F->off.push_back(F->off.back() + e.len); }
  const uint64_t n = F->off.back();
  if (n >= (1ull << 32)) { F->err = "reference >= 2^32 bases"; return PS_ERR_UNSUPPORTED; }
  for (size_t c = 0; c < fai.size(); ++c) {
    const Fai& e = fai[c];
    const uint64_t bytes = e.len ? (e.len - 1) / e.linebases * e.linewidth + (e.len - 1) % e.linebases + 1 : 0;
    if (e.offset + bytes > mf.n) { F->err = "FASTA shorter than its index says (" + e.name + ")"; return PS_ERR_FORMAT; }
  }
  F->seq2.assign((n + 15) / 16 + 8, 0);
  F->inv.assign((n + 31) / 32 + 8, 0);
  uint8_t code[256];
  memset(code, 4, sizeof code);
  code['A'] = code['a'] = 0; code['C'] = code['c'] = 1; code['G'] = code['g'] = 2; code['T'] = code['t'] = 3;
  // chunks of 2^20 bases aligned to 32: threads never share a word
  const uint64_t chunk = 1u << 20, n_chunks = (n + chunk - 1) / chunk;
  uint32_t* seq2 = F->seq2.data();
  uint32_t* inv = F->inv.data();
  const std::vector<uint64_t>& off = F->off;
  parallel_for(threads, n_chunks, [&](int, uint64_t lo, uint64_t hi) {
    for (uint64_t ch = lo; ch < hi; ++ch) {
      uint64_t g = ch * chunk;
      const uint64_t gend = std::min(n, g + chunk);
      size_t c = std::upper_bound(off.begin(), off.end(), g) - off.begin() - 1;
      while (g < gend) {
        while (off[c + 1] <= g) ++c;
        const Fai& e = fai[c];
        const uint64_t in = g - off[c];                                   // position inside the contig
        const uint64_t stop = std::min(gend, off[c + 1]);
        uint64_t line = in / e.linebases, col = in % e.linebases;
        const uint8_t* src = mf.p + e.offset + line * e.linewidth + col;
        while (g < stop) {
          const uint64_t take = std::min<uint64_t>(e.linebases - col, stop - g);
          for (uint64_t k = 0; k < take; ++k, ++g) {
            const uint8_t cd = code[src[k]];
            if (cd == 4) inv[g >> 5] |= 1u << (g & 31);
            else seq2[g >> 4] |= (uint32_t)cd << (2 * (g & 15));
          }
          src += take + (e.linewidth - e.linebases);
          if (col + take < e.linebases) src -= (e.linewidth - e.linebases);   // stopped inside a line
          col = 0;
        }
      }
    }
  });
  for (auto& s : F->names) F->name_ptrs.push_back(s.c_str());
  F->view.n_bases = n;
  F->view.seq2 = F->seq2.data();
  F->view.inv = F->inv.data();
  F->view.n_contigs = (uint32_t)F->names.size();
  F->view.contig_off = F->off.data();
  return PS_OK;
}

// ---------------------------------------------------------------------------------------------------------
// BAM
// ---------------------------------------------------------------------------------------------------------
namespace {

// Page-locked slabs are expensive to make (cudaHostAlloc pins every page: ~0.1 s for a window of a few million reads),
// and a process that runs `error` and then `clust` on one file, or a file after the other, would pay that per call: a
// closed batcher hands its slabs to a small process-wide pool (at most kSlabPoolBytes), the next one takes them from there.
struct SlabMem { uint8_t* p; size_t cap; };
constexpr size_t kSlabPoolBytes = (size_t)3 << 30;
std::mutex g_slab_mu;
std::vector<SlabMem> g_slab_pool;
size_t g_slab_pool_bytes = 0;

struct Slab {            // one SoA batch in a single (page-locked when possible) allocation
  uint8_t* p = nullptr;
  size_t cap = 0;
  bool pinned = false;
  void release() {
    if (!p) return;
    if (pinned) {
      std::lock_guard<std::mutex> g(g_slab_mu);
      if (g_slab_pool_bytes + cap <= kSlabPoolBytes && g_slab_pool.size() < 8) {
        g_slab_pool.push_back({p, cap});
        g_slab_pool_bytes += cap;
        p = nullptr; cap = 0;
        return;
      }
    }
    if (pinned) cudaFreeHost(p); else free(p);
    p = nullptr; cap = 0;
  }
  bool reserve(size_t n) {
    if (n <= cap) return true;
    release();
    {
      std::lock_guard<std::mutex> g(g_slab_mu);
      int best = -1;
      for (int k = 0; k < (int)g_slab_pool.size(); ++k)
        if (g_slab_pool[k].cap >= n && (best < 0 || g_slab_pool[k].cap < g_slab_pool[best].cap)) best = k;
      if (best >= 0) {
        p = g_slab_pool[best].p; cap = g_slab_pool[best].cap; pinned = true;
        g_slab_pool_bytes -= cap;
        g_slab_pool.erase(g_slab_pool.begin() + best);
        return true;
      }
    }
    const size_t want = n + n / 8 + 4096;
    void* q = nullptr;
    if (cudaHostAlloc(&q, want, cudaHostAllocDefault) == cudaSuccess) { p = (uint8_t*)q; pinned = true; }
    else { cudaGetLastError(); p = (uint8_t*)malloc(want); pinned = false; }
    if (!p) return false;
    cap = want;
    return true;
  }
};

struct Block { uint64_t coff; uint32_t clen, isize; };

struct ByteBuf {         // growable byte buffer without value-initialisation (inflate writes every byte it exposes)
  uint8_t* p = nullptr;
  size_t n = 0, cap = 0;
  ~ByteBuf() { free(p); }
  uint8_t* data() { return p; }
  const uint8_t* data() const { return p; }
  size_t size() const { return n; }
  bool grow_to(size_t want) {       // keeps the first n bytes
    if (want > cap) {
      size_t c = cap ? cap : ((size_t)1 << 20);
      while (c < want) c += c / 2 + 4096;
      uint8_t* q = (uint8_t*)realloc(p, c);
      if (!q) return false;
      p = q; cap = c;
    }
    n = want;
    return true;
  }
  void drop_front(size_t k) {       // discard the first k bytes
    if (k == 0) return;
    if (k < n) memmove(p, p + k, n - k);
    n -= k;
  }
};

}  // namespace

struct ps_bam {
  MappedFile mf;
  std::vector<Block> blocks;
  size_t next_block = 0;
  ByteBuf buf;                     // inflated bytes not yet consumed
  size_t head = 0;
  bool header_done = false;
  bool sorted = false;
  std::vector<std::string> ref_names;
  std::vector<int64_t> ref_to_contig;   // BAM refID -> FASTA contig (-1: absent from the FASTA)
  std::vector<uint32_t> contig_order;   // FASTA contigs in @SQ order, those the FASTA lacks left out (ps_bam_contig_order)
  const ps_packed_fasta* fa = nullptr;
  uint64_t max_batch = 0;
  int threads = 1;
  Slab slab[3];                    // a batch's arrays stay valid until the third-next ps_bam_next: the file tools keep one
  int cur = 0;                     // window on the device, one with the host writer and fill the third
  uint64_t ordinal = 0;
  std::string err;
  std::vector<uint64_t> rec_off;   // scratch: offsets of the records of the batch being built
  // SAM text input (htsjdk opens SAM and BAM through one factory, ErrorProfiling.java:104-107): the text is turned into
  // the byte stream an inflated BAM would give -- header, then records in BAM encoding -- so everything behind
  // bam_fill is shared
  bool sam_text = false;
  size_t sam_at = 0;               // next unread byte of the text
  std::unordered_map<std::string, int32_t> sam_ref_id;
  double t_fill = 0, t_locate = 0, t_pass1 = 0, t_pass2 = 0;   // seconds (PARASUITE_B200_BATCHER_TIMING=1 prints them)
};

static int bam_fail(ps_bam* B, int st, const std::string& m) { B->err = m; return st; }

static int bam_scan_blocks(ps_bam* B) {
  const uint8_t* p = B->mf.p;
  const size_t n = B->mf.n;
  size_t o = 0;
  while (o < n) {
    if (o + 18 > n || p[o] != 0x1f || p[o + 1] != 0x8b || p[o + 2] != 8 || !(p[o + 3] & 4))
      return bam_fail(B, PS_ERR_FORMAT, "not a BGZF file (bad block header)");
    const uint32_t xlen = rd16(p + o + 10);
    uint32_t bsize = 0;
    size_t x = o + 12;
    const size_t xend = x + xlen;
    if (xend > n) return bam_fail(B, PS_ERR_FORMAT, "truncated BGZF block");
    while (x + 4 <= xend) {
      const uint32_t slen = rd16(p + x + 2);
      if (x + 4 + (size_t)slen > xend) return bam_fail(B, PS_ERR_FORMAT, "BGZF extra subfield runs past the extra field");
      if (p[x] == 'B' && p[x + 1] == 'C' && slen == 2) bsize = (uint32_t)rd16(p + x + 4) + 1;
      x += 4 + slen;
    }
    if (bsize < xlen + 20 || o + bsize > n) return bam_fail(B, PS_ERR_FORMAT, "truncated BGZF block");
    const uint32_t isize = rd32(p + o + bsize - 4);
    if (isize) B->blocks.push_back({o + 12 + xlen, bsize - xlen - 20, isize});
    o += bsize;
  }
  return PS_OK;
}

// inflate blocks until at least `want` unconsumed bytes are buffered (or the file ends)
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// ---- SAM text ---------------------------------------------------------------------------------------------------
static void put32(ByteBuf& b, size_t at, uint32_t v) { memcpy(b.data() + at, &v, 4); }

// header lines ('@...') -> "BAM\1" l_text text n_ref (l_name name l_ref)*
static int sam_header(ps_bam* B) {
  const uint8_t* p = B->mf.p;
  const size_t n = B->mf.n;
  size_t o = 0;
  std::vector<std::pair<std::string, uint32_t>> refs;
  while (o < n && p[o] == '@') {
    size_t e = o;
    while (e < n && p[e] != '\n') ++e;
    const std::string line((const char*)p + o, e - o);
    if (line.compare(0, 3, "@SQ") == 0) {
      std::string name;
      uint32_t len = 0;
      size_t a = 0;
      while (a < line.size()) {
        size_t b = line.find('\t', a);
        if (b == std::string::npos) b = line.size();
        if (line.compare(a, 3, "SN:") == 0) name = line.substr(a + 3, b - a - 3);
        if (line.compare(a, 3, "LN:") == 0) len = (uint32_t)strtoul(line.c_str() + a + 3, nullptr, 10);
        a = b + 1;
      }
      while (!name.empty() && name.back() == '\r') name.pop_back();
      B->sam_ref_id.emplace(name, (int32_t)refs.size());
      refs.emplace_back(name, len);
    }
    o = e < n ? e + 1 : e;
  }
  const std::string text((const char*)p, o);
  size_t bytes = 12 + text.size();
  for (auto& r : refs) bytes += 8 + r.first.size() + 1;
  if (!B->buf.grow_to(bytes)) return bam_fail(B, PS_ERR_OOM, "out of host memory");
  uint8_t* d = B->buf.data();
  memcpy(d, "BAM\1", 4);
  put32(B->buf, 4, (uint32_t)text.size());
  memcpy(d + 8, text.data(), text.size());
  size_t at = 8 + text.size();
  put32(B->buf, at, (uint32_t)refs.size());
  at += 4;
  for (auto& r : refs) {
    put32(B->buf, at, (uint32_t)r.first.size() + 1);
    memcpy(d + at + 4, r.first.c_str(), r.first.size() + 1);
    put32(B->buf, at + 4 + r.first.size() + 1, r.second);
    at += 8 + r.first.size() + 1;
  }
  B->sam_at = o;
  return PS_OK;
}

// alignment lines -> BAM records, until `want` unconsumed bytes are buffered or the text ends.  What SAMLineParser hands
// the loops: FLAG, RNAME, POS, CIGAR, SEQ (upper-cased, '.' -> N: SAMRecord.setReadString), QUAL - 33 ('*' -> none).
static int sam_fill(ps_bam* B, size_t want) {
  auto nib = [](uint8_t c) -> uint8_t {
    switch (c >= 'a' && c <= 'z' ? c - 32 : c) {
      case '=': return 0; case 'A': return 1; case 'C': return 2; case 'M': return 3; case 'G': return 4; case 'R': return 5;
      case 'S': return 6; case 'V': return 7; case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11;
      case 'K': return 12; case 'D': return 13; case 'B': return 14; default: return 15;          // N, '.', anything else
    }
  };
  const uint8_t* p = B->mf.p;
  const size_t n = B->mf.n;
  while (B->buf.size() - B->head < want && B->sam_at < n) {
    size_t o = B->sam_at, e = o;
    while (e < n && p[e] != '\n') ++e;
    B->sam_at = e < n ? e + 1 : e;
    size_t le = e;
    while (le > o && (p[le - 1] == '\r')) --le;
    if (le == o) continue;                                                       // blank line
    const char* f[11];
    size_t fl[11];
    int nf = 0;
    for (size_t a = o; nf < 11;) {
      size_t b = a;
      while (b < le && p[b] != '\t') ++b;
      f[nf] = (const char*)p + a; fl[nf] = b - a; ++nf;
      if (b >= le) break;
      a = b + 1;
    }
    if (nf < 11) return bam_fail(B, PS_ERR_FORMAT, "SAM alignment line with fewer than 11 fields");
    const uint32_t flag = (uint32_t)strtoul(std::string(f[1], fl[1]).c_str(), nullptr, 10);
    const std::string rname(f[2], fl[2]);
    int32_t ref_id = -1;
    if (rname != "*") { auto it = B->sam_ref_id.find(rname); if (it != B->sam_ref_id.end()) ref_id = it->second; }
    const int32_t pos = (int32_t)strtol(std::string(f[3], fl[3]).c_str(), nullptr, 10) - 1;
    std::vector<uint32_t> cig;
    if (!(fl[5] == 1 && f[5][0] == '*')) {
      uint32_t num = 0;
      for (size_t k = 0; k < fl[5]; ++k) {
        const char c = f[5][k];
        if (c >= '0' && c <= '9') { num = num * 10 + (uint32_t)(c - '0'); continue; }
        const char* ops = "MIDNSHP=X";
        const char* w = strchr(ops, c);
        if (!w || !c) return bam_fail(B, PS_ERR_FORMAT, "SAM: unknown CIGAR operator");
        cig.push_back((num << 4) | (uint32_t)(w - ops));
        num = 0;
      }
    }
    if (cig.size() > 0xFFFFu) return bam_fail(B, PS_ERR_UNSUPPORTED, "SAM: more than 65535 CIGAR operations");
    const bool no_seq = fl[9] == 1 && f[9][0] == '*';
    const uint32_t l_seq = no_seq ? 0u : (uint32_t)fl[9];
    const bool no_qual = (fl[10] == 1 && f[10][0] == '*') || fl[10] != l_seq;
    const uint32_t bs = 32 + 2 + 4 * (uint32_t)cig.size() + (l_seq + 1) / 2 + l_seq;
    const size_t at = B->buf.size();
    if (!B->buf.grow_to(at + 4 + bs)) return bam_fail(B, PS_ERR_OOM, "out of host memory for the records");
    uint8_t* d = B->buf.data() + at;
    memset(d, 0, 4 + bs);
    put32(B->buf, at, bs);
    put32(B->buf, at + 4, (uint32_t)ref_id);
    put32(B->buf, at + 8, (uint32_t)pos);
    d[12] = 2;                                                                   // l_read_name ("r\0": names are never read)
    const uint16_t ncg = (uint16_t)cig.size(), fl16 = (uint16_t)flag;
    memcpy(d + 16, &ncg, 2);
    memcpy(d + 18, &fl16, 2);
    put32(B->buf, at + 20, l_seq);
    put32(B->buf, at + 24, 0xFFFFFFFFu);
    put32(B->buf, at + 28, 0xFFFFFFFFu);
    d[36] = 'r';
    uint8_t* q = d + 38;
    if (!cig.empty()) memcpy(q, cig.data(), 4 * cig.size());
    q += 4 * cig.size();
    for (uint32_t k = 0; k < l_seq; ++k) q[k >> 1] |= (uint8_t)(nib((uint8_t)f[9][k]) << ((~k & 1) * 4));
    q += (l_seq + 1) / 2;
    for (uint32_t k = 0; k < l_seq; ++k) q[k] = no_qual ? 0xFF : (uint8_t)((uint8_t)f[10][k] - 33);
  }
  return PS_OK;
}

static int bam_fill(ps_bam* B, size_t want) {
  const double t0 = now_s();
  struct Acc { ps_bam* b; double t0; ~Acc() { b->t_fill += now_s() - t0; } } acc{B, t0};
  if (B->sam_text) return sam_fill(B, want);
  while (B->buf.size() - B->head < want && B->next_block < B->blocks.size()) {
    // a window of blocks: enough for `want`, at least 64 MB when a big batch is being assembled
    size_t b1 = B->next_block, total = 0;
    const size_t target = std::max<size_t>(want - (B->buf.size() - B->head), (size_t)128 << 20);
    std::vector<size_t> at;
    while (b1 < B->blocks.size() && total < target) { at.push_back(total); total += B->blocks[b1].isize; ++b1; }
    const size_t base = B->buf.size();
    if (!B->buf.grow_to(base + total)) return bam_fail(B, PS_ERR_OOM, "out of host memory for the inflated records");
    std::atomic<int> bad{0};
    const size_t b0 = B->next_block;
    parallel_for(B->threads, b1 - b0, [&](int, uint64_t lo, uint64_t hi) {
      z_stream zs;
      memset(&zs, 0, sizeof zs);
      if (inflateInit2(&zs, -15) != Z_OK) { bad = 1; return; }
      for (uint64_t k = lo; k < hi; ++k) {
        const Block& bl = B->blocks[b0 + k];
        inflateReset(&zs);
        zs.next_in = const_cast<Bytef*>(B->mf.p + bl.coff);
        zs.avail_in = bl.clen;
        zs.next_out = B->buf.data() + base + at[k];
        zs.avail_out = bl.isize;
        const int rc = inflate(&zs, Z_FINISH);
        if (rc != Z_STREAM_END || zs.avail_out != 0) { bad = 1; break; }
      }
      inflateEnd(&zs);
    });
    if (bad) return bam_fail(B, PS_ERR_FORMAT, "corrupt BGZF block (inflate failed)");
    B->next_block = b1;
  }
  return PS_OK;
}

static int bam_header(ps_bam* B, bool any_contig_order) {
  int st = bam_fill(B, 12);
  if (st) return st;
  auto avail = [&] { return B->buf.size() - B->head; };
  if (avail() < 12 || memcmp(B->buf.data() + B->head, "BAM\1", 4) != 0) return bam_fail(B, PS_ERR_FORMAT, "not a BAM file");
  const uint32_t l_text = rd32(B->buf.data() + B->head + 4);
  st = bam_fill(B, 12 + (size_t)l_text);
  if (st) return st;
  if (avail() < 12 + (size_t)l_text) return bam_fail(B, PS_ERR_FORMAT, "truncated BAM header");
  const std::string text((const char*)B->buf.data() + B->head + 8, l_text);
  // @HD ... SO:coordinate  (SAMFileHeader.getSortOrder; ErrorProfiling.java:124-132)
  {
    size_t hd = text.rfind("@HD", 0) == 0 ? 0 : text.find("\n@HD");
    if (hd != std::string::npos) {
      const size_t eol = text.find('\n', hd + 1);
      const std::string line = text.substr(hd, eol == std::string::npos ? std::string::npos : eol - hd);
      B->sorted = line.find("\tSO:coordinate") != std::string::npos;
    }
  }
  size_t o = B->head + 8 + l_text;
  const uint32_t n_ref = rd32(B->buf.data() + o);
  o += 4;
  for (uint32_t r = 0; r < n_ref; ++r) {
    st = bam_fill(B, o - B->head + 4);
    if (st) return st;
    if (B->buf.size() < o + 4) return bam_fail(B, PS_ERR_FORMAT, "truncated BAM header");
    const uint32_t l_name = rd32(B->buf.data() + o);
    st = bam_fill(B, o - B->head + 8 + (size_t)l_name);
    if (st) return st;
    if (B->buf.size() < o + 8 + (size_t)l_name) return bam_fail(B, PS_ERR_FORMAT, "truncated BAM header");
    std::string name((const char*)B->buf.data() + o + 4, l_name ? l_name - 1 : 0);
    B->ref_names.push_back(name);
    o += 8 + (size_t)l_name;
  }
  B->head = o;
  // contigs are matched by name (getSubsequenceAt(chr, ..), ErrorProfiling.java:169-172, PileupClusters.java:598-601):
  // the header may list them in any order; the records follow the header's order, which the pileup keys take over
  // (ps_bam_contig_order).  A caller that has not asked for that (PS_BAM_ANY_CONTIG_ORDER) keys the pileup in FASTA
  // order and is told at once that the file does not follow it.
  std::unordered_map<std::string, int64_t> idx;
  for (size_t c = 0; c < B->fa->names.size(); ++c) idx.emplace(B->fa->names[c], (int64_t)c);
  std::vector<char> listed(B->fa->names.size(), 0);
  int64_t last = -1;
  for (auto& nm : B->ref_names) {
    auto it = idx.find(nm);
    const int64_t c = it == idx.end() ? -1 : it->second;
    B->ref_to_contig.push_back(c);
    if (c >= 0 && !listed[(size_t)c]) {
      if (!any_contig_order && c < last)
        return bam_fail(B, PS_ERR_UNSUPPORTED, "the BAM header lists contigs in a different order than the FASTA index: "
                                               "open it with PS_BAM_ANY_CONTIG_ORDER and key the pileup in the header's "
                                               "order (ps_bam_contig_order, ps_reference_set_contig_order)");
      last = c;
      listed[(size_t)c] = 1;
      B->contig_order.push_back((uint32_t)c);
    }
  }
  B->header_done = true;
  return PS_OK;
}

extern "C" {

int ps_fasta_pack(const char* fasta_path, ps_packed_fasta** out) {
  if (!fasta_path || !out) return PS_ERR_INVALID_ARG;
  ps_packed_fasta* F = new ps_packed_fasta();
  *out = F;      // returned even on failure so the caller can read ps_fasta_error
  unsigned hc = std::thread::hardware_concurrency();
  return fasta_pack(fasta_path, F, hc ? (int)std::min(hc, 32u) : 4);
}
const ps_reference* ps_fasta_reference(const ps_packed_fasta* f) { return f ? &f->view : nullptr; }
const char* ps_fasta_contig_name(const ps_packed_fasta* f, uint32_t i) {
  return f && i < f->names.size() ? f->names[i].c_str() : nullptr;
}
const char* ps_fasta_error(const ps_packed_fasta* f) { return f ? f->err.c_str() : "no object"; }
void ps_fasta_free(ps_packed_fasta* f) { delete f; }

int ps_bam_open(ps_bam** out, const char* bam_path, const ps_packed_fasta* ref, uint64_t max_batch_reads, int threads) {
  return ps_bam_open_ex(out, bam_path, ref, max_batch_reads, threads, 0);
}

int ps_bam_open_ex(ps_bam** out, const char* bam_path, const ps_packed_fasta* ref, uint64_t max_batch_reads, int threads,
                   uint32_t flags) {
  if (!out || !bam_path || !ref) return PS_ERR_INVALID_ARG;
  ps_bam* B = new ps_bam();
  *out = B;      // returned even on failure so the caller can read ps_bam_error
  B->fa = ref;
  B->max_batch = max_batch_reads ? max_batch_reads : (1ull << 22);
  if (B->max_batch >= 0xFFFFFF00ull) B->max_batch = 0xFFFFFF00ull;
  if (threads <= 0) {
    unsigned hc = std::thread::hardware_concurrency();
    threads = hc ? (int)std::min(hc, 32u) : 4;
  }
  B->threads = threads;
  if (!B->mf.open(bam_path)) return bam_fail(B, PS_ERR_IO, std::string("cannot open ") + bam_path);
  int st;
  if (B->mf.n >= 2 && B->mf.p[0] == 0x1f && B->mf.p[1] == 0x8b) st = bam_scan_blocks(B);      // BGZF: a BAM
  else { B->sam_text = true; st = sam_header(B); }                                             // anything else: SAM text
  if (st) return st;
  st = bam_header(B, (flags & PS_BAM_ANY_CONTIG_ORDER) != 0);
  if (st) return st;
  // SamReader header check of both tools (ErrorProfiling.java:124-132, PileupClusters.java:85-92)
  if (!B->sorted) return bam_fail(B, PS_ERR_UNSORTED, ps_strerror(PS_ERR_UNSORTED));
  return PS_OK;
}

const char* ps_bam_error(const ps_bam* b) { return b ? b->err.c_str() : "no object"; }

int64_t ps_bam_contig_order(const ps_bam* b, uint32_t* order, uint64_t max) {
  if (!b || !b->header_done) return PS_ERR_INVALID_ARG;
  const uint64_t n = b->contig_order.size();
  if (!order) return (int64_t)n;
  if (n > max) return PS_ERR_INVALID_ARG;
  if (n) memcpy(order, b->contig_order.data(), n * 4);
  return (int64_t)n;
}

void ps_bam_close(ps_bam* b) {
  if (!b) return;
  if (getenv("PARASUITE_B200_BATCHER_TIMING"))
    fprintf(stderr, "[ps_bam] inflate %.3f s, locate %.3f s, sizes %.3f s, pack %.3f s, %llu records, %d threads\n", b->t_fill, b->t_locate,
            b->t_pass1, b->t_pass2, (unsigned long long)b->ordinal, b->threads);
  for (Slab& s : b->slab) s.release();
  delete b;
}

// Next batch of at most max_batch_reads records, in file order.  Returns 1 (batch filled; its arrays stay valid until
// the third-next call), 0 at end of file, or a negative status.
int ps_bam_next(ps_bam* B, ps_read_batch* out) {
  if (!B || !out) return PS_ERR_INVALID_ARG;
  if (!B->header_done) return bam_fail(B, PS_ERR_STATE, "BAM not open");
  // drop consumed bytes (offsets below are relative to the new start)
  if (B->head) {
    B->buf.drop_front(B->head);
    B->head = 0;
  }
  // ---- locate records -------------------------------------------------------------------------------------
  // A record's place is known only from the block_size of the one before it: a chain.  The bytes at hand are cut into
  // one span per thread; a thread whose span does not start the batch looks for the first offset from which a chain
  // of plausible records runs (the test a BAM split guesser makes: block_size against the lengths inside the record,
  // reference ids inside the header's range, a NUL-terminated printable name), all spans are walked at once, and the
  // result is accepted only where every span's walk lands exactly on the start the next span assumed -- from the first
  // span that does not, the chain is walked again the plain way.
  const double t_loc0 = now_s(), fill0 = B->t_fill;
  std::vector<uint64_t>& ro = B->rec_off;
  ro.clear();
  size_t o = 0;
  const int64_t n_ref = (int64_t)B->ref_names.size();
  auto plausible = [&](const uint8_t* d, size_t p, size_t end) -> int {     // 1 yes, 0 no, -1 cannot tell (runs past `end`)
    if (end - p < 36) return -1;
    const uint32_t bs = rd32(d + p);
    if (bs < 32 || bs > (1u << 26)) return 0;
    const int32_t ref_id = (int32_t)rd32(d + p + 4), pos = (int32_t)rd32(d + p + 8), nref = (int32_t)rd32(d + p + 24);
    const uint32_t l_name = d[p + 12], n_cig = rd16(d + p + 16), l_seq = rd32(d + p + 20);
    if (ref_id < -1 || ref_id >= n_ref || nref < -1 || nref >= n_ref || pos < -1 || l_name == 0) return 0;
    if (32ull + l_name + 4ull * n_cig + (l_seq + 1) / 2 + (uint64_t)l_seq > bs) return 0;
    if (end - p < 36 + (size_t)l_name) return -1;
    if (d[p + 36 + l_name - 1] != 0) return 0;
    for (uint32_t k = 0; k + 1 < l_name; ++k)
      if (d[p + 36 + k] < 0x21 || d[p + 36 + k] > 0x7e) return 0;
    return 1;
  };
  auto chain_start = [&](const uint8_t* d, size_t from, size_t end) -> size_t {   // first offset >= from that starts a chain
    const size_t stop = std::min(end, from + ((size_t)4 << 20));
    for (size_t p = from; p < stop; ++p) {
      size_t q = p;
      int k = 0, v = 1;
      for (; k < 12; ++k) {
        v = plausible(d, q, end);
        if (v != 1) break;
        q += 4 + (size_t)rd32(d + q);
        if (q > end) { v = -1; break; }
        if (q == end) break;
      }
      if (v == 1 || (v == -1 && k >= 3)) return p;
    }
    return (size_t)-1;
  };
  auto walk = [&](const uint8_t* d, size_t p, size_t until, size_t end, std::vector<uint64_t>& out, int* bad) -> size_t {
    // complete records starting before `until`; stops in front of the first one that is malformed or runs past `end`
    while (p < until && end - p >= 4) {
      const uint32_t bs = rd32(d + p);
      if (bs < 32) { *bad = 1; break; }
      if (end - p < 4 + (size_t)bs) break;
      out.push_back(p);
      p += 4 + (size_t)bs;
    }
    return p;
  };
  for (;;) {
    if (B->buf.size() - o < 4) {
      int st = bam_fill(B, o + 4);
      if (st) return st;
      if (B->buf.size() - o < 4) {
        if (B->buf.size() != o) return bam_fail(B, PS_ERR_FORMAT, "truncated BAM record");
        break;
      }
    }
    const uint8_t* d = B->buf.data();
    const size_t end = B->buf.size();
    const int T = (end - o > ((size_t)8 << 20) && B->threads > 1) ? B->threads : 1;
    int bad = 0;
    if (T == 1) {
      o = walk(d, o, end, end, ro, &bad);
    } else {
      std::vector<size_t> start(T + 1, (size_t)-1);
      std::vector<std::vector<uint64_t>> part(T);
      std::vector<size_t> stop_at(T, 0);
      std::vector<int> tbad(T, 0);
      start[0] = o;
      start[T] = end;
      parallel_for(T, (uint64_t)T - 1, [&](int, uint64_t lo, uint64_t hi) {
        for (uint64_t t = lo + 1; t < hi + 1; ++t) start[t] = chain_start(d, o + (end - o) / T * t, end);
      });
      for (int t = T - 1; t >= 1; --t)
        if (start[t] == (size_t)-1) start[t] = start[t + 1];          // no start found: the span before runs through
      parallel_for(T, (uint64_t)T, [&](int, uint64_t lo, uint64_t hi) {
        for (uint64_t t = lo; t < hi; ++t)
          if (start[t] < start[t + 1]) stop_at[t] = walk(d, start[t], start[t + 1], end, part[t], &tbad[t]);
          else stop_at[t] = start[t];
      });
      size_t p = o;
      int t = 0;
      for (; t < T; ++t) {
        if (t > 0 && stop_at[t - 1] != start[t]) break;      // the chain does not arrive where span t assumed its start
        ro.insert(ro.end(), part[t].begin(), part[t].end());
        p = stop_at[t];
        if (tbad[t]) { bad = 1; break; }
      }
      if (!bad && t < T && p < end) p = walk(d, p, end, end, ro, &bad);    // the plain way from where the spans disagree
      o = p;
    }
    if (bad) return bam_fail(B, PS_ERR_FORMAT, "malformed BAM record (block_size < 32)");
    if (ro.size() >= B->max_batch) {
      if (ro.size() > B->max_batch) { o = ro[B->max_batch]; ro.resize(B->max_batch); }
      break;
    }
    // the record at o is incomplete (or the bytes are used up): bring in more, or find the file's end
    size_t want = o + 4;
    if (B->buf.size() - o >= 4) want = o + 4 + (size_t)rd32(B->buf.data() + o);
    const size_t before = B->buf.size();
    int st = bam_fill(B, want);
    if (st) return st;
    if (B->buf.size() == before) {
      if (B->buf.size() != o) return bam_fail(B, PS_ERR_FORMAT, "truncated BAM record");
      break;
    }
  }
  B->head = o;
  B->t_locate += (now_s() - t_loc0) - (B->t_fill - fill0);
  const uint64_t n = ro.size();
  memset(out, 0, sizeof *out);
  if (n == 0) return 0;
  const uint8_t* buf = B->buf.data();
  const uint64_t n_tiles = (n + PS_TILE_READS - 1) / PS_TILE_READS;

  // ---- pass 1: sizes, per tile ----------------------------------------------------------------------------
  const double t_p1 = now_s();
  std::vector<uint64_t> tb(n_tiles + 1, 0), tq(n_tiles + 1, 0), tc(n_tiles + 1, 0);
  std::vector<uint32_t> te(n_tiles + 1, 0);
  std::atomic<int> bad{0};
  std::atomic<uint64_t> many_ops{~0ull};      // first record (index in this batch) with more than 255 CIGAR operations
  std::atomic<uint32_t> lens_min{0xFFFFFFFFu}, lens_max{0}, nc_min{0xFFFFFFFFu}, nc_max{0};
  auto amin = [](std::atomic<uint32_t>& a, uint32_t v) { uint32_t c = a.load(); while (v < c && !a.compare_exchange_weak(c, v)) {} };
  auto amax = [](std::atomic<uint32_t>& a, uint32_t v) { uint32_t c = a.load(); while (v > c && !a.compare_exchange_weak(c, v)) {} };
  parallel_for(B->threads, n_tiles, [&](int, uint64_t lo, uint64_t hi) {
    uint32_t lmin = 0xFFFFFFFFu, lmax = 0, cmin = 0xFFFFFFFFu, cmax = 0;
    for (uint64_t t = lo; t < hi; ++t) {
      uint64_t sb = 0, sq = 0, sc = 0;
      uint32_t se = 0;
      const uint64_t r1 = std::min(n, (t + 1) * PS_TILE_READS);
      for (uint64_t r = t * PS_TILE_READS; r < r1; ++r) {
        const uint8_t* p = buf + ro[r] + 4;
        const uint32_t bs = rd32(p - 4);
        const uint32_t l_name = p[8], n_cig = rd16(p + 12), l_seq = rd32(p + 16);
        if (32ull + l_name + 4ull * n_cig + (l_seq + 1) / 2 + l_seq > bs || l_seq > 0xFFFFu) { bad = 1; return; }
        const uint32_t nc = n_cig > 255 ? 0 : n_cig;
        if (n_cig > 255) { uint64_t c = many_ops.load(); while (r < c && !many_ops.compare_exchange_weak(c, r)) {} }
        sb += (l_seq + 3) / 4; sq += l_seq; sc += nc;
        const uint8_t* sq4 = p + 32 + l_name + 4ull * n_cig;
        for (uint32_t k = 0; k < l_seq; ++k) {
          const uint32_t nib = (sq4[k >> 1] >> ((~k & 1) * 4)) & 15u;
          se += !(nib == 1 || nib == 2 || nib == 4 || nib == 8);
        }
        lmin = std::min(lmin, l_seq); lmax = std::max(lmax, l_seq); cmin = std::min(cmin, nc); cmax = std::max(cmax, nc);
      }
      tb[t + 1] = sb; tq[t + 1] = sq; tc[t + 1] = sc; te[t + 1] = se;
    }
    amin(lens_min, lmin); amax(lens_max, lmax); amin(nc_min, cmin); amax(nc_max, cmax);
  });
  if (bad) return bam_fail(B, PS_ERR_FORMAT, "malformed BAM record (lengths exceed block_size, or read longer than 65535)");
  if (many_ops.load() != ~0ull) {
    // htsjdk takes any number of CIGAR elements (ErrorProfiling.java:206-207); the SoA holds 255 per record.  Fail
    // here, by name, instead of handing the kernels a record they can only refuse (PS_FAULT_CIGAR_OPS).
    char msg[160];
    snprintf(msg, sizeof msg, "record %llu has more than 255 CIGAR operations (not supported)",
             (unsigned long long)(B->ordinal + many_ops.load()));
    return bam_fail(B, PS_ERR_UNSUPPORTED, msg);
  }
  for (uint64_t t = 0; t < n_tiles; ++t) { tb[t + 1] += tb[t]; tq[t + 1] += tq[t]; tc[t + 1] += tc[t]; te[t + 1] += te[t]; }
  const uint64_t bases_bytes = tb[n_tiles], qual_bytes = tq[n_tiles], cigar_count = tc[n_tiles], exc_count = te[n_tiles];

  B->t_pass1 += now_s() - t_p1;
  // ---- slab layout ----------------------------------------------------------------------------------------------
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  size_t off_meta = 0, off_start = up(off_meta + n * 4), off_bases = up(off_start + n * 4);
  size_t off_qual = up(off_bases + bases_bytes + 64), off_cigar = up(off_qual + qual_bytes + 64);
  size_t off_exc = up(off_cigar + (cigar_count + 16) * 4), off_tb = up(off_exc + (exc_count + 16) * 4);
  size_t off_tq = up(off_tb + (n_tiles + 1) * 8), off_tc = up(off_tq + (n_tiles + 1) * 8), off_te = up(off_tc + (n_tiles + 1) * 8);
  const size_t total = up(off_te + (n_tiles + 1) * 4);
  Slab& S = B->slab[B->cur];
  B->cur = (B->cur + 1) % 3;
  if (!S.reserve(total)) return bam_fail(B, PS_ERR_OOM, "out of host memory for the batch");
  uint32_t* meta = (uint32_t*)(S.p + off_meta);
  uint32_t* ref_start = (uint32_t*)(S.p + off_start);
  uint8_t* bases2 = S.p + off_bases;
  uint8_t* qual = S.p + off_qual;
  uint32_t* cigar = (uint32_t*)(S.p + off_cigar);
  uint32_t* exc = (uint32_t*)(S.p + off_exc);
  memcpy(S.p + off_tb, tb.data(), (n_tiles + 1) * 8);
  memcpy(S.p + off_tq, tq.data(), (n_tiles + 1) * 8);
  memcpy(S.p + off_tc, tc.data(), (n_tiles + 1) * 8);
  memcpy(S.p + off_te, te.data(), (n_tiles + 1) * 4);
  memset(bases2 + bases_bytes, 0, 64);
  memset(qual + qual_bytes, 0, 64);
  memset(cigar + cigar_count, 0, 64);
  memset(exc + exc_count, 0, 64);

  // ---- pass 2: fill ---------------------------------------------------------------------------------------------
  const double t_p2 = now_s();
  static const int8_t kNib[16] = {-1, 0, 1, -1, 2, -1, -1, -1, 3, -1, -1, -1, -1, -1, -1, -1};   // "=ACMGRSVTWYHKDBN"
  const ps_packed_fasta* fa = B->fa;
  std::atomic<uint64_t> past_end{UINT64_MAX};           // ordinal of the first record counted in ps_read_batch.past_end
  parallel_for(B->threads, n_tiles, [&](int, uint64_t lo, uint64_t hi) {
    for (uint64_t t = lo; t < hi; ++t) {
      uint64_t ob = tb[t], oq = tq[t], oc = tc[t];
      uint32_t oe = te[t];
      const uint64_t r1 = std::min(n, (t + 1) * PS_TILE_READS);
      for (uint64_t r = t * PS_TILE_READS; r < r1; ++r) {
        const uint8_t* p = buf + ro[r] + 4;
        const int32_t refID = (int32_t)rd32(p), pos = (int32_t)rd32(p + 4);
        const uint32_t l_name = p[8], n_cig = rd16(p + 12), flag = rd16(p + 14), l_seq = rd32(p + 16);
        const uint8_t* cg = p + 32 + l_name;
        const uint8_t* sq4 = cg + 4ull * n_cig;
        const uint8_t* ql = sq4 + (l_seq + 1) / 2;
        uint32_t fl = 0;
        if (flag & 0x4) fl |= PS_RF_UNMAPPED;
        if (flag & 0x10) fl |= PS_RF_REVERSE;
        if (flag & 0x400) fl |= PS_RF_DUPLICATE;
        // getAlignmentStart() == 0 <=> stored pos == -1.  A stored pos < -1 is outside the BAM format (htsjdk would hand the
        // Java a negative start, which passes the == 0 filters and dies in the FASTA fetch); such records are folded into
        // the same class here instead of modelling a malformed file.
        if (pos < 0) fl |= PS_RF_POS_ZERO;
        if (l_seq == 0 || ql[0] == 0xFF) fl |= PS_RF_QUAL_MISSING;
        uint32_t nc = n_cig;
        if (n_cig > 255) { fl |= PS_RF_CIGAR_OVERFLOW; nc = 0; }
        uint64_t R = 0;
        for (uint32_t e = 0; e < nc; ++e) {
          const uint32_t c = rd32(cg + 4 * e), op = c & 15u;
          cigar[oc + e] = c;
          if ((0x18Du >> op) & 1u) R += c >> 4;                  // M, D, N, =, X consume the reference
        }
        // bases: 2-bit codes, 4 per byte; everything that is not A, C, G, T goes to the exception list as code 0
        for (uint32_t k = 0; k < (l_seq + 3) / 4; ++k) bases2[ob + k] = 0;
        bool any_inv = false;
        for (uint32_t k = 0; k < l_seq; ++k) {
          const int8_t cd = kNib[(sq4[k >> 1] >> ((~k & 1) * 4)) & 15u];
          if (cd < 0) { any_inv = true; exc[oe++] = ((uint32_t)(r % PS_TILE_READS) << 16) | k; }
          else bases2[ob + (k >> 2)] |= (uint8_t)(cd << (2 * (k & 3)));
        }
        if (any_inv) fl |= PS_RF_HAS_INVALID;
        memcpy(qual + oq, ql, l_seq);
        uint32_t g32 = 0;
        if (!(fl & (PS_RF_UNMAPPED | PS_RF_POS_ZERO))) {
          const int64_t c = (refID >= 0 && (size_t)refID < B->ref_to_contig.size()) ? B->ref_to_contig[refID] : -1;
          if (c < 0) fl |= PS_RF_REF_RANGE;                       // getSubsequenceAt on an unknown contig: SAMException
          else {
            const uint64_t clen = fa->off[c + 1] - fa->off[c];
            if ((uint64_t)pos + R > clen) fl |= PS_RF_REF_RANGE;  // stop > contig length: SAMException
            uint64_t g = fa->off[c] + (uint64_t)pos;
            if (R == 0 && (uint64_t)pos >= clen && !(fl & PS_RF_CIGAR_OVERFLOW)) {
              // no reference span and POS past the contig's end: its offset would name the next contig (the tools refuse
              // the first such record by its ordinal); the contig's last base keeps every later one on its own contig
              g = fa->off[c] + clen - 1;
              uint64_t cur = past_end.load();
              while (r < cur && !past_end.compare_exchange_weak(cur, r)) {}
            }
            g32 = g > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)g;
          }
        }
        ref_start[r] = g32;
        meta[r] = PS_MAKE_META(l_seq, nc, fl);
        ob += (l_seq + 3) / 4; oq += l_seq; oc += nc;
      }
    }
  });

  B->t_pass2 += now_s() - t_p2;
  out->n_reads = n;
  out->meta = meta;
  out->ref_start = ref_start;
  out->bases2 = bases2;
  out->qual = qual;
  out->cigar = cigar;
  out->tile_base_off = (const uint64_t*)(S.p + off_tb);
  out->tile_qual_off = (const uint64_t*)(S.p + off_tq);
  out->tile_cigar_off = (const uint64_t*)(S.p + off_tc);
  out->tile_exc_off = (const uint32_t*)(S.p + off_te);
  out->exc = exc;
  out->uniform_len = lens_min.load() == lens_max.load() ? lens_max.load() : 0;
  out->uniform_ncigar = nc_min.load() == nc_max.load() ? nc_max.load() : 0;
  out->bases_bytes = bases_bytes;
  out->qual_bytes = qual_bytes;
  out->cigar_count = cigar_count;
  out->exc_count = exc_count;
  out->max_len = lens_max.load();
  out->uniform_cigar = 0;
  out->flags8 = nullptr;
  out->qual6 = nullptr;
  out->start16 = nullptr;
  out->tile_start = nullptr;
  out->past_end = past_end.load() == UINT64_MAX ? 0 : past_end.load() + 1;
  B->ordinal += n;
  return 1;
}

// ---- whole-tool entry points -------------------------------------------------------------------------------------
int ps_reference_load_fasta(ps_ctx* ctx, const char* fasta_path) {
  if (!ctx || !fasta_path) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_packed_fasta* F = nullptr;
  int st = ps_fasta_pack(fasta_path, &F);
  if (st != PS_OK) {
    st = set_error(ctx, st, F ? F->err : "FASTA pack failed");
    ps_fasta_free(F);
    return st;
  }
  st = ps_reference_upload(ctx, &F->view);
  if (st != PS_OK) { ps_fasta_free(F); return st; }
  if (ctx->fasta && !ctx->fasta_shared) ps_fasta_free(ctx->fasta);
  ctx->fasta = F;      // contig names for the BAM header; the packed words stay on the host for later uploads
  ctx->fasta_shared = false;
  ctx->fasta_path = fasta_path;
  return PS_OK;
}

int open_for_ctx(ps_ctx* ctx, const char* bam_path, uint64_t max_batch, ps_bam** B) {
  if (!ctx->fasta) return set_error(ctx, PS_ERR_STATE, "ps_reference_load_fasta must come first (contig names are needed)");
  // the file tools follow the header's contig order (the pileup loop sets it on its contexts: tool_loops.cpp)
  int st = ps_bam_open_ex(B, bam_path, ctx->fasta, max_batch, 0, PS_BAM_ANY_CONTIG_ORDER);
  if (st != PS_OK) {
    st = set_error(ctx, st, *B ? (*B)->err : "cannot open BAM");
    ps_bam_close(*B);
    *B = nullptr;
  }
  return st;
}

// ErrorProfiling.inferErrorProfile up to the end of the record loop (:104-409), streaming in batches
int ps_profile_bam(ps_ctx* ctx, const char* bam_path, const ps_profile_opts* opts, ps_profile_result* out) {
  if (!ctx || !bam_path || !opts || !out) return set_error(ctx, PS_ERR_INVALID_ARG, "NULL argument");
  ps_bam* B = nullptr;
  uint64_t batch_reads = 1ull << 22;     // ~280 MB of SoA per batch at 36 nt; two slabs + two staging slots in flight
  if (const char* e = getenv("PARASUITE_B200_BATCH_READS")) { const long long v = atoll(e); if (v > 0) batch_reads = (uint64_t)v; }
  int st = open_for_ctx(ctx, bam_path, batch_reads, &B);
  if (st) return st;
  st = ps_profile_begin(ctx, opts);
  ps_read_batch hb;
  while (st == PS_OK) {
    // the slab ps_bam_next is about to fill was handed to the batch before last: wait for its copy (staging slots
    // and slabs alternate in lock-step)
    if (ctx->staged_done[ctx->staged_next]) cudaEventSynchronize(ctx->staged_done[ctx->staged_next]);
    const int k = ps_bam_next(B, &hb);
    if (k < 0) { st = set_error(ctx, k, B->err); break; }
    if (k == 0) break;
    st = ps_profile_batch(ctx, &hb);      // staged asynchronously; the slab stays valid until the second-next batch
  }
  if (st == PS_OK) st = ps_profile_end(ctx, out);
  else if (ctx->profile_open) { ps_profile_result dump; memset(&dump, 0, sizeof dump); ps_profile_end(ctx, &dump); }
  ps_bam_close(B);
  return st;
}

}  // extern "C"
