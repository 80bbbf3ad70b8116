// TEST INFRASTRUCTURE ONLY -- parity unpinned.
//
// CPU restatement (C++17, no dependencies) of the two PARA-suite hot loops, fed the same SoA read
// batches and packed reference as the CUDA path (include/parasuite_b200.h):
//
//   error profile : /root/reference/src/src/utils/errorprofile/ErrorProfiling.java:146-409, :633-664
//   T>C pileup    : /root/reference/src/src/utils/pileupclusters/PileupClusters.java:137-500, :585-673,
//                   StrandOrientation.java:14-56
//
// "Parity unpinned": the reference ships no tests, golden vectors or expected outputs for this path and
// its jar cannot run here (no JVM).  This file is pinned instead against the hand-derived vectors of
// SURVEY.md 8(c) and against an independent pure-Python transliteration (oracle/py_oracle.py) that works
// on raw ASCII/FASTA bytes; see tests/test_oracle_*.py.
//
// Every read is first expanded back to what htsjdk would present (ASCII bases, reference window bytes),
// then the Java statements are followed one by one -- including the temp-array walk, the caught
// ArrayIndexOutOfBoundsException (skip) and the uncaught ones (reported as ps_fault, the JVM would die).
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <map>
#include <thread>
#include <vector>

#include "../include/parasuite_b200.h"

namespace {

const char kBase[4] = {'A', 'C', 'G', 'T'};

// ErrorProfiling.java:633-664 / PileupClusters.java:690-721
inline int array_pos(uint8_t b) {
  switch (b) {
    case 65: case 97: return 0;
    case 67: case 99: return 1;
    case 71: case 103: return 2;
    case 84: case 116: return 3;
  }
  return -1;
}

// htsjdk SequenceUtil.reverseComplement: in place; complement maps only ACGTacgt
inline uint8_t complement(uint8_t b) {
  switch (b) {
    case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
    case 'a': return 't'; case 'c': return 'g'; case 'g': return 'c'; case 't': return 'a';
  }
  return b;
}
inline void reverse_complement(std::vector<uint8_t>& a) {
  std::reverse(a.begin(), a.end());
  for (auto& b : a) b = complement(b);
}

struct ReadView {
  uint32_t flags, L, ncig;
  uint64_t ref_start;
  const uint32_t* cigar;
  const uint8_t* bases2;
  const uint8_t* qual;
  std::vector<uint32_t> invalid_pos;  // exceptions of this read
};

// walks the tile structure of a batch sequentially
struct BatchCursor {
  const ps_read_batch* b;
  uint64_t r = 0;
  uint64_t boff = 0, qoff = 0, coff = 0;
  uint32_t eidx = 0;
  explicit BatchCursor(const ps_read_batch* bb) : b(bb) {}
  void seek(uint64_t read) {
    // jump to the tile, then walk
    uint64_t t = read / PS_TILE_READS;
    r = t * PS_TILE_READS;
    enter_tile(t);
    while (r < read) advance();
  }
  void enter_tile(uint64_t t) {
    if (b->uniform_len) {
      boff = r * ((b->uniform_len + 3) / 4);
      qoff = r * (uint64_t)b->uniform_len;
    } else {
      boff = b->tile_base_off[t];
      qoff = b->tile_qual_off[t];
    }
    coff = b->uniform_ncigar ? r * (uint64_t)b->uniform_ncigar : b->tile_cigar_off[t];
    eidx = b->tile_exc_off ? b->tile_exc_off[t] : 0;
  }
  void get(ReadView& v) {
    uint32_t m = b->meta[r];
    v.flags = PS_META_FLAGS(m);
    v.L = PS_META_LEN(m);
    v.ncig = PS_META_NCIGAR(m);
    v.ref_start = b->ref_start[r];
    v.cigar = b->cigar + coff;
    v.bases2 = b->bases2 + boff;
    v.qual = b->qual + qoff;
    v.invalid_pos.clear();
    if ((v.flags & PS_RF_HAS_INVALID) && b->tile_exc_off) {
      uint64_t t = r / PS_TILE_READS;
      uint32_t rit = (uint32_t)(r % PS_TILE_READS);
      for (uint32_t e = b->tile_exc_off[t]; e < b->tile_exc_off[t + 1]; ++e)
        if ((b->exc[e] >> 16) == rit) v.invalid_pos.push_back(b->exc[e] & 0xFFFFu);
    }
  }
  void advance() {
    uint32_t m = b->meta[r];
    boff += (PS_META_LEN(m) + 3) / 4;
    qoff += PS_META_LEN(m);
    coff += PS_META_NCIGAR(m);
    ++r;
    if (r % PS_TILE_READS == 0 && r < b->n_reads) enter_tile(r / PS_TILE_READS);
  }
};

// what SAMRecord.getReadBases() would return
void read_ascii(const ReadView& v, std::vector<uint8_t>& out) {
  out.resize(v.L);
  for (uint32_t p = 0; p < v.L; ++p) out[p] = kBase[(v.bases2[p >> 2] >> (2 * (p & 3))) & 3];
  for (uint32_t p : v.invalid_pos)
    if (p < v.L) out[p] = 'N';
}

// what IndexedFastaSequenceFile.getSubsequenceAt would return (case folded; non-ACGT -> 'N')
void ref_ascii(const ps_reference* ref, uint64_t g0, uint64_t n, std::vector<uint8_t>& out, size_t at) {
  for (uint64_t k = 0; k < n; ++k) {
    uint64_t g = g0 + k;
    bool inv = (ref->inv[g >> 5] >> (g & 31)) & 1u;
    out[at + k] = inv ? 'N' : kBase[(ref->seq2[g >> 4] >> (2 * (g & 15))) & 3];
  }
}

inline uint32_t contig_of(const ps_reference* ref, uint64_t g) {
  const uint64_t* lo = ref->contig_off;
  const uint64_t* it = std::upper_bound(lo, lo + ref->n_contigs + 1, g);
  return (uint32_t)(it - lo) - 1;
}

inline uint32_t cigar_ref_len(const uint32_t* c, uint32_t n) {  // htsjdk Cigar.getReferenceLength
  uint32_t r = 0;
  for (uint32_t k = 0; k < n; ++k) {
    uint32_t op = c[k] & 15;
    if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) r += c[k] >> 4;
  }
  return r;
}

struct Fault {
  int32_t code = 0;
  uint64_t ordinal = ~0ull;
  void raise(int32_t c, uint64_t o) {
    if (o < ordinal) { ordinal = o; code = c; }
  }
};

struct ProfileAcc {
  uint32_t max_len;
  bool infer_q;
  std::vector<int64_t> v;
  int64_t* conv() { return v.data(); }
  int64_t* qsum() { return v.data() + 16 * (size_t)max_len; }
  int64_t* qcnt() { return qsum() + 16; }
  int64_t* ins() { return qcnt() + 16; }
  int64_t* del() { return ins() + max_len; }
  int64_t* ctr() { return del() + max_len; }
  int64_t* qhist() { return ctr() + PS_PC_COUNT; }
};

// One iteration of ErrorProfiling.java:146-409.  Returns false when the JVM would have died.
bool profile_one(ProfileAcc& A, const ps_reference* ref, const ReadView& v, uint64_t ordinal, Fault& fault,
                 std::vector<uint8_t>& readSequence, std::vector<uint8_t>& refSequenceForRead,
                 std::vector<uint8_t>& readTemp, std::vector<uint8_t>& refTemp) {
  int64_t* C = A.ctr();
  if (v.flags & PS_RF_UNMAPPED) { C[PS_PC_UNMAPPED]++; return true; }     // :155
  if (v.flags & PS_RF_DUPLICATE) { C[PS_PC_DUPLICATES]++; return true; }  // :159
  if (v.flags & PS_RF_POS_ZERO) { C[PS_PC_START_ZERO]++; return true; }   // :163
  read_ascii(v, readSequence);                                            // :168
  uint32_t R = cigar_ref_len(v.cigar, v.ncig);
  // :169-172 getSubsequenceAt(chr, start, end)
  bool range_bad = (v.flags & PS_RF_REF_RANGE) != 0;
  if (!range_bad) {
    if (v.ref_start >= ref->n_bases) range_bad = true;
    else {
      uint32_t c = contig_of(ref, v.ref_start);
      if (v.ref_start + R > ref->contig_off[c + 1]) range_bad = true;
    }
  }
  if (range_bad) { fault.raise(PS_THROW_REF_RANGE, ordinal); return false; }
  refSequenceForRead.resize(R);
  ref_ascii(ref, v.ref_start, R, refSequenceForRead, 0);
  C[PS_PC_NUM_READS_PROCESSED]++;                                         // :174
  if (R == 0) { fault.raise(PS_THROW_EMPTY_REF, ordinal); return false; } // :180 ref[0] on empty array
  bool skip = false;
  uint32_t L = v.L;
  uint32_t mappingLength = L > R ? L : R;                                 // :189-193
  bool walked = false;
  if (L != R) {                                                           // :194
    walked = true;
    refTemp.assign(mappingLength, 0);
    readTemp.assign(mappingLength, 0);
    int64_t passedRef = 0, passedRead = 0, passedMatches = 0;
    for (uint32_t e = 0; e < v.ncig; ++e) {                               // :206
      uint32_t op = v.cigar[e] & 15;
      int64_t n = v.cigar[e] >> 4;
      if (op == 0 || op == 8 || op == 7) {                                // M, X, EQ :214-246
        for (int64_t z = 0; z < n; ++z) {
          // two statements inside one try: the first can succeed before the second throws
          if (z + passedMatches >= mappingLength || z + passedRef >= R) { skip = true; continue; }
          refTemp[z + passedMatches] = refSequenceForRead[z + passedRef];
          if (z + passedRead >= L) { skip = true; continue; }
          readTemp[z + passedMatches] = readSequence[z + passedRead];
        }
        passedMatches += n; passedRef += n; passedRead += n;
      } else if (op == 3) {                                               // N :247-251 (read cursor too)
        passedRef += n; passedRead += n;
      } else if (op == 1) {                                               // I :252-270
        for (int64_t z = 0; z < n; ++z) {
          if (passedMatches + z >= mappingLength) { fault.raise(PS_THROW_INDEL_FILL, ordinal); return false; }
          refTemp[passedMatches + z] = 45;
        }
        passedMatches += n; passedRead += n;
        for (int64_t q = 1; q <= n; ++q) {
          if (passedMatches + q >= A.max_len) { fault.raise(PS_THROW_INDEL_POS, ordinal); return false; }
          A.ins()[passedMatches + q] += 1;
        }
        if (n > 1) C[PS_PC_LONGER_INDELS]++;
      } else if (op == 2) {                                               // D :272-294
        for (int64_t z = 0; z < n; ++z) {
          if (passedMatches + z >= mappingLength) { fault.raise(PS_THROW_INDEL_FILL, ordinal); return false; }
          readTemp[passedMatches + z] = 45;
        }
        passedMatches += n; passedRef += n;
        for (int64_t q = 1; q <= n; ++q) {
          if (passedMatches + q >= A.max_len) { fault.raise(PS_THROW_INDEL_POS, ordinal); return false; }
          A.del()[passedMatches + q] += 1;
        }
        if (n > 1) C[PS_PC_LONGER_INDELS]++;
      }
      // S, H, P: no branch
    }
    C[PS_PC_INDEL_READ]++;                                                // :296
  }
  std::vector<uint8_t>& rd = walked ? readTemp : readSequence;            // :297-298
  std::vector<uint8_t>& rf = walked ? refTemp : refSequenceForRead;
  uint32_t qual_len = (v.flags & PS_RF_QUAL_MISSING) ? 0 : L;             // :301
  if (skip) { C[PS_PC_SKIPPED_READS]++; return true; }                    // :303-306
  if (v.flags & PS_RF_REVERSE) {                                          // :311-316
    reverse_complement(rd);
    reverse_complement(rf);
  }
  // :320-348 dead filter (isFilter=false)
  bool has_indel = false;                                                 // getCigarString().contains("D"/"I")
  for (uint32_t e = 0; e < v.ncig; ++e) {
    uint32_t op = v.cigar[e] & 15;
    if (op == 1 || op == 2) has_indel = true;
  }
  for (uint32_t i = 0; i < rd.size(); ++i) {                              // :349
    int a = array_pos(rf[i]);
    int b = array_pos(rd[i]);
    if (a >= 0 && b >= 0) {                                               // :376
      if (i >= A.max_len) { fault.raise(PS_THROW_POS_MAXLEN, ordinal); return false; }
      A.conv()[i * 16 + a * 4 + b]++;
      if (!has_indel) {
        if (i >= qual_len) { fault.raise(PS_THROW_QUAL_RANGE, ordinal); return false; }
        A.qsum()[a * 4 + b] += (int8_t)v.qual[i];                         // byte[] is signed
        A.qcnt()[a * 4 + b]++;
      }
      C[PS_PC_TOTAL_BASES_CHECKED]++;
    }
    if (A.infer_q) {                                                      // :402-407
      if (i >= A.max_len) { fault.raise(PS_THROW_POS_MAXLEN, ordinal); return false; }
      if (i >= qual_len) { fault.raise(PS_THROW_QUAL_RANGE, ordinal); return false; }
      A.qhist()[(size_t)i * 256 + v.qual[i]]++;
    }
  }
  return true;
}

void profile_range(const ps_reference* ref, const ps_read_batch* b, uint64_t lo, uint64_t hi, uint64_t ordinal0,
                   ProfileAcc& A, Fault& fault) {
  BatchCursor cur(b);
  cur.seek(lo);
  ReadView v;
  std::vector<uint8_t> s1, s2, s3, s4;
  for (uint64_t r = lo; r < hi; ++r) {
    cur.get(v);
    if (!profile_one(A, ref, v, ordinal0 + r, fault, s1, s2, s3, s4)) return;  // JVM would be dead
    cur.advance();
  }
}

// calculateClusterInformation :585-613 up to the count loop: the read and reference bases of the alignment blocks
// (SAMUtils.getAlignmentBlocks), strand-oriented.  Returns 0, or the PS_THROW code of the JVM's death on this record.
int32_t cluster_read_bases(const ps_reference* ref, const ReadView& v, int64_t contig, int64_t start,
                           std::vector<uint8_t>& readBases, std::vector<uint8_t>& readSequence,
                           std::vector<uint8_t>& refSequenceForRead) {
  read_ascii(v, readBases);
  readSequence.clear();
  refSequenceForRead.clear();
  int64_t rd = 0;        // 0-based read cursor  (block.getReadStart()-1)
  int64_t rf = start;    // 1-based reference cursor
  for (uint32_t e = 0; e < v.ncig; ++e) {
    uint32_t op = v.cigar[e] & 15;
    int64_t n = v.cigar[e] >> 4;
    if (op == 5 || op == 6) continue;                  // H, P
    if (op == 4 || op == 1) rd += n;                   // S, I
    else if (op == 2 || op == 3) rf += n;              // D, N
    else if (op == 0 || op == 7 || op == 8) {          // M, =, X
      if (rd + n > (int64_t)v.L) return PS_THROW_BLOCK_RANGE;
      // FASTA fetch [rf, rf+n-1] on this contig
      bool bad = (v.flags & PS_RF_REF_RANGE) != 0;
      uint64_t g0 = 0;
      if (!bad) {
        g0 = ref->contig_off[contig] + (uint64_t)(rf - 1);
        if (g0 + n > ref->contig_off[contig + 1]) bad = true;
      }
      if (bad) return PS_THROW_REF_RANGE;
      readSequence.insert(readSequence.end(), readBases.begin() + rd, readBases.begin() + rd + n);
      size_t at = refSequenceForRead.size();
      refSequenceForRead.resize(at + n);
      ref_ascii(ref, g0, n, refSequenceForRead, at);
      rd += n; rf += n;
    }
  }
  if (v.flags & PS_RF_REVERSE) {                       // :606-613
    reverse_complement(readSequence);
    reverse_complement(refSequenceForRead);
  }
  return 0;
}

}  // namespace

extern "C" {

size_t or_profile_acc_len(uint32_t max_len, uint32_t infer_q) {
  return 16 * (size_t)max_len + 32 + 2 * (size_t)max_len + PS_PC_COUNT + (infer_q ? 256 * (size_t)max_len : 0);
}

// Adds the contributions of reads [first, first+count) of `b` to acc (int64, or_profile_acc_len long).
// threads > 1 splits the range into tile-aligned chunks with private accumulators (sums commute, Q12).
int or_profile_run(const ps_reference* ref, const ps_read_batch* b, uint32_t max_len, uint32_t infer_q,
                   uint64_t first, uint64_t count, uint64_t ordinal0, int threads, int64_t* acc, ps_fault* fault_out) {
  if (first + count > b->n_reads) return PS_ERR_INVALID_ARG;
  size_t n = or_profile_acc_len(max_len, infer_q);
  if (threads < 1) threads = 1;
  uint64_t tiles = (count + PS_TILE_READS - 1) / PS_TILE_READS;
  if ((uint64_t)threads > tiles) threads = (int)std::max<uint64_t>(1, tiles);
  std::vector<ProfileAcc> accs(threads);
  std::vector<Fault> faults(threads);
  std::vector<std::thread> pool;
  for (int t = 0; t < threads; ++t) {
    accs[t].max_len = max_len;
    accs[t].infer_q = infer_q != 0;
    accs[t].v.assign(n, 0);
    uint64_t tlo = tiles * t / threads, thi = tiles * (t + 1) / threads;
    uint64_t lo = first + tlo * PS_TILE_READS, hi = std::min(first + count, first + thi * PS_TILE_READS);
    if (first % PS_TILE_READS) {  // unaligned start: single chunk only
      if (t == 0) { lo = first; hi = first + count; } else { lo = hi = first; }
    }
    auto work = [&, t, lo, hi]() { profile_range(ref, b, lo, hi, ordinal0, accs[t], faults[t]); };
    if (threads == 1) work(); else pool.emplace_back(work);
  }
  for (auto& th : pool) th.join();
  Fault f;
  for (int t = 0; t < threads; ++t) {
    for (size_t k = 0; k < n; ++k) acc[k] += accs[t].v[k];
    if (faults[t].code) f.raise(faults[t].code, faults[t].ordinal);
  }
  if (fault_out) {
    fault_out->code = f.code;
    fault_out->read_ordinal = f.code ? f.ordinal : 0;
  }
  return f.code ? PS_ERR_REFERENCE_WOULD_THROW : PS_OK;
}

// ------------------------------------------------------------------------------------------------
// T>C pileup: PileupClusters.java:137-500 up to (not including) the flush-time SNP filter; emits the
// per-cluster state the flush reads (the device contract of include/parasuite_b200.h).
// ------------------------------------------------------------------------------------------------
struct or_pileup_result {
  std::vector<ps_cluster> clusters;
  std::vector<ps_site> sites;
  ps_cluster open_cluster;
  std::vector<ps_site> open_sites;
  // sharding emulation only (not reference behaviour): the records at the head of a shard that continue the
  // cluster the preceding shard left open, and baseCoveredMap of the two boundary clusters
  ps_cluster head_partial;
  std::vector<ps_site> head_sites;
  bool has_head = false;
  std::map<int32_t, uint32_t> open_cov, head_cov;
  ps_pileup_counters counters;
  ps_fault fault;
};

or_pileup_result* or_pileup_run(const ps_reference* ref, const ps_read_batch* b, const ps_pileup_opts* opts) {
  auto* R = new or_pileup_result();
  std::memset(&R->counters, 0, sizeof(R->counters));
  std::memset(&R->open_cluster, 0, sizeof(ps_cluster));
  R->fault.code = 0;
  R->fault.read_ordinal = 0;
  // Java locals (PileupClusters.java:118-133)
  int64_t tempClusterStart = 0, tempClusterEnd = 0;
  int64_t tempClusterChr = -1;  // "" : equals no contig
  uint32_t numReadsPerCluster = 0, numT2C = 0;
  uint32_t runningID = opts ? opts->first_running_id : 1;
  // opts->carry_*: sharding emulation for the CPU tests of the halo merge -- start as if the preceding shard had
  // left a cluster open with this (chr, end).  The whole-stream runs that pin parity never set it.
  bool in_head = opts && opts->carry_valid;
  if (in_head) {
    tempClusterChr = opts->carry_contig;
    tempClusterEnd = opts->carry_cluster_end;
  }
  int isReverse = 0;  // 0 false, 1 true, 2 null (StrandOrientation)
  bool tempIsReverse = false;
  uint64_t mask51 = 0;
  uint32_t minusAfterFirst = 0;
  uint64_t firstRead = 0;
  struct Site { uint32_t t2c = 0, cov = 0; uint64_t key = ~0ull; };
  std::map<int32_t, Site> mutationMap;           // key -> (t2c, first insertion)
  std::map<int32_t, uint32_t> baseCoveredMap;
  bool have = false;

  auto snapshot = [&](ps_cluster& c, std::vector<ps_site>& sites) {
    c.first_read = firstRead;
    c.running_id = runningID;
    c.contig = (uint32_t)tempClusterChr;
    c.start = (int32_t)tempClusterStart;
    c.end = (int32_t)tempClusterEnd;
    c.num_reads = numReadsPerCluster;
    c.num_t2c = numT2C;
    c.minus_after_first = minusAfterFirst;
    c.first_reverse = tempIsReverse;
    c.combined_strand = (uint8_t)isReverse;
    c.reserved = 0;
    c.mask51 = mask51;
    c.site_begin = sites.size();
    for (auto& kv : mutationMap) {
      ps_site s;
      s.pos = kv.first;
      s.t2c = kv.second.t2c;
      s.cov = baseCoveredMap[kv.first];
      s.reserved = 0;
      s.order_key = kv.second.key;
      sites.push_back(s);
    }
    c.site_end = sites.size();
  };

  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  std::vector<uint8_t> readBases, readSequence, refSequenceForRead;
  for (uint64_t ord = 0; ord < b->n_reads; ++ord, cur.advance()) {
    cur.get(v);
    R->counters.num_reads_processed++;                                    // :138
    if (v.flags & PS_RF_UNMAPPED) continue;                               // :146
    bool hasI = false, hasD = false, hasN = false;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      uint32_t op = v.cigar[e] & 15;
      hasI |= op == 1; hasD |= op == 2; hasN |= op == 3;
    }
    if ((hasI || hasD) && hasN) { R->counters.skipped_due_indel++; continue; }  // :152-157
    if (b->past_end && ord == b->past_end - 1) {                          // no contig to put it on: refused
      R->fault.code = PS_FAULT_PAST_END; R->fault.read_ordinal = ord; return R;
    }
    // getAlignmentStart / getAlignmentEnd / getReferenceName
    int64_t contig, start, end;
    uint32_t refLen = cigar_ref_len(v.cigar, v.ncig);
    if (v.flags & PS_RF_POS_ZERO) {
      // mapped flag but POS==0: getReferenceName() is "*" and any block fetch raises SAMException.
      // (Only a record without a single M/=/X block would survive in the JVM; treated as a fault too.)
      R->fault.code = PS_THROW_REF_RANGE; R->fault.read_ordinal = ord; return R;
    } else {
      contig = contig_of(ref, v.ref_start);
      start = (int64_t)(v.ref_start - ref->contig_off[contig]) + 1;
      end = start + refLen - 1;
    }
    bool newCluster = (tempClusterEnd - start) < 5 || contig != tempClusterChr;  // :175-176
    if (newCluster) {
      if (have) {  // close the previous one (flush itself is host-side, later)
        ps_cluster c;
        snapshot(c, R->sites);
        R->clusters.push_back(c);
      } else if (in_head && numReadsPerCluster) {
        snapshot(R->head_partial, R->head_sites);
        R->head_partial.running_id = 0;
        R->head_partial.minus_after_first = minusAfterFirst;
        R->head_cov = baseCoveredMap;
        R->has_head = true;
      }
      in_head = false;
      tempClusterStart = start; tempClusterEnd = end; tempClusterChr = contig;   // :346-357
      numReadsPerCluster = 1; numT2C = 0; isReverse = 0;
      mutationMap.clear(); baseCoveredMap.clear();
      runningID++;
      mask51 = 0; minusAfterFirst = 0; firstRead = ord; have = true;
    } else {
      if (in_head && numReadsPerCluster == 0) { tempClusterStart = start; firstRead = ord; tempIsReverse = (v.flags & PS_RF_REVERSE) != 0; }
      if (end > tempClusterEnd) tempClusterEnd = end;                     // :421,:480
      numReadsPerCluster++;                                               // :488
    }
    // calculateClusterInformation :585-673
    if (int32_t code = cluster_read_bases(ref, v, contig, start, readBases, readSequence, refSequenceForRead)) {
      R->fault.code = code; R->fault.read_ordinal = ord; return R;
    }
    bool neg = (v.flags & PS_RF_REVERSE) != 0;
    if (neg) isReverse = 1;                                               // :606-613
    for (size_t i = 0; i < readSequence.size(); ++i) {                    // :637
      int32_t checkPosition = (int32_t)(neg ? end - (int64_t)i : start + (int64_t)i);
      if (array_pos(refSequenceForRead[i]) == 3 && array_pos(readSequence[i]) == 1) {  // :651
        numT2C++;
        if (i >= 51) { R->fault.code = PS_THROW_MASK51; R->fault.read_ordinal = ord; return R; }
        mask51 |= 1ull << i;
        Site& s = mutationMap[checkPosition];
        if (s.t2c == 0) s.key = (ord << 6) | (uint64_t)i;
        s.t2c++;
      }
      baseCoveredMap[checkPosition]++;                                    // :662-667
    }
    if (newCluster) tempIsReverse = isReverse == 1;                       // :364
    else if (!in_head && isReverse != 2 && tempIsReverse != (isReverse == 1)) {       // :494-498
      R->counters.double_stranded++;
      isReverse = 2;
    }
    if (!newCluster && neg) minusAfterFirst++;
  }
  if (have) {
    snapshot(R->open_cluster, R->open_sites);
    R->open_cov = baseCoveredMap;
    R->counters.has_open_cluster = 1;
  } else if (in_head && numReadsPerCluster) {
    snapshot(R->head_partial, R->head_sites);
    R->head_partial.running_id = 0;
    R->head_partial.minus_after_first = minusAfterFirst;
    R->head_cov = baseCoveredMap;
    R->has_head = true;
  }
  R->counters.n_clusters = R->clusters.size();
  R->counters.n_sites = R->sites.size();
  return R;
}

// Per read, what the pileup loop's mutationMapInRead would hold (PileupClusters.java:637-661) without the 51-entry
// array: bit i = T>C at index i of the strand-oriented read, for i < 62 (the layout of the profile kernel's mask words,
// whose bits 62 and 63 are flags).  0 for a record the loop skips (unmapped, I/D with N) or would die on.
int or_read_t2c_masks(const ps_reference* ref, const ps_read_batch* b, uint64_t* out) {
  BatchCursor cur(b);
  if (b->n_reads) cur.enter_tile(0);
  ReadView v;
  std::vector<uint8_t> readBases, readSequence, refSequenceForRead;
  for (uint64_t r = 0; r < b->n_reads; ++r, cur.advance()) {
    cur.get(v);
    out[r] = 0;
    if (v.flags & (PS_RF_UNMAPPED | PS_RF_POS_ZERO)) continue;          // :146; POS 0 kills the JVM
    bool hasID = false, hasN = false;
    for (uint32_t e = 0; e < v.ncig; ++e) {
      uint32_t op = v.cigar[e] & 15;
      hasID |= op == 1 || op == 2; hasN |= op == 3;
    }
    if (hasID && hasN) continue;                                          // :152-157
    const int64_t contig = contig_of(ref, v.ref_start);
    const int64_t start = (int64_t)(v.ref_start - ref->contig_off[contig]) + 1;
    if (cluster_read_bases(ref, v, contig, start, readBases, readSequence, refSequenceForRead)) continue;
    for (size_t i = 0; i < readSequence.size() && i < 62; ++i)
      if (array_pos(refSequenceForRead[i]) == 3 && array_pos(readSequence[i]) == 1) out[r] |= 1ull << i;
  }
  return PS_OK;
}

int or_pileup_counters(const or_pileup_result* r, ps_pileup_counters* out) { *out = r->counters; return PS_OK; }
int or_pileup_fault(const or_pileup_result* r, ps_fault* out) { *out = r->fault; return PS_OK; }
int64_t or_pileup_copy(const or_pileup_result* r, ps_cluster* clusters, uint64_t max_clusters, ps_site* sites,
                       uint64_t max_sites) {
  if (r->clusters.size() > max_clusters || r->sites.size() > max_sites) return PS_ERR_INVALID_ARG;
  std::copy(r->clusters.begin(), r->clusters.end(), clusters);
  std::copy(r->sites.begin(), r->sites.end(), sites);
  return (int64_t)r->clusters.size();
}
int64_t or_pileup_open(const or_pileup_result* r, ps_cluster* c, ps_site* sites, uint64_t max_sites) {
  if (!r->counters.has_open_cluster) return 0;
  if (r->open_sites.size() > max_sites) return PS_ERR_INVALID_ARG;
  *c = r->open_cluster;
  std::copy(r->open_sites.begin(), r->open_sites.end(), sites);
  return 1 + (int64_t)r->open_sites.size();
}
int64_t or_pileup_head(const or_pileup_result* r, ps_cluster* c, ps_site* sites, uint64_t max_sites) {
  if (!r->has_head) return 0;
  if (r->head_sites.size() > max_sites) return PS_ERR_INVALID_ARG;
  *c = r->head_partial;
  std::copy(r->head_sites.begin(), r->head_sites.end(), sites);
  return 1 + (int64_t)r->head_sites.size();
}
// dense baseCoveredMap of a boundary cluster (which: 0 head partial, 1 open cluster)
int64_t or_pileup_boundary_cov(const or_pileup_result* r, int which, int32_t* first_pos, uint32_t* cov, uint64_t max) {
  const std::map<int32_t, uint32_t>& m = which ? r->open_cov : r->head_cov;
  if (m.empty()) { *first_pos = 0; return 0; }
  int32_t lo = m.begin()->first, hi = m.rbegin()->first;
  *first_pos = lo;
  uint64_t n = (uint64_t)(hi - lo + 1);
  if (!cov) return (int64_t)n;
  if (n > max) return PS_ERR_INVALID_ARG;
  std::fill(cov, cov + n, 0u);
  for (auto& kv : m) cov[kv.first - lo] = kv.second;
  return (int64_t)n;
}
void or_pileup_free(or_pileup_result* r) { delete r; }

}  // extern "C"
