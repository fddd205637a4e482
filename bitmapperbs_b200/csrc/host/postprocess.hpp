// Host-side post-processing that follows the GPU seed-and-verify path:
// reference-window decode, CIGAR refinement (banded affine-gap DP with
// quality-scaled mismatch penalties), MAPQ, chromosome lookup.  These are the
// "next" rows of SURVEY.md §8(f)-1 and stay on the host, as in the reference.
//
// Behaviour mirrors (results must be identical on identical inputs):
//   window decode           Schema.cpp:4998-5115 (get_actuall_genome / _rc_genome)
//   ungapped shortcut       ksw.cpp:2515-2570    (try_cigar_without_path)
//   CIGAR refinement        ksw.cpp:2578-3148    (fast_recalculate_bs_Cigar)
//   banded DP + traceback   ksw.cpp:1850-2045    (ksw_semi_global_quality_back)
//   mismatch penalty        ksw.h:148-162        (MismatchPenaltyByQuality)
//   MAPQ table              Schema.cpp:168-405   (MAP_Calculation)
//   coordinate conversion   Schema.cpp:12596-12650, :9188-9244
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "../../../include/bmbs.h"
#include "../bmbs_refine_ends.h"

namespace bmbs {

struct Scoring {
  int mp_max = 6, mp_min = 2, n_pen = 1, gap_open = 5, gap_ext = 3, q_base = 33;
};

struct ChromTable {
  std::vector<std::string> name;
  std::vector<uint64_t> len, start, end;
  uint64_t N = 0;
  // <prefix>.index : u64 nChrom; {u64 nameLen; name; u64 len}*; u64 N   (Index.cpp:134-159, :940-980)
  bool load(const std::string& path) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    uint64_t nc = 0, s = 0;
    bool ok = fread(&nc, 8, 1, f) == 1;
    for (uint64_t i = 0; ok && i < nc; ++i) {
      uint64_t l = 0, cl = 0;
      ok = fread(&l, 8, 1, f) == 1 && l < (1u << 20);
      std::string nm(l, '\0');
      ok = ok && (l == 0 || fread(&nm[0], 1, l, f) == l) && fread(&cl, 8, 1, f) == 1;
      name.push_back(nm); len.push_back(cl); start.push_back(s); end.push_back(s + cl - 1);
      s += cl;
    }
    ok = ok && fread(&N, 8, 1, f) == 1;
    fclose(f);
    return ok;
  }
  // linear scan like the reference; returns name.size() when nothing contains pos
  size_t find(uint64_t pos) const {
    size_t c = 0;
    for (; c < name.size(); ++c) if (pos >= start[c] && pos <= end[c]) break;
    return c;
  }
};

// 2-bit genome, four bases per byte, first base in the top bits, A0 C1 G2 T3.
struct Genome2bit {
  // <prefix>.index.bs.pac: u64 nBytes; u8[] -- mapped, not read (only the windows of refined alignments are ever touched)
  struct Bytes {
    const uint8_t* p = nullptr; size_t n = 0; void* map = nullptr; size_t map_size = 0;
    Bytes() = default; Bytes(const Bytes&) = delete; Bytes& operator=(const Bytes&) = delete;
    uint8_t operator[](size_t i) const { return p[i]; }
    size_t size() const { return n; }
    ~Bytes() { if (map) munmap(map, map_size); }
  } pac;
  uint64_t N = 0;
  bool load(const std::string& path, uint64_t n_bases) {
    const int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 8) { ::close(fd); return false; }
    void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    ::close(fd);
    if (m == MAP_FAILED) return false;
    uint64_t nb = 0; memcpy(&nb, m, 8);
    if (nb > (uint64_t)st.st_size - 8) { munmap(m, (size_t)st.st_size); return false; }
    pac.map = m; pac.map_size = (size_t)st.st_size; pac.p = (const uint8_t*)m + 8; pac.n = (size_t)nb;
    N = n_bases;
    return true;
  }
  inline char base(uint64_t i) const { return "ACGT"[(pac[i >> 2] >> (6 - 2 * (i & 3))) & 3]; }
  // Forward-strand window [start, start+len); all-zero bytes when it would leave
  // the genome (such windows can never match).  Arithmetic is modulo 2^64 exactly
  // like the reference's (Schema.cpp:4998-5050).
  void window_fwd(uint64_t start, uint64_t len, char* out) const {
    if (start >= N || start + len > N) { memset(out, 0, len); return; }
    uint64_t i = 0, pos = start;
    for (; i < len && (pos & 3); ++i, ++pos) out[i] = base(pos);                       // up to the next byte boundary
    const uint32_t* lut = fwd_lut();
    for (; i + 4 <= len; i += 4, pos += 4) memcpy(out + i, &lut[pac[pos >> 2]], 4);     // four bases per byte
    for (; i < len; ++i, ++pos) out[i] = base(pos);
  }
  // Reverse-complement window: out[i] = complement(G[N-1-rc_start-i]) (Schema.cpp:5061-5115).
  void window_rc(uint64_t rc_start, uint64_t len, char* out) const {
    uint64_t last = N - rc_start - 1;
    if (last < len - 1 || (last >> 2) >= pac.size()) { memset(out, 0, len); return; }
    uint64_t i = 0, pos = last;                                                         // walks down the genome
    for (; i < len && (pos & 3) != 3; ++i, --pos) out[i] = "TGCA"[(pac[pos >> 2] >> (6 - 2 * (pos & 3))) & 3];
    const uint32_t* lut = rc_lut();
    for (; i + 4 <= len; i += 4, pos -= 4) memcpy(out + i, &lut[pac[pos >> 2]], 4);     // a whole byte, last base first, complemented
    for (; i < len; ++i, --pos) out[i] = "TGCA"[(pac[pos >> 2] >> (6 - 2 * (pos & 3))) & 3];
  }
  // byte -> its four bases as characters (first base in the low byte of the word), and reversed + complemented
  static const uint32_t* fwd_lut() {
    static const struct T { uint32_t v[256]; T() { for (int b = 0; b < 256; ++b) { char c[4]; for (int t = 0; t < 4; ++t) c[t] = "ACGT"[(b >> (6 - 2 * t)) & 3]; memcpy(&v[b], c, 4); } } } t;
    return t.v;
  }
  static const uint32_t* rc_lut() {
    static const struct T { uint32_t v[256]; T() { for (int b = 0; b < 256; ++b) { char c[4]; for (int t = 0; t < 4; ++t) c[t] = "TGCA"[(b >> (2 * t)) & 3]; memcpy(&v[b], c, 4); } } } t;
    return t.v;
  }
  // Double-strand coordinate: [0,N) forward strand, [N,2N) reverse complement.
  void window(uint64_t site, uint64_t len, char* out) const {
    if (site < N) window_fwd(site, len, out); else window_rc(site - N, len, out);
  }
};

inline int mismatch_penalty(const Scoring& sc, int q) {
  double phred = q - sc.q_base;
  if (phred > 40) phred = 40;
  phred = phred / 40;
  int p = phred * (sc.mp_max - sc.mp_min);
  return p + sc.mp_min;
}

// Bowtie2-like MAPQ from (second-best edit-distance gap, alignment score).
inline int mapq_from(unsigned second_best_diff, unsigned k, int score, const Scoring& sc) {
  int worst = std::max(sc.gap_open + sc.gap_ext, sc.mp_max);
  int score_min = (int)((unsigned)(-worst) * k);
  int range = -score_min;
  int sdiff = score - score_min;
  if (sdiff < 0) { fprintf(stderr, "error best_score: %d, scoreMax: %d\n", score, score_min); sdiff = 0; }
  int ediff = (int)second_best_diff;
  if (second_best_diff > k) ediff = (int)(k + 1);
  double rank = (double)sdiff / (double)range;
  if ((unsigned)ediff > k) {
    static const double th[6] = {0.8, 0.7, 0.6, 0.5, 0.4, 0.3};
    static const int q[6] = {42, 40, 24, 23, 8, 3};
    for (int i = 0; i < 6; ++i) if (rank >= th[i]) return q[i];
    return 0;
  }
  double re = (double)ediff / (double)k;
  const bool perfect = score == 0;
  // rows: error-gap rank >= t ; columns: q(perfect score), then (rank threshold, q) pairs, then fallback
  struct Row { double t; int q0; double r1; int q1; double r2; int q2; int q3; };
  static const Row rows[9] = {
    {0.9, 39, -1, 33, -1, 33, 33}, {0.8, 38, -1, 27, -1, 27, 27}, {0.7, 37, -1, 26, -1, 26, 26},
    {0.6, 36, -1, 22, -1, 22, 22}, {0.5, 35, 0.84, 25, 0.68, 16, 5}, {0.4, 34, 0.84, 21, 0.68, 14, 4},
    {0.3, 32, 0.88, 18, 0.67, 15, 3}, {0.2, 31, 0.88, 17, 0.67, 11, 0}, {0.1, 30, 0.88, 12, 0.67, 7, 0}};
  for (const Row& r : rows) {
    if (re >= r.t) {
      if (perfect) return r.q0;
      if (r.r1 < 0 || rank >= r.r1) return r.q1;
      if (rank >= r.r2) return r.q2;
      return r.q3;
    }
  }
  if (ediff == 0) return rank >= 0.67 ? 1 : 0;
  return rank >= 0.67 ? 6 : 2;
}

struct Refined {
  int start_site = 0;        // first window position used by the alignment
  uint64_t end_site = 0;     // last window position used
  unsigned err = 0;          // NM
  int score = 0;
  std::string cigar;
};

namespace detail {
inline int nt4(char c) {
  switch (c) { case 'A': case 'a': return 0; case 'C': case 'c': return 1; case 'G': case 'g': return 2; case 'T': case 't': return 3; default: return 4; }
}
// substitution score of read base t against reference base q at a read position
// whose scaled quality is `phred` in [.,1]; read T on reference C is a match.
inline int sub_score(int t, int q, double phred, const Scoring& sc) {
  if (t == 4 || q == 4) return -sc.n_pen;
  if (t == q || (t == 3 && q == 1)) return 0;
  return -sc.mp_min - (int)((int8_t)(sc.mp_max - sc.mp_min) * phred);
}
}  // namespace detail

// Banded (2k+1) semi-global affine-gap alignment of the read against the
// window with traceback.  ops: (len<<4)|op with op 0=M, 1=D (reference only),
// 2=I (read only), in read order.
inline void banded_affine_align(const char* win, int wlen, const char* read, int rlen, int k,
                                const char* qual, const Scoring& sc,
                                int& score, int& qb, int& qe, std::vector<uint32_t>& ops) {
  const int NEG = -0x40000000;
  const int band = 2 * k + 1, goe = sc.gap_open + sc.gap_ext, ge = sc.gap_ext;
  std::vector<int32_t> H(wlen + 2, NEG), E(wlen + 2, NEG);
  std::vector<uint8_t> dir((size_t)band * rlen);
  for (int j = 0; j < band; ++j) { H[j] = 0; E[j] = -goe; }
  int beg = 0, end = 0;
  for (int i = 0; i < rlen; ++i) {
    int t = detail::nt4(read[i]);
    double phred = qual[i] - sc.q_base;
    if (phred > 40) phred = 40;
    phred = phred / 40;
    beg = i; end = i + band;
    int32_t f = NEG, left = NEG;
    uint8_t* d_row = &dir[(size_t)i * band];
    for (int j = beg; j < end; ++j) {
      int32_t m = H[j], e = E[j];
      H[j] = left;
      m += detail::sub_score(t, detail::nt4(win[j]), phred, sc);
      uint8_t d = m >= e ? 0 : 1;
      int32_t h = m >= e ? m : e;
      d = h >= f ? d : 2;
      h = h >= f ? h : f;
      left = h;
      int32_t open = m - goe;
      e -= ge;
      if (e > open) d |= 1 << 2; else e = open;
      E[j] = e;
      f -= ge;
      if (f > open) d |= 2 << 4; else f = open;
      d_row[j - beg] = d;
    }
    H[end] = left; E[end] = NEG;
  }
  int best = rlen + k;
  score = H[best];
  for (int j = end; j > beg; --j) if (H[j] > score) { score = H[j]; best = j; }
  qe = best - 1;
  ops.clear();
  auto push = [&](uint32_t op, uint32_t len) {
    if (ops.empty() || (ops.back() & 0xf) != op) ops.push_back(len << 4 | op); else ops.back() += len << 4;
  };
  int i = rlen - 1, j = best - 1, state = 0;
  while (i >= 0 && j >= 0) {
    state = dir[(size_t)i * band + (j - i)] >> (state << 1) & 3;
    if (state == 0) { push(0, 1); --i; --j; }
    else if (state == 1) { push(2, 1); --i; }
    else { push(1, 1); --j; }
  }
  if (i >= 0) push(2, i + 1);
  std::reverse(ops.begin(), ops.end());
  qb = j + 1;
}

// Where the banded DP of refine_alignment runs.  The mapper sends a whole sub-block's DPs to the GPU in one bmbs_refine
// call: a first pass over the sub-block COLLECTs the requests (the unit that asked is marked pending and re-done later),
// a second pass REPLAYs the results in the same order.  Without a queue the DP runs here on the CPU (oracle, tests).
struct DpQueue {
  enum Mode { COLLECT = 1, REPLAY = 2 };
  int mode = COLLECT;
  bool pending = false;                                 // COLLECT: the current unit asked for a DP
  std::string seqs, quals; std::vector<bmbs_refine_item> items; size_t ops_bound = 0;
  std::vector<bmbs_refine_result> res; std::vector<uint32_t> ops; size_t next = 0;   // REPLAY
  // REPLAY from results that live elsewhere (the mapper refines a whole launch's alignments in one call and every sub-block
  // replays its own range); reads handed back to the host reduction then run their DP on the CPU
  const bmbs_refine_result* xres = nullptr; const uint32_t* xops = nullptr; bool external = false;
  void clear() { mode = COLLECT; pending = false; seqs.clear(); quals.clear(); items.clear(); ops_bound = 0; res.clear(); ops.clear(); next = 0; xres = nullptr; xops = nullptr; external = false; }
  void replay_from(const bmbs_refine_result* r, const uint32_t* o, size_t first) { mode = REPLAY; external = true; xres = r; xops = o; next = first; }
  // COLLECT: one alignment for the device (read as aligned, qualities in the DP's order)
  void request(uint64_t site, const char* read, const char* qual, int rlen, int k) {
    bmbs_refine_item it; it.site = site; it.seq_off = (uint32_t)seqs.size(); it.len = (uint16_t)rlen; it.k = (uint8_t)k; it.pad = 0;
    seqs.append(read, (size_t)rlen); quals.append(qual, (size_t)rlen); items.push_back(it);
    ops_bound += 2 * (size_t)rlen + 2 * (size_t)k + 2;
    pending = true;
  }
  // REPLAY: the next result as the reference's (start, end, NM, score, CIGAR); a reverse-strand hit prints its operations last to first
  template <class R> void take(bool forward, R& out) {
    const bmbs_refine_result& r = external ? xres[next++] : res[next++];
    const uint32_t* ops = external ? xops : this->ops.data();
    out.score = r.score; out.start_site = r.qb; out.end_site = (uint64_t)(int64_t)r.qe; out.err = r.nm;
    out.cigar.clear();
    char buf[16];
    for (uint32_t x = 0; x < r.n_ops; ++x) {
      const uint32_t o = ops[r.ops_off + (forward ? x : r.n_ops - 1 - x)];
      uint32_t len = o >> 4; int p = 16; buf[--p] = "MDISH"[o & 0xf];
      do { buf[--p] = (char)('0' + len % 10); len /= 10; } while (len);
      out.cigar.append(buf + p, (size_t)(16 - p));
    }
  }
};

// NM over the final operations (ksw.cpp:2990-3143): mismatches of the match runs (read T on window C is none) + gap lengths
inline unsigned recount_nm(const char* win, const char* read, const std::vector<uint32_t>& ops, int cb, int ce, int qb) {
  unsigned nm = 0; int wi = qb, ri = 0;
  for (int i = cb; i <= ce; ++i) {
    const uint32_t op = ops[i] & 0xf, len = ops[i] >> 4;
    if (op == 0) { for (uint32_t x = 0; x < len; ++x, ++wi, ++ri) nm += win[wi] != read[ri] && !(win[wi] == 'C' && read[ri] == 'T'); }
    else if (op == 1) { wi += len; nm += len; }
    else { ri += len; nm += len; }
  }
  return nm;
}

// CIGAR / NM / score / start / end of the best hit, given the verifier's
// (end_site, err).  `qual` is the quality string in FASTQ order; mate 2 of a
// pair is aligned as its reverse complement, so its qualities are reversed
// (reverse_quality) for the DP and restored.
inline void refine_alignment(const char* win, int wlen, const char* read, int rlen, int k,
                             int end_site, unsigned err, bool forward, const char* qual_in,
                             bool reverse_quality, const Scoring& sc, Refined& out, uint64_t site = 0, DpQueue* dq = nullptr) {
  out.cigar.clear();
  if (err == 0) {
    out.score = 0; out.start_site = end_site - rlen + 1; out.end_site = end_site; out.err = 0;
    out.cigar = std::to_string(rlen) + "M";
    return;
  }
  std::string qual(qual_in, rlen);
  if (reverse_quality) std::reverse(qual.begin(), qual.end());
  {  // ungapped attempt: exactly `err` mismatches on the diagonal ending at end_site
    int start = end_site - rlen + 1, mism = 0, score = 0;
    bool ok = start >= 0;
    for (int i = 0; ok && i < rlen; ++i) {
      char t = read[i], p = win[i + start];
      if (t != p && !(t == 'T' && p == 'C')) {
        if (++mism > (int)err) { ok = false; break; }
        if (t == 'N' || p == 'N') score -= sc.n_pen; else score -= mismatch_penalty(sc, qual[i]);
      }
    }
    if (ok && mism == (int)err) {
      out.score = score; out.start_site = start; out.end_site = end_site; out.err = err;
      out.cigar = std::to_string(rlen) + "M";
      return;
    }
  }
  int score, qb, qe; std::vector<uint32_t> ops;
  if (!dq) banded_affine_align(win, wlen, read, rlen, k, qual.data(), sc, score, qb, qe, ops);
  else if (dq->mode == DpQueue::COLLECT) { dq->request(site, read, qual.data(), rlen, k); out.score = 0; out.start_site = end_site - rlen + 1; out.end_site = end_site; out.err = err; out.cigar = "*"; return; }   // placeholder, the unit is redone
  else { dq->take(forward, out); return; }       // the device returns the final operations: fix-ups and NM recount included
  int cb, ce;
  refine_fix_ends(ops.data(), (int)ops.size(), qb, qe, cb, ce);
  const unsigned nm = recount_nm(win, read, ops, cb, ce, qb);
  char buf[32];
  for (int x = cb; x <= ce; ++x) {
    const uint32_t o = ops[forward ? x : ce - (x - cb)];
    snprintf(buf, sizeof buf, "%u%c", o >> 4, "MDISH"[o & 0xf]); out.cigar += buf;
  }
  out.score = score; out.start_site = qb; out.end_site = qe; out.err = nm;
}

// Double-strand window coordinates -> (flag 0/16, chromosome, 1-based POS).
struct Placed { int flag; size_t chrom; uint64_t pos; bool off_chrom; };
inline Placed place(const ChromTable& ct, uint64_t site, uint64_t start_site, uint64_t end_site) {
  Placed p;
  uint64_t loc = site;
  if (loc >= ct.N) { loc = ct.N * 2 - (loc + end_site) - 1; p.flag = 16; }
  else { loc = loc + start_site; p.flag = 0; }
  p.chrom = ct.find(loc);
  size_t c = p.chrom < ct.name.size() ? p.chrom : ct.name.size() - 1;  // reference reads past the table here
  p.chrom = c;
  p.pos = loc + 1 - ct.start[c];
  p.off_chrom = p.pos + end_site - start_site > ct.len[c];
  return p;
}

}  // namespace bmbs
