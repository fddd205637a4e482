// oracle/oracle_capi.cpp -- TEST INFRASTRUCTURE: C entry points (ctypes) into the CPU restatement, shaped like
// include/bmbs.h so that tests can compare the CUDA path record by record.  Never linked by the product.
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>
#include "oracle_core.hpp"
#include "oracle_pe.hpp"
#include "oracle_pe_sensitive.hpp"
#include "../include/bmbs.h"

using namespace oracle;

extern "C" {

void* orc_load(const char* prefix) { Index* ix = new Index(); if (!ix->load(prefix)) { delete ix; return nullptr; } return ix; }
void orc_free(void* h) { delete (Index*)h; }
uint64_t orc_genome_length(void* h) { return ((Index*)h)->N; }

int orc_bpm(const char* win, const char* read, int L, unsigned k, uint32_t* err) { return banded_bs_edit(win, read, L, k, *err); }
void orc_window(void* h, uint64_t site, uint64_t len, char* out) { ((Index*)h)->genome.window(site, len, out); }
uint64_t orc_lf(void* h, uint64_t row, int c) { return ((Index*)h)->lf(row, c); }
int orc_locate(void* h, uint64_t row, uint64_t* sa) { return ((Index*)h)->locate_row(row, *sa) ? 1 : 0; }
uint64_t orc_seed(void* h, const char* pat, uint64_t len, uint64_t* sp, uint64_t* ep, uint64_t* mlen) {
  SeedHit r = seed_until_unique(*(Index*)h, pat, len, *sp, *ep); *mlen = r.mlen; return r.hits;
}
uint64_t orc_count(void* h, const char* pat, uint64_t len, uint64_t* sp, uint64_t* ep) { return count_exact(*(Index*)h, pat, len, *sp, *ep); }

static void put(bmbs_cand& o, const Vote& v) {
  o.site = v.site; o.vote = (uint32_t)v.vote; o.end_site = (int16_t)(int64_t)v.end_site; o.err = v.err == 0xFFFFFFFFu ? 0xFFFF : (uint16_t)v.err;
}

// Same record layout and semantics as bmbs_map_batch_se.
int orc_map_se(void* h, const char* seqs, const uint64_t* offs, int n, double e_rate, int seed_len, bmbs_read_result* res, bmbs_cand* cand,
               size_t cap, size_t* used) {
  const Index& ix = *(Index*)h; Params P; P.e_rate = e_rate; P.seed_len = seed_len;
  size_t w = 0; std::vector<char> win;
  for (int r = 0; r < n; ++r) {
    const char* read = seqs + offs[r]; const int L = (int)(offs[r + 1] - offs[r]);
    const u64 k = u64_k(e_rate, L);
    SeedTrace t; std::string rd(read, L); seed_read(ix, P, rd.c_str(), L, t);
    bmbs_read_result& o = res[r]; memset(&o, 0, sizeof o);
    o.first_cand = (uint32_t)w; o.is_multiple_map = t.is_multi; o.one_mismatch_pos = (int16_t)t.one_mismatch_site;
    if (t.exact_unique) { o.state = BMBS_EXACT_UNIQUE; o.site = t.cand[0]; continue; }
    if (t.multi_exact_noC) { o.state = BMBS_MULTI_EXACT; continue; }
    if (t.cand.empty()) { o.state = BMBS_NONE; continue; }
    if (!t.extra && (t.cand.size() == 1 || (t.cand.size() == 2 && t.cand[0] == t.cand[1]))) { o.state = BMBS_ONE_MISMATCH; o.site = t.cand[0]; continue; }
    o.state = BMBS_VERIFY;
    std::vector<u64> c = t.cand; std::sort(c.begin(), c.end());
    std::vector<Vote> v; votes_from_sorted(c, k, v);
    o.n_cand = (uint32_t)v.size();
    for (auto& x : v) { verify_one(ix, rd.c_str(), L, k, x, win); if (w < cap) put(cand[w], x); ++w; }
  }
  *used = w;
  return w <= cap ? 0 : BMBS_ERR_CAPACITY;
}

// Same record layout and semantics as bmbs_map_batch_pe: lists after the pair distance filter, every
// unresolved entry verified.
int orc_map_pe(void* h, const char* seqs, const uint64_t* offs, int n_pairs, double e_rate, int seed_len, int min_ins, int max_ins,
               bmbs_read_result* res, bmbs_cand* cand, size_t cap, size_t* used) {
  const Index& ix = *(Index*)h; Params P; P.e_rate = e_rate; P.seed_len = seed_len; P.min_ins = min_ins; P.max_ins = max_ins;
  size_t w = 0; std::vector<char> win;
  for (int p = 0; p < n_pairs; ++p) {
    MateCands m[2]; std::string rd[2]; int L[2]; u64 k[2];
    for (int s = 0; s < 2; ++s) {
      const int r = 2 * p + s; L[s] = (int)(offs[r + 1] - offs[r]); rd[s].assign(seqs + offs[r], L[s]); k[s] = u64_k(e_rate, L[s]);
      mate_candidates(ix, P, rd[s].c_str(), L[s], k[s], m[s]);
    }
    const u64 kl = k[0] > k[1] ? k[0] : k[1];
    const int dmax = (int)((u64)max_ins + kl * 2), dmin = (int)((u64)min_ins - kl * 2 - (u64)(L[0] > L[1] ? L[0] : L[1]));
    const bool res0 = m[0].occ > 0, res1 = m[1].occ > 0;
    if (!(res0 && res1)) {
      if (m[0].v.empty() || m[1].v.empty()) { m[0].v.clear(); m[1].v.clear(); }
      else { filter_pairs(m[0].v, m[1].v, dmax, dmin); if (m[0].v.empty() || m[1].v.empty()) { m[0].v.clear(); m[1].v.clear(); } }
    }
    for (int s = 0; s < 2; ++s) {
      bmbs_read_result& o = res[2 * p + s]; memset(&o, 0, sizeof o);
      const SeedTrace& t = m[s].trace;
      o.first_cand = (uint32_t)w; o.is_multiple_map = t.is_multi; o.one_mismatch_pos = (int16_t)t.one_mismatch_site;
      if (t.exact_unique) { o.state = BMBS_EXACT_UNIQUE; o.site = t.cand[0]; }
      else if (t.multi_exact_noC) o.state = BMBS_MULTI_EXACT;
      else if (m[s].occ == 1) { o.state = BMBS_ONE_MISMATCH; o.site = t.cand[0]; }
      else if (m[s].occ == 0) o.state = BMBS_NONE;
      else o.state = BMBS_VERIFY;
      o.n_cand = (uint32_t)m[s].v.size();
      for (auto& x : m[s].v) { if (o.state == BMBS_VERIFY) verify_one(ix, rd[s].c_str(), L[s], k[s], x, win); if (w < cap) put(cand[w], x); ++w; }
    }
  }
  *used = w;
  return w <= cap ? 0 : BMBS_ERR_CAPACITY;
}

// Same record layout and semantics as bmbs_map_batch_pe with sensitive=1: every read's slice holds its FINAL hits
// (primary: verified hits; secondary: hits near a primary hit, after re-seeding when there were none).
int orc_map_pe_sensitive(void* h, const char* seqs, const uint64_t* offs, int n_pairs, double e_rate, int seed_len, int min_ins, int max_ins,
                         bmbs_read_result* res, bmbs_cand* cand, size_t cap, size_t* used, uint8_t* reseeded) {
  const Index& ix = *(Index*)h; Params P; P.e_rate = e_rate; P.seed_len = seed_len; P.min_ins = min_ins; P.max_ins = max_ins; P.sensitive = true;
  size_t w = 0;
  for (int p = 0; p < n_pairs; ++p) {
    std::string rd[2]; int L[2];
    for (int s = 0; s < 2; ++s) { const int r = 2 * p + s; L[s] = (int)(offs[r + 1] - offs[r]); rd[s].assign(seqs + offs[r], L[s]); }
    PairOutcome o; Stats st; SensDebug d;
    std::string q0(L[0], 'I'), q1(L[1], 'I');
    run_pe_sensitive_pair(ix, P, rd[0].c_str(), q0.c_str(), L[0], rd[1].c_str(), q1.c_str(), L[1], o, st, &d);
    const SensMate* m[2] = {&d.a, &d.b};
    const bool dead = m[d.primary]->occ == 0;
    for (int s = 0; s < 2; ++s) {
      bmbs_read_result& r = res[2 * p + s]; memset(&r, 0, sizeof r);
      const SeedTrace& t = m[s]->t;
      r.first_cand = (uint32_t)w; r.is_multiple_map = t.is_multi; r.one_mismatch_pos = (int16_t)t.one_mismatch_site;
      if (t.exact_unique) { r.state = BMBS_EXACT_UNIQUE; r.site = t.cand[0]; }
      else if (t.multi_exact_noC) r.state = BMBS_MULTI_EXACT;
      else if (t.cand.empty()) r.state = BMBS_NONE;
      else if (!t.extra && (t.cand.size() == 1 || (t.cand.size() == 2 && t.cand[0] == t.cand[1]))) { r.state = BMBS_ONE_MISMATCH; r.site = t.cand[0]; }
      else r.state = BMBS_VERIFY;
      const int occ = dead ? 0 : m[s]->occ;
      r.n_cand = (uint32_t)occ;
      if (reseeded) reseeded[2 * p + s] = m[s]->reseeded ? 1 : 0;
      for (int i = 0; i < occ; ++i) { if (w < cap) put(cand[w], m[s]->v[i]); ++w; }
    }
  }
  *used = w;
  return w <= cap ? 0 : BMBS_ERR_CAPACITY;
}

// CPU restatement of the device finishing (finish_se / finish_sorted, include/bmbs.h bmbs_final) the way the reference does it:
// std::sort by vote (Schema.cpp:27612, comparator :560-563), the walk of Map_candidate_votes_mutiple_* (:7847-8056 / :8325-8745,
// early exit of the is_multiple_map variant included), try_cigar_without_path (ksw.cpp:2515-2570) on the chosen window, and the
// coordinate conversion (Schema.cpp:12596-12650).  Never returns BMBS_FIN_HOST.
int orc_finish_se(void* h, const char* seqs, const uint64_t* offs, int n, double e_rate, int ambiguous_out, const bmbs_read_result* res,
                  const bmbs_cand* cand, bmbs_final* fin, uint16_t* mism, size_t mism_cap, size_t* mism_used) {
  const Index& ix = *(Index*)h;
  size_t w = 0; std::vector<char> win;
  struct Hit { u64 site, vote; uint32_t err; u64 end_site; };
  std::vector<Hit> hits;
  for (int r = 0; r < n; ++r) {
    const char* read = seqs + offs[r]; const int L = (int)(offs[r + 1] - offs[r]);
    const u64 k = u64_k(e_rate, L);
    bmbs_final& o = fin[r]; memset(&o, 0, sizeof o); o.sbd = 255; o.k = (uint8_t)k;
    const bmbs_read_result& rs = res[r];
    auto placed = [&](u64 site, int start, u64 end_site) {
      const bmbs::Placed p = bmbs::place(ix.chroms, site, (u64)(long long)start, end_site);
      if (p.off_chrom) { o.status = BMBS_FIN_UNMAPPED; return false; }
      o.status = BMBS_FIN_UNIQUE; o.chrom_pos = ((u64)p.chrom << 40) | p.pos; if (p.flag) o.flags |= BMBS_FINF_REVERSE;
      return true;
    };
    if (rs.state == BMBS_EXACT_UNIQUE) { o.site = rs.site; o.end_site = (int16_t)(L - 1); o.mapq_fixed = 42; placed(rs.site, 0, L - 1); continue; }
    if (rs.state == BMBS_ONE_MISMATCH) {
      o.site = rs.site; o.end_site = (int16_t)(L - 1); o.nm = 1;
      if (placed(rs.site, 0, L - 1)) { o.aux_first = (uint32_t)w; o.n_aux = 1; if (w < mism_cap) mism[w] = (uint16_t)rs.one_mismatch_pos; ++w; }
      continue;
    }
    if (rs.state == BMBS_MULTI_EXACT) {
      if (!ambiguous_out) { o.status = BMBS_FIN_AMBIGUOUS; continue; }
      for (uint32_t j = 0; j < rs.n_cand; ++j) {
        const u64 site = cand[rs.first_cand + j].site;
        if (!bmbs::place(ix.chroms, site, 0, L - 1).off_chrom) { o.site = site; o.end_site = (int16_t)(L - 1); o.mapq_fixed = 1; o.flags |= BMBS_FINF_AMBIGUOUS; placed(site, 0, L - 1); break; }
      }
      continue;
    }
    if (rs.state != BMBS_VERIFY) continue;
    hits.resize(rs.n_cand);
    for (uint32_t j = 0; j < rs.n_cand; ++j) { const bmbs_cand& c = cand[rs.first_cand + j]; hits[j] = {c.site, c.vote, c.err == 0xFFFF ? 0xFFFFFFFFu : c.err, (u64)(int64_t)c.end_site}; }
    std::sort(hits.begin(), hits.end(), [](const Hit& a, const Hit& b) { return a.vote > b.vote; });
    uint32_t min_err = 0xFFFFFFFEu, sbd = 0; long idx = -1; u64 best_end = ~0ull;
    for (size_t i = 0; i < hits.size(); ++i) {
      const uint32_t e = hits[i].err; const u64 end_abs = hits[i].site + hits[i].end_site;
      if (!rs.is_multiple_map) {
        if (e == min_err && best_end != end_abs && idx >= 0) { sbd = 0; idx = -2 - idx; }
        else if (e < min_err) { sbd = min_err - e; min_err = e; idx = (long)i; best_end = end_abs; }
      } else {
        if (e == min_err && best_end != end_abs) { sbd = 0; if (idx >= 0) idx = -2 - idx; if (min_err == 0) break; }
        else if (e < min_err) { sbd = min_err - e; min_err = e; idx = (long)i; best_end = end_abs; }
      }
    }
    const bool ambiguous = idx <= -2;
    if (ambiguous) { if (!ambiguous_out) { o.status = BMBS_FIN_AMBIGUOUS; continue; } idx = -2 - idx; o.flags |= BMBS_FINF_AMBIGUOUS; }
    if (idx < 0) continue;
    const Hit& b = hits[idx];
    o.site = b.site; o.end_site = (int16_t)(int64_t)b.end_site; o.nm = (uint8_t)b.err; o.sbd = (uint8_t)(sbd > 255 ? 255 : sbd);
    const int start = (int)(int64_t)b.end_site - L + 1;
    if (b.err != 0) {
      const int plen = L + 2 * (int)k; win.resize(plen + 8);
      ix.genome.window(b.site, plen, win.data());
      bool ok = start >= 0; size_t w0 = w; unsigned mis = 0;
      for (int i = 0; ok && i < L; ++i) {
        const char t = read[i], p = win[i + start];
        if (t != p && !(t == 'T' && p == 'C')) { if (++mis > b.err) { ok = false; break; } if (w < mism_cap) mism[w] = (uint16_t)i; ++w; }
      }
      if (!(ok && mis == b.err)) { w = w0; o.status = BMBS_FIN_DP; continue; }
      if (placed(b.site, start, b.end_site)) { o.aux_first = (uint32_t)w0; o.n_aux = mis; } else w = w0;
    } else placed(b.site, start, b.end_site);
  }
  *mism_used = w;
  return w <= mism_cap ? 0 : BMBS_ERR_CAPACITY;
}

// What the reference's pair workers do between their verification calls and the CIGAR / SAM code, on the records and verified
// hit lists of a paired batch (same layout as bmbs_batch_finish on a paired batch returns): in fast mode the hit compaction
// (Schema.cpp:7502-7608, as verify_keep_hits without the verification), filter_pairs_single_side (:16186-16288) on the longer
// list, the compaction of that list; in sensitive mode and for mates that seeding resolved the lists are final as they stand
// (Schema.cpp:22014-22130 / :23562-23690); then the pair pick new_faster_verify_pairs (:15773-15959), try_cigar_without_path
// (ksw.cpp:2515-2570) on the two chosen hits and their coordinates (Schema.cpp:9188-9244; the end-of-chromosome test comes later
// in the reference, with the final spans of both mates, :22310-22330, so a mate keeps its coordinates here).
int orc_finish_pe(void* h, const char* seqs, const uint64_t* offs, int n_pairs, double e_rate, int min_ins, int max_ins, int sensitive, int ambiguous_out,
                  const bmbs_read_result* res, const bmbs_cand* cand, bmbs_final* fin, uint16_t* mism, size_t mism_cap, size_t* mism_used) {
  const Index& ix = *(Index*)h;
  size_t w = 0; std::vector<char> win;
  auto resolved = [](const bmbs_read_result& r) { return r.state == BMBS_EXACT_UNIQUE || r.state == BMBS_MULTI_EXACT || r.state == BMBS_ONE_MISMATCH; };
  auto keep = [](std::vector<Vote>& v, u64 k) {      // Schema.cpp:7502-7512: hits within k whose absolute end differs from the entry before
    int kept = 0; u64 prev = (u64)-1;
    for (size_t i = 0; i < v.size(); ++i) {
      const u64 e = v[i].site + v[i].end_site;
      if (v[i].err <= k && prev != e) { v[kept].site = v[i].site; v[kept].err = v[i].err; v[kept].end_site = v[i].end_site; ++kept; }
      prev = e;
    }
    return kept;
  };
  for (int p = 0; p < n_pairs; ++p) {
    const int r1 = 2 * p, r2 = r1 + 1;
    const char* read[2] = {seqs + offs[r1], seqs + offs[r2]};
    const int L[2] = {(int)(offs[r1 + 1] - offs[r1]), (int)(offs[r2 + 1] - offs[r2])};
    const u64 k[2] = {u64_k(e_rate, L[0]), u64_k(e_rate, L[1])}, kl = k[0] > k[1] ? k[0] : k[1];
    bmbs_final* o[2] = {&fin[r1], &fin[r2]};
    for (int m = 0; m < 2; ++m) { memset(o[m], 0, sizeof(bmbs_final)); o[m]->sbd = 255; o[m]->k = (uint8_t)k[m]; }
    const bmbs_read_result& q1 = res[r1]; const bmbs_read_result& q2 = res[r2];
    if (q1.n_cand == 0 || q2.n_cand == 0) continue;
    const int dmax = (int)((u64)(long long)max_ins + kl * 2);
    const int dmin = (int)((u64)(long long)min_ins - kl * 2 - (u64)(L[0] > L[1] ? L[0] : L[1]));
    std::vector<Vote> v[2];
    for (int m = 0; m < 2; ++m) {
      const bmbs_read_result& q = m ? q2 : q1;
      v[m].resize(q.n_cand);
      for (uint32_t j = 0; j < q.n_cand; ++j) { const bmbs_cand& c = cand[q.first_cand + j]; v[m][j] = {c.site, c.vote, c.err == 0xFFFF ? 0xFFFFFFFFu : c.err, (u64)(int64_t)c.end_site}; }
    }
    int occ[2] = {(int)v[0].size(), (int)v[1].size()};
    const bool res1 = resolved(q1), res2 = resolved(q2);
    if (!(sensitive || (res1 && res2))) {
      if (!res1 && !res2) {
        const int a = v[0].size() <= v[1].size() ? 0 : 1, b = 1 - a;      // the shorter list is compacted first, the other filtered by it
        occ[a] = keep(v[a], k[a]);
        if (occ[a] == 0) continue;
        filter_single_side(v[a], occ[a], v[b], dmax, dmin);
        occ[b] = keep(v[b], k[b]);
      } else if (res1) occ[1] = keep(v[1], k[1]);
      else occ[0] = keep(v[0], k[0]);
    }
    const PairPick pk = pick_pair(v[0], occ[0], v[1], occ[1], (int)kl, dmax, dmin);
    if (pk.n > 1 && !ambiguous_out) { o[0]->status = BMBS_FIN_AMBIGUOUS; continue; }
    if (pk.n < 1) continue;
    const long long pick[2] = {pk.i1, pk.i2};
    for (int m = 0; m < 2; ++m) {
      const Vote& b = v[m][pick[m]];
      bmbs_final& f = *o[m];
      f.sbd = (uint8_t)(pk.second_best_diff > 255 ? 255 : pk.second_best_diff);
      if (pk.n > 1) f.flags |= BMBS_FINF_AMBIGUOUS;
      f.site = b.site; f.end_site = (int16_t)(int64_t)b.end_site; f.nm = (uint8_t)b.err;
      const int start = (int)(int64_t)b.end_site - L[m] + 1;
      size_t w0 = w; unsigned mis = 0;
      if (b.err != 0) {
        const int plen = L[m] + 2 * (int)k[m]; win.resize(plen + 8);
        ix.genome.window(b.site, plen, win.data());
        bool ok = start >= 0;
        for (int i = 0; ok && i < L[m]; ++i) {
          const char t = read[m][i], g = win[i + start];
          if (t != g && !(t == 'T' && g == 'C')) { if (++mis > b.err) { ok = false; break; } if (w < mism_cap) mism[w] = (uint16_t)i; ++w; }
        }
        if (!(ok && mis == b.err)) { w = w0; f.status = BMBS_FIN_DP; continue; }
      }
      const bmbs::Placed pl = bmbs::place(ix.chroms, b.site, (u64)(long long)start, b.end_site);
      f.status = BMBS_FIN_UNIQUE; f.chrom_pos = ((u64)pl.chrom << 40) | pl.pos; if (pl.flag) f.flags |= BMBS_FINF_REVERSE;
      if (mis) { f.aux_first = (uint32_t)w0; f.n_aux = mis; }
    }
  }
  *mism_used = w;
  return w <= mism_cap ? 0 : BMBS_ERR_CAPACITY;
}

// The order std::sort leaves the reference's 32-byte vote records in (Schema.cpp:27612, comparator :560-563): order[] receives
// the original positions.  What the device's sort replay (bmbs_debug_sort_order) is compared with.
void orc_std_sort_order(const uint32_t* votes, uint32_t n, uint32_t* order) {
  struct Rec { u64 site, vote; uint32_t err; u64 end_site; };
  std::vector<Rec> v(n);
  for (uint32_t i = 0; i < n; ++i) v[i] = {i, votes[i], 0, 0};
  std::sort(v.begin(), v.end(), [](const Rec& a, const Rec& b) { return a.vote > b.vote; });
  for (uint32_t i = 0; i < n; ++i) order[i] = (uint32_t)v[i].site;
}

int orc_verify(void* h, const char* seqs, const uint64_t* offs, int n_reads, const uint32_t* read_idx, const uint64_t* sites, size_t n,
               double e_rate, int32_t* end_site, uint32_t* err, int threads) {
  const Index& ix = *(Index*)h;
  if (threads < 1) threads = 1;
  auto work = [&](int t) {
    std::vector<char> win;
    for (size_t i = t; i < n; i += threads) {
      const uint32_t r = read_idx[i]; const int L = (int)(offs[r + 1] - offs[r]); const u64 k = u64_k(e_rate, L);
      std::string rd(seqs + offs[r], L);
      Vote v{sites[i], 0, 0, 0}; verify_one(ix, rd.c_str(), L, k, v, win);
      end_site[i] = (int32_t)(int64_t)v.end_site; err[i] = v.err;
    }
  };
  std::vector<std::thread> th; for (int t = 1; t < threads; ++t) th.emplace_back(work, t);
  work(0); for (auto& x : th) x.join();
  (void)n_reads;
  return 0;
}

// CIGAR refinement of one alignment on the CPU (host/postprocess.hpp refine_alignment, the restatement of
// fast_recalculate_bs_Cigar, ksw.cpp:2578-3148); window given as decoded characters
int orc_refine(const char* win, int wlen, const char* read, int rlen, int k, int end_site, unsigned err, int forward, const char* qual,
               int reverse_quality, int mp_max, int mp_min, int n_pen, int gap_open, int gap_ext, int q_base,
               int* start_site, uint64_t* out_end, unsigned* out_err, int* score, char* cigar, int cigar_cap) {
  bmbs::Scoring sc; sc.mp_max = mp_max; sc.mp_min = mp_min; sc.n_pen = n_pen; sc.gap_open = gap_open; sc.gap_ext = gap_ext; sc.q_base = q_base;
  bmbs::Refined rf;
  bmbs::refine_alignment(win, wlen, read, rlen, k, end_site, err, forward != 0, qual, reverse_quality != 0, sc, rf);
  *start_site = rf.start_site; *out_end = rf.end_site; *out_err = rf.err; *score = rf.score;
  snprintf(cigar, (size_t)cigar_cap, "%s", rf.cigar.c_str());
  return 0;
}
// the banded DP alone (banded_affine_align = ksw_semi_global_quality_back, ksw.cpp:1850-2045) on the window at `site`:
// what the refine_warp kernels must reproduce value for value
int orc_banded_align(void* h, uint64_t site, const char* read, const char* qual, int rlen, int k, int mp_max, int mp_min, int n_pen, int gap_open,
                     int gap_ext, int q_base, int* score, int* qb, int* qe, uint32_t* ops, int ops_cap) {
  bmbs::Scoring sc; sc.mp_max = mp_max; sc.mp_min = mp_min; sc.n_pen = n_pen; sc.gap_open = gap_open; sc.gap_ext = gap_ext; sc.q_base = q_base;
  const int wlen = rlen + 2 * k;
  std::vector<char> win((size_t)wlen + 8);
  ((Index*)h)->genome.window(site, (uint64_t)wlen, win.data());
  std::vector<uint32_t> o;
  bmbs::banded_affine_align(win.data(), wlen, read, rlen, k, qual, sc, *score, *qb, *qe, o);
  if ((int)o.size() > ops_cap) return -1;
  for (size_t i = 0; i < o.size(); ++i) ops[i] = o[i];
  return (int)o.size();
}

// The whole refinement of an alignment with indels as the reference finishes it: the DP above, then the end fix-ups and the NM
// recount (refine_fix_ends of csrc/bmbs_refine_ends.h and host/postprocess.hpp recount_nm, pinned to fast_recalculate_bs_Cigar by tests/test_refine_vs_reference.py).
// What bmbs_refine returns is compared with this.  ops[] receives the final operations in read order.
int orc_refine_final(void* h, uint64_t site, const char* read, const char* qual, int rlen, int k, int mp_max, int mp_min, int n_pen, int gap_open,
                     int gap_ext, int q_base, int* score, int* qb, int* qe, unsigned* nm, uint32_t* ops, int ops_cap) {
  bmbs::Scoring sc; sc.mp_max = mp_max; sc.mp_min = mp_min; sc.n_pen = n_pen; sc.gap_open = gap_open; sc.gap_ext = gap_ext; sc.q_base = q_base;
  const int wlen = rlen + 2 * k;
  std::vector<char> win((size_t)wlen + 8);
  ((Index*)h)->genome.window(site, (uint64_t)wlen, win.data());
  std::vector<uint32_t> o;
  bmbs::banded_affine_align(win.data(), wlen, read, rlen, k, qual, sc, *score, *qb, *qe, o);
  int cb, ce;
  bmbs::refine_fix_ends(o.data(), (int)o.size(), *qb, *qe, cb, ce);
  *nm = bmbs::recount_nm(win.data(), read, o, cb, ce, *qb);
  if (ce - cb + 1 > ops_cap) return -1;
  for (int i = cb; i <= ce; ++i) ops[i - cb] = o[i];
  return ce - cb + 1;
}

}  // extern "C"
