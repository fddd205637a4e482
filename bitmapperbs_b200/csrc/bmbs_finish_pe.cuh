// Paired-end finishing on the device (SURVEY 8a V4 / V5, 8f-1): what Map_Pair_Seq_split_fast / Map_Pair_Seq_split do after their
// verification calls, for every pair of a paired batch -- included by bmbs_kernels.cuh.
//   * hit compaction (map_candidate_votes_mutiple_cut_end_to_end_*_for_paired_end, Schema.cpp:7502-7608): hits within k whose
//     absolute end differs from the entry before them, in site order;
//   * filter_pairs_single_side (:16186-16288): the longer list keeps the windows within [dmin, dmax] of a hit of the shorter one;
//   * new_faster_verify_pairs (:15773-15959): the pair with the smallest err sum, how many pairs share it, second_best_diff as
//     the running best stood before the winner (first winner kept);
//   * per chosen mate: try_cigar_without_path (ksw.cpp:2515-2570) and the coordinates, as finish_hit does for single-end reads.
// One thread per pair walks the lists literally, in the reference's order (the walks carry `first`, a skip pointer whose
// value depends on every earlier step; lists are a handful of entries outside repeats).  Two bmbs_final records per pair come
// back (mates 2p, 2p+1) instead of both mates' window lists:
//   mate 1's record carries the pair's outcome: status BMBS_FIN_UNMAPPED (no pair: both records blank), BMBS_FIN_AMBIGUOUS
//   (several equally good pairs, not reported), else both mates are BMBS_FIN_UNIQUE (ungapped: chrom_pos, strand, nm, mismatch
//   positions) or BMBS_FIN_DP (site, end_site, nm = the verifier's err); sbd = second_best_diff of the pair (both records),
//   BMBS_FINF_AMBIGUOUS = reported although several pairs tie (--ambiguous_out).  A mate that runs over the end of its
//   chromosome keeps its coordinates: the pair is dropped by the caller's span check (Schema.cpp:22310-22330), as in the reference.
#pragma once

namespace pe_fin {
// b keeps the entries within range of one of a[0..na), each at most once, in order; returns how many
__device__ __forceinline__ int single_side(const bmbs_cand* a, int na, bmbs_cand* b, int nb, int dmax, int dmin) {
  long long first = 0; int kept = 0;
  for (long long i = 0; i < na; ++i) {
    const u64 as = a[i].site;
    for (long long j = first; j < nb; ++j) {
      bool stop; const bool in = in_range(as, b[j].site, dmax, dmin, j, first, stop);
      if (stop) break;
      if (in) { b[kept++] = b[j]; first = j + 1; }
    }
  }
  return na > 0 ? kept : 0;
}
}  // namespace pe_fin

// ---- the pair logic in three steps, on the two hit lists v1 / v2 (global memory, or a warp's copy in shared memory)
struct PePick { int n_best; long long i1, i2; u32 sbd; };

// hit compaction and single-side filter, in place; false: one side is left without a hit
__device__ __forceinline__ bool pe_compact(const BatchView& b, int r1, int r2, const bmbs_read_result& q1, const bmbs_read_result& q2,
                                           bmbs_cand* v1, bmbs_cand* v2, int dmax, int dmin, int& occ1, int& occ2) {
  const u32 k1 = b.kk[r1], k2 = b.kk[r2];
  const bool res1 = is_resolved(q1.state), res2 = is_resolved(q2.state);
  occ1 = (int)q1.n_cand; occ2 = (int)q2.n_cand;
  auto keep_hits = [](bmbs_cand* v, int n, u32 k) { return (int)keep_hits_inplace(v, (u32)n, k, nullptr, 0, 0, 0); };
  // --pe --sensitive: sens_pair / sens_reseed_finish already left each mate's final hits
  if (b.sensitive || (res1 && res2)) return true;
  if (!res1 && !res2) {
    if (q1.n_cand <= q2.n_cand) {
      occ1 = keep_hits(v1, occ1, k1);
      if (occ1 == 0) return false;
      occ2 = pe_fin::single_side(v1, occ1, v2, occ2, dmax, dmin); occ2 = keep_hits(v2, occ2, k2);
    } else {
      occ2 = keep_hits(v2, occ2, k2);
      if (occ2 == 0) return false;
      occ1 = pe_fin::single_side(v2, occ2, v1, occ1, dmax, dmin); occ1 = keep_hits(v1, occ1, k1);
    }
  } else if (res1) occ2 = keep_hits(v2, occ2, k2);
  else occ1 = keep_hits(v1, occ1, k1);
  return true;
}

// the pair pick, literally (new_faster_verify_pairs): smallest err sum, the first such pair, how many, and what the best stood
// at before it
__device__ __forceinline__ PePick pe_pick_seq(const bmbs_cand* v1, int occ1, const bmbs_cand* v2, int occ2, int kl, int dmax, int dmin) {
  PePick r; r.n_best = 0; r.i1 = 0; r.i2 = 0; r.sbd = 0;
  int best = 4 * kl + 2; long long second = 2LL * best, first = 0;
  if (occ1 > 0 && occ2 > 0)
    for (int i = 0; i < occ1; ++i) {
      const bmbs_cand a = v1[i];
      for (int j = (int)first; j < occ2; ++j) {
        const bmbs_cand c = v2[j];
        bool stop; const bool in = in_range(a.site, c.site, dmax, dmin, j, first, stop);
        if (stop) break;
        if (!in) continue;
        const long long sum = (long long)a.err + c.err;
        if (sum < best) { second = best; best = (int)sum; r.i1 = i; r.i2 = j; r.n_best = 1; }
        else if (sum == best) { second = best; ++r.n_best; if (best == 0) { r.sbd = 0; return r; } }
      }
    }
  if (r.n_best) r.sbd = (u32)(second - best);
  return r;
}

// The same answer by a whole warp, for lists in ascending site order without wrapped coordinates (what the skip pointer of the
// literal walk assumes to be worth anything): then "j is visited for row i" is the pure predicate |a - b| <= dmax, the rows are
// independent, and the outcome is a function of (i) the smallest sum, (ii) its first position p* in row-major order, (iii) how
// often it occurs -- two or more: second_best_diff 0, as the last equal pair sets second = best -- and (iv) for a single
// occurrence the smallest sum met before p*, which is what `best` stood at when p* was reached.  Lane l takes rows l, l + 32, ...;
// a row's partners start at a binary-searched lower bound.  ok = false: the lists do not qualify (or a sum reaches the initial
// bound 4k + 2, which the literal walk treats specially) and the caller walks them literally.
__device__ __forceinline__ PePick pe_pick_warp(const bmbs_cand* v1, int occ1, const bmbs_cand* v2, int occ2, int kl, int dmax, int dmin, int lane, bool& ok) {
  PePick r; r.n_best = 0; r.i1 = 0; r.i2 = 0; r.sbd = 0;
  bool fine = dmax >= 0;
  for (int i = lane; i < occ1; i += 32) fine = fine && v1[i].site < SITE_SANE && (i == 0 || v1[i - 1].site <= v1[i].site);
  for (int j = lane; j < occ2; j += 32) fine = fine && v2[j].site < SITE_SANE && (j == 0 || v2[j - 1].site <= v2[j].site);
  const int init = 4 * kl + 2;
  int m = 0x7FFFFFFF, cnt = 0; unsigned long long pos = ~0ull;
  auto in_pure = [&](u64 a, u64 c) { return a > c ? (long long)(a - c) >= dmin : (long long)(c - a) >= dmin; };   // |a - c| <= dmax is given
  if (__all_sync(0xffffffffu, fine)) {
    for (int i = lane; i < occ1; i += 32) {
      const bmbs_cand a = v1[i];
      const u64 lo = a.site > (u64)dmax ? a.site - (u64)dmax : 0ull, hi = a.site + (u64)dmax;
      for (int j = lower_bound_site(v2, occ2, lo); j < occ2; ++j) {
        const bmbs_cand c = v2[j];
        if (c.site > hi) break;
        if (!in_pure(a.site, c.site)) continue;
        const int sum = (int)a.err + (int)c.err;
        if (sum >= init) fine = false;
        if (sum < m) { m = sum; cnt = 1; pos = (unsigned long long)i << 32 | (unsigned)j; }
        else if (sum == m) ++cnt;
      }
    }
  }
  ok = __all_sync(0xffffffffu, fine);
  if (!ok) return r;
  int best = m;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, d));
  if (best == 0x7FFFFFFF) return r;                        // no pair within range
  int n = m == best ? cnt : 0; unsigned long long first = m == best ? pos : ~0ull;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { n += __shfl_xor_sync(0xffffffffu, n, d); const unsigned long long o = __shfl_xor_sync(0xffffffffu, first, d); first = o < first ? o : first; }
  r.n_best = n; r.i1 = (long long)(first >> 32); r.i2 = (long long)(first & 0xFFFFFFFFull);
  if (n >= 2) return r;                                    // sbd 0
  int before = init;                                       // what the running best stood at when the one best pair was reached
  for (int i = lane; i <= (int)r.i1 && i < occ1; i += 32) {
    const bmbs_cand a = v1[i];
    const u64 lo = a.site > (u64)dmax ? a.site - (u64)dmax : 0ull, hi = a.site + (u64)dmax;
    const int j_end = i == (int)r.i1 ? (int)r.i2 : occ2;
    for (int j = lower_bound_site(v2, occ2, lo); j < j_end; ++j) {
      const bmbs_cand c = v2[j];
      if (c.site > hi) break;
      if (in_pure(a.site, c.site)) before = min(before, (int)a.err + (int)c.err);
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) before = min(before, __shfl_xor_sync(0xffffffffu, before, d));
  r.sbd = (u32)(before - best);
  return r;
}

// the records of the two chosen hits
__device__ __forceinline__ void pe_emit(const DevIndex& ix, const BatchView& b, int r1, int r2, const PePick& pk, const bmbs_cand* v1, const bmbs_cand* v2,
                                        bmbs_final& o1, bmbs_final& o2, unsigned short* mm1, unsigned short* mm2, u32& n_mm1, u32& n_mm2) {
  if (pk.n_best > 1 && !b.amb_out) { o1.status = BMBS_FIN_AMBIGUOUS; return; }
  if (pk.n_best < 1) return;
  const uint8_t s8 = (uint8_t)(pk.sbd > 255u ? 255u : pk.sbd);
  o1.sbd = s8; o2.sbd = s8;
  if (pk.n_best > 1) { o1.flags |= BMBS_FINF_AMBIGUOUS; o2.flags |= BMBS_FINF_AMBIGUOUS; }
  n_mm1 = finish_hit<true>(ix, b, r1, b.len[r1], b.kk[r1], v1[pk.i1], mm1, o1);
  n_mm2 = finish_hit<true>(ix, b, r2, b.len[r2], b.kk[r2], v2[pk.i2], mm2, o2);
}

// the mismatch positions of both mates of a pair, stored from `at` on (mate 2's follow mate 1's): each record's slice, and the
// copies when they fit
__device__ __forceinline__ void pe_store_mm(const FinishView& f, unsigned long long at, bmbs_final& o1, bmbs_final& o2,
                                            const unsigned short* mm1, const unsigned short* mm2, u32 n_mm1, u32 n_mm2) {
  if (n_mm1) { o1.aux_first = (u32)at; o1.n_aux = n_mm1; }
  if (n_mm2) { o2.aux_first = (u32)(at + n_mm1); o2.n_aux = n_mm2; }
  if (at + n_mm1 + n_mm2 <= f.mism_cap) {
    for (u32 j = 0; j < n_mm1; ++j) f.mism[at + j] = mm1[j];
    for (u32 j = 0; j < n_mm2; ++j) f.mism[at + n_mm1 + j] = mm2[j];
  }
}

constexpr int PE_FIN_STAGE = 768;     // entries of each list a warp stages in shared memory in finish_pe_long

// One thread per pair; pairs with more than `pe_short` hits in both lists together (a single thread pays an L2 round trip per
// entry: a thousand entries are a millisecond) are left to finish_pe_long.
__global__ void __launch_bounds__(128) finish_pe(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  __shared__ unsigned short s_mm[128][2 * FIN_MM + 2];
  const int lane = threadIdx.x & 31;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = 2 * p + 1 < b.n_reads;
  const int r1 = 2 * p, r2 = r1 + 1;
  bmbs_final o1 = fin_blank(0), o2 = fin_blank(0);
  unsigned short* mm1 = s_mm[threadIdx.x]; unsigned short* mm2 = mm1 + FIN_MM + 1;
  u32 n_mm1 = 0, n_mm2 = 0;
  bool is_long = false;
  if (live) {
    const bmbs_read_result q1 = b.out_res[r1], q2 = b.out_res[r2];
    o1.k = b.kk[r1]; o2.k = b.kk[r2];
    if (q1.n_cand != 0 && q2.n_cand != 0) {                    // else: a mate without candidates, or nothing survived the distance filter
      if (q1.n_cand + q2.n_cand > f.pe_short) is_long = true;
      else {
        bmbs_cand* v1 = b.out_cand + q1.first_cand; bmbs_cand* v2 = b.out_cand + q2.first_cand;
        int dmax, dmin, occ1, occ2; pair_bounds(b, r1, r2, dmax, dmin);
        if (pe_compact(b, r1, r2, q1, q2, v1, v2, dmax, dmin, occ1, occ2)) {
          const int kl = max((int)b.kk[r1], (int)b.kk[r2]);
          pe_emit(ix, b, r1, r2, pe_pick_seq(v1, occ1, v2, occ2, kl, dmax, dmin), v1, v2, o1, o2, mm1, mm2, n_mm1, n_mm2);
        }
      }
    }
  }
  list_append(f.long_list, &f.fc->n_long, is_long, (u32)p);
  {
    const u32 ndp = (live && o1.status == BMBS_FIN_DP ? 1u : 0u) + (live && o2.status == BMBS_FIN_DP ? 1u : 0u);
    u32 tot = ndp;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, d);
    if (lane == 0 && tot) atomicAdd(&f.fc->n_dp, (unsigned long long)tot);
  }
  const unsigned long long at = warp_reserve(&f.fc->mism_used, n_mm1 + n_mm2);
  if (n_mm1 + n_mm2) pe_store_mm(f, at, o1, o2, mm1, mm2, n_mm1, n_mm2);
  if (live && !is_long) { f.fin[r1] = o1; f.fin[r2] = o2; }
}

// One warp per pair with long lists: the lanes copy both lists into shared memory with coalesced loads; lane 0 runs the
// in-place compaction there, the pair pick is done by the whole warp (pe_pick_warp) where the lists qualify, literally by lane 0
// otherwise (lists beyond the staging area stay in global memory).
constexpr int PE_FIN_WARPS = 4;
__global__ void __launch_bounds__(32 * PE_FIN_WARPS) finish_pe_long(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  extern __shared__ bmbs_cand s_lists[];                      // [PE_FIN_WARPS][2][PE_FIN_STAGE]
  __shared__ unsigned short s_mm[PE_FIN_WARPS][2 * FIN_MM + 2];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const u32 n_long = (u32)f.fc->n_long;
  bmbs_cand* s1 = s_lists + (size_t)w * 2 * PE_FIN_STAGE; bmbs_cand* s2 = s1 + PE_FIN_STAGE;
  for (;;) {
    const u32 g = warp_next(&f.fc->cursor_long);
    if (g >= n_long) break;
    const int p = (int)f.long_list[g], r1 = 2 * p, r2 = r1 + 1;
    const bmbs_read_result q1 = b.out_res[r1], q2 = b.out_res[r2];
    bmbs_cand* v1 = b.out_cand + q1.first_cand; bmbs_cand* v2 = b.out_cand + q2.first_cand;
    if (q1.n_cand <= (u32)PE_FIN_STAGE && q2.n_cand <= (u32)PE_FIN_STAGE) {
      for (u32 i = lane; i < q1.n_cand; i += 32) s1[i] = v1[i];
      for (u32 i = lane; i < q2.n_cand; i += 32) s2[i] = v2[i];
      v1 = s1; v2 = s2;
    }
    __syncwarp();
    int dmax, dmin, occ1 = 0, occ2 = 0; pair_bounds(b, r1, r2, dmax, dmin);
    const int kl = max((int)b.kk[r1], (int)b.kk[r2]);
    int alive = 0;
    if (lane == 0) alive = pe_compact(b, r1, r2, q1, q2, v1, v2, dmax, dmin, occ1, occ2) ? 1 : 0;
    __syncwarp();
    alive = __shfl_sync(0xffffffffu, alive, 0); occ1 = __shfl_sync(0xffffffffu, occ1, 0); occ2 = __shfl_sync(0xffffffffu, occ2, 0);
    PePick pk; pk.n_best = 0; pk.i1 = 0; pk.i2 = 0; pk.sbd = 0;
    if (alive) {
      bool ok = false;
      pk = pe_pick_warp(v1, occ1, v2, occ2, kl, dmax, dmin, lane, ok);
      if (!ok && lane == 0) pk = pe_pick_seq(v1, occ1, v2, occ2, kl, dmax, dmin);
    }
    if (lane == 0) {
      bmbs_final o1 = fin_blank(b.kk[r1]), o2 = fin_blank(b.kk[r2]);
      unsigned short* mm1 = s_mm[w]; unsigned short* mm2 = mm1 + FIN_MM + 1;
      u32 n_mm1 = 0, n_mm2 = 0;
      if (alive) pe_emit(ix, b, r1, r2, pk, v1, v2, o1, o2, mm1, mm2, n_mm1, n_mm2);
      const u32 ndp = (o1.status == BMBS_FIN_DP ? 1u : 0u) + (o2.status == BMBS_FIN_DP ? 1u : 0u);
      if (ndp) atomicAdd(&f.fc->n_dp, (unsigned long long)ndp);
      if (n_mm1 + n_mm2) pe_store_mm(f, atomicAdd(&f.fc->mism_used, (unsigned long long)(n_mm1 + n_mm2)), o1, o2, mm1, mm2, n_mm1, n_mm2);
      f.fin[r1] = o1; f.fin[r2] = o2;
    }
    __syncwarp();
  }
}
