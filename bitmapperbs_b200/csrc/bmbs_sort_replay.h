// The order libstdc++'s std::sort leaves a vote-sorted window list in, recomputed without std::sort.
//
// The reference reduces a read's verified windows in the order `std::sort(votes, votes + n, by vote descending)` leaves them
// (Schema.cpp:27612, comparator :560-563).  That sort is unstable, and second_best_diff / the chosen window depend on the order
// among equal votes, so the device finishing (finish_sorted, bmbs_kernels.cuh) replays the algorithm itself: the sequence of
// comparisons and moves depends only on the keys, so sorting (vote << 16 | position) words yields the permutation the
// reference's 32-byte structs end up in.  Algorithm = GCC's bits/stl_algo.h (unchanged since 4.x; checked against the
// std::sort of this toolchain in tests/test_sort_replay.py): introsort loop with depth limit 2*floor(log2 n), median of
// (first+1, middle, last-1) moved to first, unguarded Hoare partition, ranges of <= 16 left for one final insertion sort
// (guarded over the first 16, unguarded after).  The heap-sort fallback of an exhausted depth limit is not replayed: the
// function returns false and the caller hands the read to the host.
#pragma once
#include <cstdint>

#ifndef BMBS_HD
#if defined(__CUDACC__)
#define BMBS_HD __host__ __device__ __forceinline__
#else
#define BMBS_HD inline
#endif
#endif

namespace bmbs {

BMBS_HD bool vote_before(uint32_t x, uint32_t y) { return (x >> 16) > (y >> 16); }   // comp(a, b): a.vote > b.vote

BMBS_HD void replay_linear_insert(uint32_t* a, int last) {                          // __unguarded_linear_insert
  const uint32_t val = a[last];
  int next = last - 1;
  while (vote_before(val, a[next])) { a[last] = a[next]; last = next; --next; }
  a[last] = val;
}

BMBS_HD void replay_insertion_sort(uint32_t* a, int first, int last) {              // __insertion_sort
  if (first == last) return;
  for (int i = first + 1; i != last; ++i) {
    if (vote_before(a[i], a[first])) {
      const uint32_t val = a[i];
      for (int j = i; j > first; --j) a[j] = a[j - 1];
      a[first] = val;
    } else replay_linear_insert(a, i);
  }
}

// a[0..n): keys (vote << 16 | anything).  Returns false when the depth limit ran out (heap sort would take over).
BMBS_HD bool sort_replay(uint32_t* a, int n) {
  if (n <= 1) return true;
  int lg = 0; while ((n >> (lg + 1)) != 0) ++lg;
  // __introsort_loop: the recursive call on the right part becomes a stack entry (the two parts are independent)
  int st_first[64], st_last[64], st_depth[64]; int sp = 0;
  st_first[0] = 0; st_last[0] = n; st_depth[0] = 2 * lg; sp = 1;
  while (sp) {
    --sp;
    int first = st_first[sp], last = st_last[sp], depth = st_depth[sp];
    while (last - first > 16) {
      if (depth == 0) return false;
      --depth;
      const int ia = first + 1, ib = first + (last - first) / 2, ic = last - 1;   // __move_median_to_first
      int pick;
      if (vote_before(a[ia], a[ib])) { if (vote_before(a[ib], a[ic])) pick = ib; else if (vote_before(a[ia], a[ic])) pick = ic; else pick = ia; }
      else if (vote_before(a[ia], a[ic])) pick = ia;
      else if (vote_before(a[ib], a[ic])) pick = ic;
      else pick = ib;
      { const uint32_t t = a[first]; a[first] = a[pick]; a[pick] = t; }
      const uint32_t pivot = a[first];                                            // __unguarded_partition(first + 1, last, first)
      int lo = first + 1, hi = last;
      for (;;) {
        while (vote_before(a[lo], pivot)) ++lo;
        --hi;
        while (vote_before(pivot, a[hi])) --hi;
        if (!(lo < hi)) break;
        const uint32_t t = a[lo]; a[lo] = a[hi]; a[hi] = t;
        ++lo;
      }
      if (sp >= 64) return false;
      st_first[sp] = lo; st_last[sp] = last; st_depth[sp] = depth; ++sp;
      last = lo;
    }
  }
  if (n > 16) {                                                                   // __final_insertion_sort
    replay_insertion_sort(a, 0, 16);
    for (int i = 16; i < n; ++i) replay_linear_insert(a, i);
  } else replay_insertion_sort(a, 0, n);
  return true;
}

}  // namespace bmbs
