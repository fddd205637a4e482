// The last column of the banded bit-vector verification, walked from VN run to VN run (BS_Reserve_Banded_BPM,
// Levenshtein_Cal.h:524-563).  Host + device: verify_windows calls it for both band widths, tests/band_walk_harness.cpp
// checks it on the CPU against the reference's cell-by-cell loop over band states produced by the column recurrence itself.
//
// After the last read base, position p = 0 .. 2k of the band is the cell whose alignment ends at window position L - 1 + p,
//   S(p) = err + (VP bits below p) - (VN bits below p),
// err being the value on the band's diagonal.  The reference walks p upwards and keeps the LAST position that holds the
// column's minimum (if that is within k), except that the un-gapped end p = k wins a tie.  S only falls on VN bits, so the
// minimum stands either on the first plateau (from p = 0 to the first set bit) or on the plateau that follows a run of VN
// bits: the walk goes from run to run (two or three per window) instead of cell by cell, and a window whose smallest possible
// value err - popc(VN) is beyond k is not walked at all.
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

template <typename W>
BMBS_HD int bw_popc(W x) {
#if defined(__CUDA_ARCH__)
  return sizeof(W) == 8 ? __popcll((unsigned long long)x) : __popc((unsigned)x);
#else
  return sizeof(W) == 8 ? __builtin_popcountll((unsigned long long)x) : __builtin_popcount((unsigned)x);
#endif
}
template <typename W>
BMBS_HD int bw_ffs(W x) {                 // 1-based position of the lowest set bit, 0 for x == 0
#if defined(__CUDA_ARCH__)
  return sizeof(W) == 8 ? __ffsll((long long)x) : __ffs((int)x);
#else
  return sizeof(W) == 8 ? __builtin_ffsll((long long)x) : __builtin_ffs((int)x);
#endif
}

// W = a 32-bit (k <= 15) or 64-bit (k <= 31) unsigned word; VP / VN: the band after the last column; err: the diagonal's value there.
// -> end_out = window position where the best alignment ends (-1: none within k), err_out = its edit distance (0xFFFFFFFF: none)
template <typename W>
BMBS_HD void band_last_column(W VP, W VN, int err, int k, int L, int& end_out, uint32_t& err_out) {
  end_out = -1; err_out = 0xFFFFFFFFu;
  const int last = L - 1;
  const W bm = (W)(((W)1 << (2 * k)) - 1);                  // bits 0 .. 2k-1
  const W vp = VP & bm, vn = VN & bm, any = vp | vn;
  if (err - bw_popc(vn) > k) return;
  uint32_t best = 0xFFFFFFFFu; int site = -1;
  if (err <= k) { best = (uint32_t)err; site = last + (any ? bw_ffs(any) - 1 : 2 * k); }
  for (W rest = vn; rest;) {
    const int a = bw_ffs(rest) - 1;                        // a run of VN bits [a, b)
    const int b = a + bw_ffs((W)~(W)(vn >> a)) - 1;
    const W below = (W)(((W)1 << b) - 1);
    const int cur = err + bw_popc((W)(vp & below)) - bw_popc((W)(vn & below));     // S(b)
    const W above = (W)(any >> b);
    if (cur <= k && (uint32_t)cur <= best) { best = (uint32_t)cur; site = last + (above ? b + bw_ffs(above) - 1 : 2 * k); }
    rest &= (W)~below;
  }
  const W below_k = (W)(((W)1 << k) - 1);
  const int ungapped = err + bw_popc((W)(vp & below_k)) - bw_popc((W)(vn & below_k));   // S(k)
  if (ungapped <= k && (uint32_t)ungapped == best) site = last + k;
  end_out = site; err_out = best;
}

}  // namespace bmbs
