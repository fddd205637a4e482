// The end fix-ups of the CIGAR refinement (fast_recalculate_bs_Cigar, ksw.cpp:2894-2990).  Host + device: refine_warp runs
// it on the device after its traceback, host/postprocess.hpp's refine_alignment on the CPU, where
// tests/test_refine_vs_reference.py pins it to the reference.
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

// ops[0..n) is the traceback in read order, (len << 4) | op with 0 = M, 1 = D, 2 = I.  The read is aligned end to end, so
// insertions at either end become matches and the window span [qb, qe] grows with them.  ops[cb..ce] is what stays.
BMBS_HD void refine_fix_ends(uint32_t* ops, int n, int& qb, int& qe, int& cb, int& ce) {
  int i = 0; uint32_t ins = 0;
  for (; i < n && (ops[i] & 0xfu) == 2u; ++i) ins += ops[i] >> 4;
  if (i != 0) {
    uint32_t op = ops[i] & 0xfu, len = ops[i] >> 4;   // (i == n cannot happen for a non-empty read with a match)
    if (op == 0) len += ins; else { op = 0; len = ins; --i; }
    ops[i] = len << 4 | op;
    qb -= (int)ins;
  }
  cb = i;
  ins = 0;
  for (i = n - 1; i >= cb && (ops[i] & 0xfu) == 2u; --i) ins += ops[i] >> 4;
  if (i != n - 1) {
    uint32_t op = ops[i] & 0xfu, len = ops[i] >> 4;
    if (op == 0) len += ins; else { op = 0; len = ins; ++i; }
    ops[i] = len << 4 | op;
    qe += (int)ins;
  }
  ce = i;
}

}  // namespace bmbs
