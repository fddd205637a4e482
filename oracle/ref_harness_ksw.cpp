// oracle/ (test infrastructure): exposes the REFERENCE's own CIGAR refinement -- fast_recalculate_bs_Cigar (ksw.cpp:2578-3148)
// with try_cigar_without_path (:2515-2570) and ksw_semi_global_quality_back (:1850-2045) -- through a C ABI, with the
// substitution matrices set up as Prepare_alignment does (Schema.cpp:828-850).  Compiled by build_ref.sh from a scratch copy
// of /root/reference; pins host/postprocess.hpp's refine_alignment (CPU) and the refine_warp kernels (GPU) for SURVEY.md 8f-1.
#include <cstdint>
#include <cstring>
#include "ksw.h"

extern "C" int ref_cigar(const char* window, int wlen, const char* read, int rlen, int k, int end_site, int err, int is_forward,
                         int mp_max, int mp_min, int n_pen, int gap_open, int gap_ext, const char* qual, int need_r_quality, int q_base,
                         int* start_site, uint64_t* out_end, unsigned* out_err, int* score, char* cigar) {
  int8_t mat[25], mat_diff[25];
  int i, j, kk;
  for (i = kk = 0; i < 4; ++i) {
    for (j = 0; j < 4; ++j) { mat_diff[kk] = i == j ? 0 : (mp_max - mp_min); mat[kk++] = i == j ? 0 : -mp_min; }
    mat_diff[kk] = 0; mat[kk++] = -n_pen;
  }
  for (j = 0; j < 5; ++j) { mat_diff[kk] = 0; mat[kk++] = -n_pen; }
  mat_diff[16] = 0; mat[16] = 0;
  char qbuf[2048]; memcpy(qbuf, qual, rlen); qbuf[rlen] = 0;     // the reference reverses the qualities in place and restores them
  bitmapper_bs_iter e = (bitmapper_bs_iter)end_site;
  *out_err = (unsigned)err;          // the reference's callers pass the candidate's own err / end_site fields as the out parameters (Schema.cpp:14753-14756)
  int r = fast_recalculate_bs_Cigar((char*)window, wlen, (char*)read, rlen, (unsigned short)k, end_site, err, start_site, &e, out_err, score, cigar,
                                    is_forward, mat, mat_diff, gap_open, gap_ext, mp_max, mp_min, n_pen, qbuf, need_r_quality, q_base);
  *out_end = e;
  return r;
}
