// CUDA kernels of the seed-and-verify path (sm_100a; integer / bit-vector work, no tensor cores).
//
//   pack_reads       ASCII -> nibble codes + bit-plane chunks, first-C position, error threshold k
//   seed_reads       kernel 1a: every seed of a read (first seed + unique-hit shortcut with direct genome compare, the
//                    one-mismatch second seed, the remaining greedy seeds), one persistent kernel, a lane per read
//   expand_locate    kernel 1b: seed intervals -> one candidate site per row (dense suffix array gather, or LF-walk to a sampled row)
//   votes_classify   kernel 2: what a read's candidates turn into; short segments sorted + run-length encoded in registers
//   votes_sort<32>, votes_mid, votes_big1k, votes_big   kernel 2 for segments of 17..32 (a warp, one key per lane), 33..256 (a warp, eight keys
//                    per lane), 257..1024 (a CTA, eight keys per thread) and longer (a CTA over shared / global memory)
//   filter_pairs_kernel         kernel 2b (paired end): distance pre-filter of the two mates' lists
//   gather_work      the surviving windows as one VerifyItem each (resolved reads get their record directly)
//   verify_windows   kernel 3: banded Myers bit-vector edit distance, read T may face reference C
//   sens_pair, reseed_clear, seed_reseed, sens_reseed_filter, sens_reseed_finish   --pe --sensitive: pair logic and the re-seeding round
//   refine_warp<1>, refine_warp<2>   CIGAR refinement: banded affine-gap DP with traceback (SURVEY 8f-1), a warp per item,
//                    one or two band cells per lane
//   finalize_reads   per-read result records
//   finish_se, finish_long, finish_huge, finish_sorted   single-end finishing on the device: a thread / a warp / a CTA per
//                    read by the length of its window list, and the replay of std::sort's order where the order decides
//   finish_pe, finish_pe_long   paired-end finishing (bmbs_finish_pe.cuh)
//   debug_sort_order test entry: the order std::sort leaves a list in, through finish_sorted's warp routine
//   scan_tiles, scan_tile_sums, scan_apply   exclusive scan of per-read counts into offsets, with capacity checks
#pragma once
#include "bmbs_device.cuh"
#include "bmbs_sort_replay.h"
#include "bmbs_band_walk.h"
#include "bmbs_refine_ends.h"
#include "../../include/bmbs.h"

namespace bmbs {

constexpr int MAX_TASKS = 28;       // 25 seeds + first-seed literal + second seed + slack
constexpr u32 MAX_SEED_HITS = 1000; // Schema.cpp:26826 max_seed_matches
constexpr u32 MAX_PE_MULTI = 10000; // Schema.cpp:21719-21737 max_candidates_occ of Map_Pair_Seq_split_fast: 25 x 1000, then clamped to 10000
constexpr u32 MAX_PE_MULTI_SENSITIVE = 10000; // Schema.cpp:22713-22716 (sensitive pair mode)

struct SeedTask { u64 sp; u32 hits; unsigned short mlen, off; };  // hits==0: `sp` is a literal site

// counters (device, u64[16]); indices follow bmbs_batch_counters
enum { CNT_HASH = 0, CNT_OCC = 1, CNT_ROWS = 2, CNT_LOCATE_LF = 3, CNT_VERIFIED = 4, CNT_CELLS = 5, CNT_CAND = 6, CNT_WINBYTES = 7 };

// One window for the bit-vector kernel, everything it needs in one 32-byte record (one load instead of a chain of
// dependent gathers through the read tables): window start, slot in out_cand, votes, where the read's nibble codes start,
// read length and error threshold.
struct __align__(16) VerifyItem { u64 site; u32 wi, vote, code_off, L, k, pad; };

struct BatchView {
  // inputs
  const char* ascii; const u64* offsets; int n_reads; int pe;
  // per read
  u32* codes; uint4* rplanes; u32* len; unsigned short* first_c; unsigned char* kk;   // rplanes: {lo, hi, not-ACGT, is-N} per 32 bases
  unsigned char* state; unsigned char* flags;  // flags: bit0 is_multi, bit1 extra==0 (second seed conclusive)
  short* one_mm; u64* site0;
  // list_count[0]: reads seed_reads has taken (its read cursor); [1]: unused; [2]: mates in list4, to re-seed;
  // [3]: windows in vitems, to verify
  u32* list_count;
  // --pe --sensitive (Map_Pair_Seq_split, Schema.cpp:22450): bookkeeping of the seeds that were used
  // {count, start[0], start[1], end of the one before last, end of the last} (select_best_seeds, :16630), the
  // number of candidates after the first seed (decides which mate goes first, :23326), the list of mates to
  // re-seed, and each read's final slice of out_cand
  unsigned short* bk; unsigned short* first_cands; u32* list4; u32* res_first; u32* res_n;
  int sensitive; int round;                     // round 1 = the re-seeding pass
  int amb_out;                                  // --ambiguous_out: single-end multi-exact reads keep their located rows, in row order
  u32 multi_cap;
  u32* ntask; u32* ncand; u32* coff;           // coff: exclusive scan of ncand, n_reads+1
  SeedTask* tasks;                              // [MAX_TASKS][n_reads]
  // per candidate slot
  u64* slot_row; u32* slot_adj; u32* slot_read; u64* cand; u32* vcnt;
  u32* nv; u32* voff;                           // votes per read, exclusive scan
  unsigned char* keep;
  // work list
  VerifyItem* vitems; bmbs_cand* out_cand;      // dense list of the windows that need the bit-vector kernel (count: list_count[3])
  bmbs_read_result* out_res;
  u32* sort32; u32* sort_count;                  // reads whose candidate segment (17..32 entries) is sorted by a warp; count in sort_count[1]
  u32* mid_list; u32* big1k_list;                // segments of 33..256 (a warp, eight keys per lane; count in sort_count[2]) and 257..1024 (a CTA; sort_count[3])
  u32* big_list; u32* big_count; u64* scratch; u32* scratch_used; u64 scratch_cap;
  u64* counters; u64* totals;   // totals[0] candidate slots, [1] verification work items of this round, [2] out_cand base of this round, [3] out_cand entries in all
  u32* status;                  // bit0 per-read task overflow, bit1 slot capacity, bit2 work capacity, bit3 scratch
  u64 slot_cap;
  double e_rate; u32 seed_len; int dmax_base, dmin_base;  // pair distance bounds before the per-pair 2k / length terms
};

// a read owns (L >> 5) + 1 chunks of 32 bases: one uint4 of bit-planes and four code words (16-byte aligned) per chunk
__device__ __forceinline__ u32 plane_chunk_offset(const u64* offsets, int r) { return (u32)(offsets[r] >> 5) + (u32)r; }
__device__ __forceinline__ u32 code_word_offset(const u64* offsets, int r) { return 4u * plane_chunk_offset(offsets, r); }

// ------------------------------------------------------------------------------------------- pack
// Eight lanes per read, one 32-base chunk per lane and pass: 32 ASCII bytes (aligned 64-bit loads + funnel shifts) become
// four u32 of nibble codes (A0 C1 G2 T3, anything else 4; used by verification) and one bit-plane chunk {lo, hi, not-ACGT,
// is-N} (used by seeding).  Four bases at a time (SWAR): code = bits 1-2 of the byte, folded; a byte is valid when it equals
// "ACGT"[code] (one PRMT); planes are gathered with a multiply.  Anything that is not A/C/G/T takes the rare slow path.
__device__ __forceinline__ u32 gather4(u32 m01) { return ((m01 * 0x01020408u) >> 24) & 0xFu; }   // byte t bit 0 -> bit t
__device__ __forceinline__ u32 nonzero_bytes(u32 d) { return ((((d & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | d) >> 7) & 0x01010101u; }

struct Packed4 { u32 nib, lo, hi, bad, isn; };
// General path, four bases: handles anything that is not A/C/G/T and the ragged end of a read.
__device__ __forceinline__ Packed4 pack4(u32 x, u32 nvalid) {
  const u32 y = (x >> 1) & 0x03030303u;
  const u32 code = y ^ ((y >> 1) & 0x01010101u);                  // A0 C1 G2 T3 when the byte is one of ACGT
  const u32 t = (code & 0x00030003u) | ((code >> 4) & 0x00300030u);
  u32 nib = (t | (t >> 8)) & 0xFFFFu;
  u32 b0 = code & 0x01010101u, b1 = (code >> 1) & 0x01010101u;
  const u32 diff = x ^ __byte_perm(0x54474341u, 0u, nib);          // "ACGT"[code] per byte
  Packed4 o; o.bad = 0; o.isn = 0;
  if (diff != 0 || nvalid < 4) {
    const u32 keep = nvalid >= 4 ? 0x01010101u : (((1u << (8 * nvalid)) - 1u) & 0x01010101u);
    const u32 bad = nonzero_bytes(diff) & keep;
    const u32 isn = (~nonzero_bytes(x ^ 0x4E4E4E4Eu)) & 0x01010101u & keep;
    b0 &= keep & ~bad; b1 &= keep & ~bad;
    const u32 cb = b0 | (b1 << 1) | (bad << 2);                     // per byte: 0..3, anything else 4
    nib = (cb & 0xFu) | ((cb >> 4) & 0xF0u) | ((cb >> 8) & 0xF00u) | ((cb >> 12) & 0xF000u);
    o.bad = gather4(bad); o.isn = gather4(isn);
  }
  o.nib = nib; o.lo = gather4(b0); o.hi = gather4(b1);
  return o;
}

// Fast path, eight bases that are all A/C/G/T (checked; false = take the general path).  For A 0x41, C 0x43, G 0x47, T 0x54
// the code (A0 C1 G2 T3) is in the byte: high bit = bit 2, low bit = bit 1 ^ bit 2.  Each plane's eight bits are gathered
// with one multiply (no two partial products meet, so no carries), the nibble codes are spread back out of the planes with
// three multiply-and-mask steps, the bytes are checked against "ACGT"[code] (PRMT).  Half of the work is IMADs, which run
// on the FMA pipe this ALU-bound kernel otherwise leaves idle.
__device__ __forceinline__ u32 spread8(u32 v) {                   // bit i of an 8-bit value -> bit 4i
  u32 t = (v * 0x1001u) & 0x000F000Fu;
  t = (t * 0x41u) & 0x03030303u;
  return (t * 9u) & 0x11111111u;
}
__device__ __forceinline__ bool pack8(u32 x0, u32 x1, u32& nib, u32& lo8, u32& hi8) {
  const u32 a1 = x0 >> 1, a2 = x0 >> 2, c1 = x1 >> 1, c2 = x1 >> 2;
  const u32 l0 = (a1 ^ a2) & 0x01010101u, h0 = a2 & 0x01010101u, l1 = (c1 ^ c2) & 0x01010101u, h1 = c2 & 0x01010101u;
  lo8 = ((l1 * 16u + l0) * 0x01020408u) >> 24;                    // bases 0-3 in bits 0-3, bases 4-7 in bits 4-7
  hi8 = ((h1 * 16u + h0) * 0x01020408u) >> 24;
  nib = spread8(hi8) * 2u + spread8(lo8);
  const u32 d0 = x0 ^ __byte_perm(0x54474341u, 0u, nib), d1 = x1 ^ __byte_perm(0x54474341u, 0u, nib >> 16);
  return (d0 | d1) == 0;
}

__global__ void __launch_bounds__(128) pack_reads(BatchView b) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, sub = threadIdx.x & 7;
  const bool live = r < b.n_reads;
  u64 beg = 0; u32 L = 0;
  if (live) { beg = b.offsets[r]; L = (u32)(b.offsets[r + 1] - beg); }
  u32* w = b.codes + (live ? code_word_offset(b.offsets, r) : 0);
  uint4* pl = b.rplanes + (live ? plane_chunk_offset(b.offsets, r) : 0);
  u32 first_c = L;
  for (u32 c = sub; c * 32 < L; c += 8) {
    const u64 addr = (u64)(b.ascii) + beg + (u64)c * 32;
    const u64* q = (const u64*)(addr & ~7ull);
    const unsigned sh = (unsigned)(addr & 7ull) * 8;
    u64 x[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) x[i] = __ldg(q + i);            // staging buffers carry 64 bytes of slack past the last read
    if (sh) {
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = (x[i] >> sh) | (x[i + 1] << (64 - sh));
    }
    const u32 left = L - c * 32;                                // >= 1
    u32 lo = 0, hi = 0, bad = 0, isn = 0;
    u32 nw[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const u32 base = 8 * i;
      u32 n8, l8, h8;
      // the bytes behind a ragged end are the next read's bases (or slack): when they happen to be A/C/G/T too the group
      // still takes the fast path and its results are cut to the bases that belong to this read
      if (base < left && pack8((u32)x[i], (u32)(x[i] >> 32), n8, l8, h8)) {
        const u32 nb = left - base;
        if (nb < 8) { n8 &= (1u << (4 * nb)) - 1u; l8 &= (1u << nb) - 1u; h8 &= (1u << nb) - 1u; }
        nw[i] = n8;
        lo |= l8 << base; hi |= h8 << base;
      } else if (base < left) {
        const Packed4 a = pack4((u32)x[i], left - base);
        const Packed4 d = pack4((u32)(x[i] >> 32), left > base + 4 ? left - base - 4 : 0);
        nw[i] = a.nib | (d.nib << 16);
        lo |= (a.lo | (d.lo << 4)) << base; hi |= (a.hi | (d.hi << 4)) << base;
        bad |= (a.bad | (d.bad << 4)) << base; isn |= (a.isn | (d.isn << 4)) << base;
      }
    }
    *reinterpret_cast<uint4*>(w + c * 4) = make_uint4(nw[0], nw[1], nw[2], nw[3]);
    pl[c] = make_uint4(lo, hi, bad, isn);
    const u32 isc = lo & ~hi & ~bad;
    if (isc) first_c = min(first_c, c * 32 + (u32)__ffs(isc) - 1u);
  }
  for (int o = 4; o; o >>= 1) first_c = min(first_c, __shfl_xor_sync(0xffffffffu, first_c, o));
  if (live && sub == 0) {
    b.len[r] = L;
    b.first_c[r] = (unsigned short)first_c;
    u64 k = (u64)(b.e_rate * (double)L);   // Schema.cpp:27121: double product truncated, capped at 31
    b.kk[r] = (unsigned char)(k >= 31 ? 31 : k);
  }
}

// ------------------------------------------------------------------------------------------- seed
struct SeedHit { u64 hits, sp, ep; u32 mlen; bool has_sa; u64 sa; };   // has_sa: one row left and its suffix-array value is already known

// Read bases as bit-planes.  FM alphabet of the reversed, C->T converted read: G0 T1 A2, anything else stops a seed;
// from the planes (A00 C01 G10 T11): fm = lo | ((~lo & ~hi) << 1).
// A seeding thread looks at its read many times (every seed, every 32 symbols of an extension); between two looks the
// random table / occ sectors of the whole SM have flushed L1 and much of L2, so the chunks are staged once per read in
// shared memory (column `threadIdx.x` of s[chunk][blockDim.x]; `ns` chunks, longer reads fall back to global memory).
constexpr int SEED_BLOCK = 128;
struct ReadPlanes {
  const uint4* p; const uint4* s; u32 ns;
  __device__ __forceinline__ void stage(const uint4* src, u32 L, uint4* smem_col, u32 cap) {
    p = src; s = smem_col;
    ns = (L >> 5) + 2; if (ns > cap) ns = cap;           // chunks 0 .. L/32 hold bases, +1 for the look-ahead of window()
    for (u32 i = 0; i < ns; ++i) smem_col[i * SEED_BLOCK] = __ldg(src + i);
  }
  __device__ __forceinline__ uint4 chunk(u32 i) const { return i < ns ? s[i * SEED_BLOCK] : __ldg(p + i); }
  __device__ __forceinline__ void window(u32 pos, u32& lo, u32& hi, u32& bad) const {   // 32 bases starting at pos
    const uint4 a = chunk(pos >> 5), c = chunk((pos >> 5) + 1);
    const unsigned s = pos & 31u;
    lo = __funnelshift_r(a.x, c.x, s); hi = __funnelshift_r(a.y, c.y, s); bad = __funnelshift_r(a.z, c.z, s);
  }
};

// base-3 value of 16 FM symbols (first base least significant) through a 4-base table in shared memory
__device__ __forceinline__ bool key16(const ReadPlanes& rp, const unsigned char* __restrict__ lut, u32 off, u32& key) {
  u32 lo, hi, bad; rp.window(off, lo, hi, bad);
  if (bad & 0xFFFFu) return false;
  const u32 a = (lo & 0xFFFFu) | ((~lo & ~hi) << 16);      // low half: fm bit 0, high half: fm bit 1
  const u32 i0 = (a & 0xFu) | ((a >> 12) & 0xF0u), i1 = ((a >> 4) & 0xFu) | ((a >> 16) & 0xF0u);
  const u32 i2 = ((a >> 8) & 0xFu) | ((a >> 20) & 0xF0u), i3 = ((a >> 12) & 0xFu) | ((a >> 24) & 0xF0u);
  key = (u32)lut[i0] + 81u * (u32)lut[i1] + 6561u * (u32)lut[i2] + 531441u * (u32)lut[i3];
  return true;
}

// FM symbols of read[pos ..], 32 at a time, consumed one per LF step; lo / hi / bad: the 32 bases from pos on
struct SymbolStream {
  const ReadPlanes& rp; u32 base, lo, hi, bad;
  __device__ __forceinline__ SymbolStream(const ReadPlanes& r, u32 pos, u32 l, u32 h, u32 b) : rp(r), base(pos), lo(l), hi(h), bad(b) {}
  __device__ __forceinline__ int at(u32 pos) {       // pos >= base, non-decreasing
    if (pos - base >= 32u) { base = pos; rp.window(pos, lo, hi, bad); }
    const unsigned s = pos - base;
    if ((bad >> s) & 1u) return 3;
    const u32 l = (lo >> s) & 1u, h = (hi >> s) & 1u;
    return (int)(l | ((~(l | h) & 1u) << 1));
  }
};

// symbols 16..K-1 of the seed at `off` as the extension index of the deep table; false when one of them is not A/C/G/T
__device__ __forceinline__ bool kmer_ext(const DevIndex& ix, const unsigned char* __restrict__ lut, u32 lo, u32 hi, u32 bad, u32& ext) {
  const u32 mask = (1u << ix.kdepth) - 1u;
  if (bad & mask) return false;
  ext = lut[(lo & mask) | (((~lo & ~hi) & mask) << 4)];
  return true;
}

// The start of a seed at read[off] (reversed, C->T converted read; the seed grows to the right, cur bases are available):
// the 16-mer key, then the deep table's entry for the first 16 + kdepth symbols or, without one, the 16-mer table.
// `exact` selects the rules of count_hash_table (bwt.h:1848-1952) over those of count_backward_as_much_1_terminate
// (bwt.h:2081-2209).  They differ in three places: at least 17 bases instead of 18; a deep entry that stops short with two
// or more rows means no hit instead of being the answer; a single-row entry goes on to the LF loop instead of being the answer.
// Returns START_NONE (no hit: m = 0, top = bot = 0), START_ANSWER (rows [top, bot) after m symbols are the seed's answer) or
// START_LF (the LF loop goes on from rows [top, bot) after m symbols).  one_sa: a single row whose suffix-array value is top
// (a deep-table entry of one row holds it).  lo / hi / bad: the 32 bases from off + 16 on, the LF loop's first window (set
// unless the key failed).  A dead seed's values are set in one place, at the end: with a return per case instead, seed_reads
// takes 64 registers instead of 56.
enum { START_NONE = 0, START_ANSWER = 1, START_LF = 2 };
__device__ __forceinline__ int seed_start(const DevIndex& ix, const ReadPlanes& rp, const unsigned char* lut, u32 off, u32 cur, bool exact,
                                          u32& m, u64& top, u64& bot, bool& one_sa, u32& lo, u32& hi, u32& bad, u32& n_hash) {
  int how = START_LF;
  u32 key;
  one_sa = false;
  if (cur < (exact ? 17u : 18u) || !key16(rp, lut, off, key)) how = START_NONE;
  else {
    m = 16;
    rp.window(off + 16, lo, hi, bad);
    bool in_table = false;                                        // the deep table has the answer (else: the 16-mer table)
    if (ix.ktab && cur >= 16 + ix.kdepth) {
      u32 ext;
      if (kmer_ext(ix, lut, lo, hi, bad, ext)) {
        const u64 e = __ldg(ix.ktab + (u64)key * ix.kpow + ext); ++n_hash;
        const u64 size = e >> 39; const u32 code = (u32)(e >> 36) & 7u;
        if (size != KTAB_SAT) {
          in_table = true;
          if (code == 0) how = START_NONE;                        // the 16-mer does not occur
          else {
            m = 15 + code; top = e & 0xFFFFFFFFFull; bot = top + size; one_sa = size == 1;
            const bool stops_short = m < 16 + ix.kdepth;
            if (!exact) { if (one_sa || stops_short) how = START_ANSWER; }
            else if (stops_short && size >= 2) how = START_NONE;   // the next symbol empties the interval
          }
        }
      }
    }
    if (!in_table) {
      hash_query(ix, key, top, bot); ++n_hash;
      if (bot <= top) how = START_NONE;
    }
  }
  if (how == START_NONE) { m = 0; top = 0; bot = 0; one_sa = false; }
  return how;
}

// read[off+from .. off+cur) against the C->T converted double-strand sequence, read[off] at s0; false on a mismatch or when
// the text ends before the pattern does.  32 bases per step on bit-planes; 3-letter equality: lo set (C/T) ignores hi.
__device__ __forceinline__ bool exact_tail_matches(const DevIndex& ix, const ReadPlanes& rp, u64 s0, u32 off, u32 from, u32 cur) {
  if (s0 + cur > 2 * ix.N) return false;
  for (u32 p = off + from; p < off + cur; p += 32) {
    u32 rlo, rhi, rbad; rp.window(p, rlo, rhi, rbad);
    const u64 g = s0 + (p - off);
    const uint2 w0 = __ldg(ix.planes + (g >> 5)), w1 = __ldg(ix.planes + (g >> 5) + 1);
    const unsigned sh = (unsigned)g & 31u;
    const u32 glo = __funnelshift_r(w0.x, w1.x, sh), ghi = __funnelshift_r(w0.y, w1.y, sh);
    u32 mism = (rlo ^ glo) | (~rlo & (rhi ^ ghi)) | rbad;
    const u32 left = off + cur - p;
    if (left < 32u) mism &= (1u << left) - 1u;
    if (mism) return false;
  }
  return true;
}

// count_backward_as_much_1_terminate (bwt.h:2081-2209) on the reversed, C->T converted read:
// the seed starts at read[off] and grows to the right; cur = L - off bases are available.
__device__ __forceinline__ SeedHit seed_until_unique(const DevIndex& ix, const ReadPlanes& rp, const unsigned char* lut, u32 off, u32 cur,
                                                     u32& n_occ, u32& n_hash) {
  u32 m = 0, lo = 0, hi = 0, bad = 0; u64 top = 0, bot = 0; bool one_sa = false;
  const int how = seed_start(ix, rp, lut, off, cur, false, m, top, bot, one_sa, lo, hi, bad, n_hash);
  SeedHit h; h.hits = 0; h.sp = 0; h.ep = 0; h.mlen = m; h.has_sa = false; h.sa = 0;
  if (how == START_NONE) return h;
  if (how == START_ANSWER) {
    if (one_sa) { h.hits = 1; h.has_sa = true; h.sa = top; }
    else { h.sp = top; h.ep = bot; h.hits = bot - top; }
    return h;
  }
  u64 ptop = ~0ull, pbot = ~0ull;
  SymbolStream ss(rp, off + 16, lo, hi, bad);
  for (; m < cur; ++m) {
    ptop = top; pbot = bot;
    if (bot - top == 1) break;
    const int c = ss.at(off + m);
    if (c > 2) { bot = top; break; }
    n_occ += lf_pair(ix, top, bot, c);
    if (bot <= top) break;
  }
  h.mlen = m;
  if (bot <= top) { h.sp = ptop; h.ep = pbot; } else { h.sp = top; h.ep = bot; }
  h.hits = h.ep - h.sp;
  return h;
}

// count_hash_table (bwt.h:1848-1952): exact interval of read[off .. off+cur).
// Once a single row is left the remaining LF steps can only keep that row or empty the interval, i.e. they compare
// the rest of the pattern with the text to the left of that one suffix.  So the row is located and the rest of
// the read is compared with the (C->T converted) double-strand sequence 32 bases at a time -- the same hits
// (1 or 0) and, via site = 2N - SA - len - off with SA(final) = SA(row) - (cur - m), the same site, without a
// chain of up to L dependent occ lookups.  hits >= 2 leave the interval in [sp, ep) for the locate kernel.
__device__ __forceinline__ u64 count_exact(const DevIndex& ix, const ReadPlanes& rp, const unsigned char* lut, u32 off, u32 cur, u64& sp, u64& ep,
                                           bool& have_site, u64& site, u32& n_occ, u32& n_hash, u32& n_rows, u32& n_llf) {
  have_site = false;
  u32 m = 0, lo = 0, hi = 0, bad = 0; u64 top = 0, bot = 0; bool one_sa = false;   // initialised: else seed_reseed takes 71 registers, not 64
  if (seed_start(ix, rp, lut, off, cur, true, m, top, bot, one_sa, lo, hi, bad, n_hash) == START_NONE) return 0;
  const u64 sa_known = top;                           // one_sa: the SA value of the single row
  SymbolStream ss(rp, off + 16, lo, hi, bad);
  for (; m < cur; ++m) {
    if (bot <= top) break;
    if (bot - top == 1) {
      int s = 0; const u64 sa = one_sa ? sa_known : locate_row(ix, top, s); n_llf += s; ++n_rows;
      const u64 s0 = 2 * ix.N - sa - m;                 // double-strand coordinate of read[off]
      if (!exact_tail_matches(ix, rp, s0, off, m, cur)) return 0;
      have_site = true; site = s0 - off;
      return 1;
    }
    const int c = ss.at(off + m);
    if (c > 2) return 0;
    n_occ += lf_pair(ix, top, bot, c);
  }
  if (one_sa) {                                       // the pattern ends exactly where the table entry stands
    const u64 s0 = 2 * ix.N - sa_known - m;
    have_site = true; site = s0 - off;
    return 1;
  }
  sp = top; ep = bot;
  return bot <= top ? 0 : bot - top;
}

// determine_seed_offset_unmatch, Schema.h:1506-1531 (step 8): skip past an N inside the next 8 bases
__device__ __forceinline__ u32 next_offset_unmatched(const ReadPlanes& rp, u32 L, u32 off) {
  if ((int)L - (int)off < 18) return L;
  const uint4 a = rp.chunk(off >> 5), c = rp.chunk((off >> 5) + 1);
  const u32 n8 = __funnelshift_r(a.w, c.w, off & 31u) & 0xFFu;
  return n8 ? off + (u32)__ffs(n8) : off + 8;
}

// Direct compare of read[from .. L) with the genome at `site` (try_process_unique_mismatch_end_to_end_*,
// Schema.cpp:15430-15478): read T may face reference C; stops at the second error.  32 bases per step on bit-planes.
__device__ __forceinline__ int compare_rest(const DevIndex& ix, const ReadPlanes& rp, u64 site, u32 L, u32& mlen) {
  int errors = 0;
  const bool inside = window_inside(ix, site, L);
  const u32 from = mlen;
  for (u32 c0 = from & ~31u; c0 < L; c0 += 32) {
    const uint4 r = rp.chunk(c0 >> 5);
    u32 mism;
    if (inside) {
      const u64 g = site + c0;
      const uint2 w0 = __ldg(ix.planes + (g >> 5)), w1 = __ldg(ix.planes + (g >> 5) + 1);
      const unsigned sh = (unsigned)g & 31u;
      const u32 glo = __funnelshift_r(w0.x, w1.x, sh), ghi = __funnelshift_r(w0.y, w1.y, sh);
      mism = (((r.x ^ glo) | (r.y ^ ghi)) & ~(r.x & r.y & glo & ~ghi)) | r.z;
    } else mism = 0xFFFFFFFFu;
    if (c0 < from) mism &= ~0u << (from - c0);
    if (L - c0 < 32u) mism &= (1u << (L - c0)) - 1u;
    if (mism) {
      if (errors == 0) { mlen = c0 + (u32)__ffs(mism) - 1u; errors = 1; mism &= mism - 1u; }
      if (mism) { errors = 2; break; }
    }
  }
  return errors;
}

// ---- what the seeding kernels (seed_reads, seed_reseed) share: work counters, the key table, list appends (sens_pair's
// too), the task records of a read
struct SeedCounters { u32 n_occ = 0, n_hash = 0, n_rows = 0, n_llf = 0; };

__device__ __forceinline__ void build_key_lut(unsigned char* lut) {
  for (u32 i = threadIdx.x; i < 256; i += blockDim.x) {     // i = fm bit0 of 4 bases | fm bit1 << 4
    u32 v = 0, p3 = 1;
    for (u32 t = 0; t < 4; ++t) { v += p3 * (((i >> t) & 1u) | (((i >> (4 + t)) & 1u) << 1)); p3 *= 3; }
    lut[i] = (unsigned char)v;
  }
}

__device__ __forceinline__ void flush_counters(u64* s_cnt, const SeedCounters& c, u64* counters) {
  atomicAdd(&s_cnt[0], (u64)c.n_hash); atomicAdd(&s_cnt[1], (u64)c.n_occ); atomicAdd(&s_cnt[2], (u64)c.n_rows); atomicAdd(&s_cnt[3], (u64)c.n_llf);
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(counters + CNT_HASH, s_cnt[0]); atomicAdd(counters + CNT_OCC, s_cnt[1]);
    atomicAdd(counters + CNT_ROWS, s_cnt[2]); atomicAdd(counters + CNT_LOCATE_LF, s_cnt[3]);
  }
}

// warp-aggregated append of read r to a list (order is irrelevant: results are indexed by read); the count is a u32 or, for
// the finishing lists, an unsigned long long of FinCounters
template <class C>
__device__ __forceinline__ void list_append(u32* list, C* count, bool pred, u32 r) {
  const u32 active = __activemask();
  const u32 m = __ballot_sync(active, pred);
  if (!m) return;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  u32 base = 0;
  if (lane == leader) base = (u32)atomicAdd(count, (C)__popc(m));
  base = __shfl_sync(active, base, leader);
  if (pred) list[base + __popc(m & ((1u << lane) - 1u))] = r;
}

// the seed tasks of read r: the first MAX_TASKS are stored; nt counts them all and nc their candidates, so that store() can
// mark an overflow (ncand = 0xFFFFFFFF).  nt and nc are references: seed_reads keeps them in shared memory.
struct TaskWriter {
  const BatchView& b; const u32& r; u32& nt; u32& nc;
  __device__ __forceinline__ void emit(u64 a, u32 hits, u32 mlen, u32 o) {
    if (nt < MAX_TASKS) { SeedTask t; t.sp = a; t.hits = hits; t.mlen = (unsigned short)mlen; t.off = (unsigned short)o; b.tasks[(size_t)nt * b.n_reads + r] = t; }
    ++nt; nc += hits ? hits : 1u;
  }
  __device__ __forceinline__ void store() { b.ntask[r] = nt < MAX_TASKS ? nt : MAX_TASKS; b.ncand[r] = nt <= MAX_TASKS ? nc : 0xFFFFFFFFu; }
};

// ---- seeding, one persistent kernel.  Every lane runs the seeding state machine of ONE read (first seed + unique-hit
// shortcut, the one-mismatch second seed, the remaining greedy seeds: Schema.cpp:27151-27515 / :19586-19906) and takes the
// next read from a global cursor when its read is finished, so no lane waits for the warp's longest read.  The machine is
// cut into four kinds of step, each at most one round of dependent memory accesses:
//   REFILL   take a read, stage its bit-plane chunks in shared memory
//   START    start a seed: 16-mer key, deep-table / 16-mer-table lookup
//   LF       one backward-extension step of the seed in progress (greedy or exact)
//   COMPARE  a single row is left: locate it and compare the rest of the read with the genome directly
//   DONE     a seed has its answer: the policy of the read's phase (which seeds count, where the next one starts), task records
// The two that happen between seeds (DONE, then REFILL or START) are run back to back as one TRANSITION, and in every
// iteration the WARP VOTES for what most of its lanes are waiting for -- TRANSITION, LF or COMPARE -- and executes only that
// (letting the LF lanes pile up before they run, with hysteresis thresholds, measured slower: 2.1-2.7 ms against 1.86 ms).  A
// loop nest per read or a loop that runs every kind each iteration keeps 4-6 of 32 lanes busy on a repeat-rich genome: the
// rare long paths are executed for one or two lanes while the others wait.  Decisions and their order per read are the
// reference's: the first seed and its unique-hit shortcut (Schema.cpp:27151-27330, try_process_unique_mismatch_end_to_end_*
// :15410-15478), the one-mismatch second seed (:27334-27401), the remaining greedy seeds (:27434-27515).
enum { SK_FIRST = 0, SK_SECOND = 1, SK_REST = 2 };
enum { PH_IDLE = 0, PH_REFILL = 1, PH_START = 2, PH_LF = 3, PH_COMPARE = 4, PH_DONE = 5 };

__global__ void __launch_bounds__(128) seed_reads(DevIndex ix, BatchView b, u32 plane_cap) {
  extern __shared__ uint4 s_planes[];      // [plane_cap][SEED_BLOCK] staged read chunks, one column per lane
  __shared__ u64 s_cnt[4];
  __shared__ unsigned char s_lut[256];
  if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
  build_key_lut(s_lut);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const u32 n_reads = (u32)b.n_reads;
  SeedCounters cn;
  ReadPlanes rp; rp.p = nullptr; rp.s = s_planes + threadIdx.x; rp.ns = 0;
  int ph = PH_REFILL;
  // What a step of the seed in progress needs stays in registers; the per-read bookkeeping that only the transitions between
  // seeds touch lives in shared memory, one column per lane (registers decide how many warps an SM holds, and the kernel
  // lives on warps in flight).
  __shared__ u32 s_w[21][SEED_BLOCK];
  __shared__ u64 s_d[4][SEED_BLOCK];
  const int tx = threadIdx.x;
  u32 &r = s_w[0][tx], &L = s_w[1][tx], &first_c = s_w[2][tx], &off = s_w[3][tx], &first_len = s_w[4][tx], &max_seeds = s_w[5][tx], &seed_id = s_w[6][tx];
  u32 &nt = s_w[7][tx], &nc = s_w[8][tx], &bn = s_w[9][tx], &bs0 = s_w[10][tx], &bs1 = s_w[11][tx], &bep = s_w[12][tx], &bel = s_w[13][tx];
  u32 &first_cands = s_w[14][tx], &g_mlen = s_w[15][tx], &is_multi = s_w[16][tx], &second_ok = s_w[17][tx];
  int &state = reinterpret_cast<int&>(s_w[18][tx]), &get_error = reinterpret_cast<int&>(s_w[19][tx]), &one_mm = reinterpret_cast<int&>(s_w[20][tx]);
  u64 &sp = s_d[0][tx], &ep = s_d[1][tx], &site0 = s_d[2][tx], &g_hits = s_d[3][tx];   // g_hits, g_mlen: answer of the first seed, kept across its COMPARE step
  u32 kind = SK_FIRST;
  u32 s_off = 0, s_cur = 0, m = 0;                       // the seed in progress: start, bases available, symbols matched
  u64 top = 0, bot = 0, ptop = 0, pbot = 0, sa_known = 0;
  bool known_sa = false;
  u32 ss_base = 0, ss_lo = 0, ss_hi = 0, ss_bad = 0;     // 32 symbols of the read from ss_base on
  TaskWriter tw{b, r, nt, nc};
  auto symbol_at = [&](u32 pos) -> int {                 // pos >= ss_base, non-decreasing within a seed
    if (pos - ss_base >= 32u) { ss_base = pos; rp.window(pos, ss_lo, ss_hi, ss_bad); }
    const unsigned sh = pos - ss_base;
    const u32 l = (ss_lo >> sh) & 1u, h = (ss_hi >> sh) & 1u, bad = (ss_bad >> sh) & 1u;
    return (int)((l | ((~(l | h) & 1u) << 1)) | (bad * 3u));
  };
  // the read is done: its records
  auto finish = [&]() {
    b.state[r] = (unsigned char)state;
    b.flags[r] = (unsigned char)((is_multi ? 1 : 0) | (second_ok ? 2 : 0));
    b.one_mm[r] = (short)one_mm;
    b.site0[r] = site0;
    tw.store();
    if (b.sensitive) {
      const bool resolved = state == BMBS_EXACT_UNIQUE || state == BMBS_MULTI_EXACT;
      unsigned short* k5 = b.bk + (size_t)r * 5;
      k5[0] = (unsigned short)(resolved ? 0 : bn); k5[1] = (unsigned short)bs0; k5[2] = (unsigned short)bs1; k5[3] = (unsigned short)bep;
      k5[4] = (unsigned short)(resolved ? 0 : bel);
      b.first_cands[r] = (unsigned short)(resolved ? 0 : first_cands);
    }
    ph = PH_REFILL;
  };
  // next seed of the greedy phase, or the end of the read (loop condition of Schema.cpp:27434)
  auto next_rest = [&]() {
    kind = SK_REST;
    if (seed_id < max_seeds && off < L) { s_off = off; s_cur = L - off; ph = PH_START; } else finish();
  };
  // first seed, after the unique-hit shortcut did not settle the read (Schema.cpp:27203-27330); mlen: the seed length as the
  // shortcut left it (clamped to the first C, or the index of the single mismatch)
  auto first_rest = [&](u32 mlen) {
    one_mm = (int)mlen;
    if (mlen == L && g_hits > 1 && (!b.pe || g_hits <= b.multi_cap)) {
      is_multi = 1;
      if (first_c == L) {
        state = BMBS_MULTI_EXACT;
        if (b.pe) tw.emit(sp, (u32)g_hits, mlen, 0);
        else if (b.amb_out) tw.emit(sp, (u32)(g_hits > MAX_SEED_HITS ? MAX_SEED_HITS : g_hits), mlen, 0);   // output_ambiguous_exact_map_output_buffer walks at most 1000 rows
        finish();
        return;
      }
    }
    if (g_hits != 1 && mlen >= b.seed_len && g_hits <= MAX_SEED_HITS && g_hits != 0) tw.emit(sp, (u32)g_hits, mlen, 0);
    const bool used = g_hits == 1 || (g_mlen >= b.seed_len && g_hits <= MAX_SEED_HITS);
    bn = used ? 1 : 0; bel = used ? first_len : 0; first_cands = nc;
    off = mlen == 0 ? next_offset_unmatched(rp, L, 0) : mlen / 2;
    seed_id = 1;
    if (get_error == 1 && L - first_len >= 17) { kind = SK_SECOND; s_off = first_len; s_cur = L - first_len; ph = PH_START; }   // one-mismatch rule
    else next_rest();
  };
  // the second seed has its answer (Schema.cpp:27334-27401): known_sa = its single site is in sa_known, else rows [top, bot)
  auto second_done = [&]() {
    const u64 hits = known_sa ? 1 : (bot > top ? bot - top : 0);
    if (hits <= MAX_SEED_HITS) {
      if (known_sa) tw.emit(sa_known, 0, 0, 0); else if (hits) tw.emit(top, (u32)hits, s_cur, s_off);
      second_ok = 1; finish();
    } else next_rest();
  };
  // a greedy seed has its answer: m symbols matched, rows [top, bot) (known_sa: one row whose suffix-array value is sa_known)
  auto greedy_done = [&]() {
    const u64 hits = known_sa ? 1 : bot - top;
    const u32 mlen = m;
    if (!known_sa) { sp = top; ep = bot; }
    if (kind == SK_FIRST) {
      g_hits = hits; g_mlen = mlen; first_len = mlen;
      if (hits == 1) ph = PH_COMPARE;                                            // unique-hit shortcut: locate + direct compare
      else first_rest(mlen);
    } else {                                                                     // Schema.cpp:27434-27515
      bool used = true;
      if (hits == 1) { if (known_sa) tw.emit(2 * ix.N - sa_known - mlen - off, 0, 0, 0); else tw.emit(sp, 1, mlen, off); }
      else if (mlen >= b.seed_len && hits <= MAX_SEED_HITS) { if (hits) tw.emit(sp, (u32)hits, mlen, off); }
      else { used = false; if (s_cur == mlen) { finish(); return; } }
      if (used) { if (bn == 0) bs0 = off; else if (bn == 1) bs1 = off; bep = bel; bel = off + mlen; ++bn; }
      off = mlen == 0 ? next_offset_unmatched(rp, L, off) : off + mlen / 2;
      ++seed_id;
      next_rest();
    }
  };
  for (;;) {
    const u32 m_lf = __ballot_sync(0xffffffffu, ph == PH_LF), m_cmp = __ballot_sync(0xffffffffu, ph == PH_COMPARE);
    const u32 m_tr = __ballot_sync(0xffffffffu, ph == PH_DONE || ph == PH_START || ph == PH_REFILL);
    if (!(m_lf | m_cmp | m_tr)) break;
    const int c_lf = __popc(m_lf), c_cmp = __popc(m_cmp), c_tr = __popc(m_tr);
    const bool do_tr = c_tr >= c_lf && c_tr >= c_cmp, do_lf = !do_tr && c_lf >= c_cmp;
    if (do_tr) {
      // ---- a seed has its answer: the policy of the read's phase
      if (ph == PH_DONE) { if (kind == SK_SECOND) second_done(); else greedy_done(); }
      const u32 m_refill = __ballot_sync(0xffffffffu, ph == PH_REFILL);
      const int c_refill = __popc(m_refill);
      // ---- lanes without a read take the next ones (one atomic per warp)
      if (m_refill) {
      u32 base = 0;
      const int leader = __ffs(m_refill) - 1;
      if (lane == leader) base = atomicAdd(b.list_count, (u32)c_refill);
      base = __shfl_sync(0xffffffffu, base, leader);
      if (ph == PH_REFILL) {
        const u32 i = base + __popc(m_refill & ((1u << lane) - 1u));
        if (i >= n_reads) ph = PH_IDLE;
        else {
          r = i;
          L = b.len[r]; first_c = b.first_c[r];
          rp.stage(b.rplanes + plane_chunk_offset(b.offsets, (int)r), L, s_planes + threadIdx.x, plane_cap);
          { u64 ms = (u64)L / 10 - 1; if (ms > 25) ms = 25; max_seeds = (u32)ms; }   // u64 wrap for L < 10, as in the reference
          nt = 0; nc = 0; off = 0; first_len = 0; seed_id = 0; sp = 0; ep = 0; site0 = 0;
          state = BMBS_NONE; get_error = -1; one_mm = 0; is_multi = 0; second_ok = 0;
          bn = 0; bs0 = 0; bs1 = 0; bep = 0; bel = 0; first_cands = 0;
          if (max_seeds > 0 && L > 0) { kind = SK_FIRST; s_off = 0; s_cur = L; ph = PH_START; }
          else finish();                                                     // no seed at all
        }
      }
      }
      if (ph == PH_START) {
        // ---- start of a seed: key, table lookup (count_backward_as_much_1_terminate bwt.h:2081 / count_hash_table :1848)
        const int how = seed_start(ix, rp, s_lut, s_off, s_cur, kind == SK_SECOND, m, top, bot, known_sa, ss_lo, ss_hi, ss_bad, cn.n_hash);
        ss_base = s_off + 16; sa_known = top;                  // sa_known is read only when known_sa
        if (how == START_LF) { ph = PH_LF; ptop = ~0ull; pbot = ~0ull; }
        else ph = PH_DONE;
      }
    } else if (do_lf) {
      if (ph == PH_LF) {
        if (kind != SK_SECOND) {
          // ---- one step of count_backward_as_much_1_terminate's loop (bwt.h:2081-2209)
          bool stop = true;
          if (m < s_cur) {
            ptop = top; pbot = bot;
            const int c = symbol_at(s_off + m);
            if (bot - top != 1) {
              if (c > 2) bot = top;
              else {
                cn.n_occ += lf_pair(ix, top, bot, c);
                if (bot > top) { ++m; stop = m >= s_cur; }
              }
            }
          }
          if (stop) { if (bot <= top) { top = ptop; bot = pbot; } ph = PH_DONE; }
        } else {
          // ---- one step of count_hash_table's loop (bwt.h:1848-1952); a single row left is located and compared directly
          if (m < s_cur && bot > top) {
            if (bot - top == 1) ph = PH_COMPARE;
            else {
              const int c = symbol_at(s_off + m);
              if (c > 2) { bot = top; ph = PH_DONE; }
              else { cn.n_occ += lf_pair(ix, top, bot, c); ++m; }
            }
          } else {
            if (known_sa) sa_known = 2 * ix.N - sa_known - m - s_off;   // the pattern ends where the table entry stands: its site
            ph = PH_DONE;
          }
        }
      }
    } else {
      if (ph == PH_COMPARE) {
        if (kind == SK_FIRST) {
          // ---- unique first seed: locate, compare the rest of the read with the genome (try_process_unique_mismatch_end_to_end_*, Schema.cpp:15410)
          int st = 0; const u64 sa = known_sa ? sa_known : locate_row(ix, sp, st); cn.n_llf += st; ++cn.n_rows;
          u32 mlen = g_mlen;
          const u64 site = 2 * ix.N - sa - mlen;
          tw.emit(site, 0, 0, 0);
          if (mlen > first_c) mlen = first_c;
          int errors = 0;
          if (mlen != L) errors = compare_rest(ix, rp, site, L, mlen);
          get_error = errors;
          if (errors == 0) { state = BMBS_EXACT_UNIQUE; site0 = site; finish(); }
          else first_rest(mlen);
        } else {
          // ---- exact seed with one row left: the remaining symbols can only keep that row or empty the interval
          int st = 0; const u64 sa = known_sa ? sa_known : locate_row(ix, top, st); cn.n_llf += st; ++cn.n_rows;
          const u64 s0 = 2 * ix.N - sa - m;                 // double-strand coordinate of read[s_off]
          known_sa = exact_tail_matches(ix, rp, s0, s_off, m, s_cur); sa_known = s0 - s_off;   // the site, or no hit
          if (!known_sa) bot = top;
          ph = PH_DONE;
        }
      }
    }
  }
  flush_counters(s_cnt, cn, b.counters);
}

// ------------------------------------------------------------------------------------------- expand + locate
// Seed tasks -> candidate sites, one kernel.  A warp owns 32 consecutive reads, i.e. one contiguous range of candidate
// slots [coff[r0], coff[r0+32]).  Its lanes first lay the reads' tasks out as a table of segments {first slot, first row or
// literal site, seed length + offset, owner} in shared memory (in slot order), then walk the slot range with consecutive
// lanes on consecutive slots: a binary search over the segment starts finds a slot's task, the row is located (one gather
// from the dense suffix array) and turned into a site, and cand[] / slot_read[] are written coalesced.
//   site = 2N - SA - seed_len - seed_off, modulo 2^64 (reverse_and_adjust_site, Schema.cpp:4657-4683)
constexpr int SEG_CAP = 256;                      // segments per warp and pass; a read has at most MAX_TASKS = 28
struct Seg { u64 sp; u32 start; u32 info; };      // info: seed_len + seed_off | literal site << 31

__global__ void __launch_bounds__(128) expand_locate(DevIndex ix, BatchView b) {
  __shared__ Seg s_seg[4][SEG_CAP];
  __shared__ u64 s_cnt[2];
  if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  Seg* seg = s_seg[threadIdx.x >> 5];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = !*b.status, live = ok && r < b.n_reads;
  const u32 nt = live ? b.ntask[r] : 0u;
  // lanes past the last read own the empty range at the end, so that a pass's slot range is [c0 of its first lane, c1 of its last)
  const u32 c0 = ok ? b.coff[min(r, b.n_reads)] : 0u, c1 = ok ? b.coff[min(r + 1, b.n_reads)] : 0u;
  u32 incl = nt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  const u32 excl = incl - nt;
  u64 steps = 0, rows = 0;
  int lo_lane = 0;
  while (lo_lane < 32) {
    // lanes [lo_lane, hi_lane) whose tasks fit into the table together (incl is monotonic, so they are contiguous)
    const u32 base = __shfl_sync(0xffffffffu, excl, lo_lane);
    const bool fits = lane >= lo_lane && incl - base <= (u32)SEG_CAP;
    const int hi_lane = lo_lane + __popc(__ballot_sync(0xffffffffu, fits));
    if (fits) {
      u32 s = c0;
      for (u32 t = 0; t < nt; ++t) {
        const SeedTask k = b.tasks[(size_t)t * b.n_reads + r];
        Seg g; g.sp = k.sp; g.start = s;
        g.info = k.hits ? (u32)k.mlen + (u32)k.off : 0x80000000u;
        seg[excl - base + t] = g;
        s += k.hits ? k.hits : 1u;
      }
    }
    __syncwarp();
    const u32 n_seg = __shfl_sync(0xffffffffu, incl, hi_lane - 1) - base;
    const u32 s_begin = __shfl_sync(0xffffffffu, c0, lo_lane), s_end = __shfl_sync(0xffffffffu, c1, hi_lane - 1);
    if (n_seg) {
      for (u32 s = s_begin + lane; s < s_end; s += 32) {
        u32 lo = 0, hi = n_seg;                              // seg[lo].start <= s < seg[hi].start
        while (hi - lo > 1) { const u32 mid = (lo + hi) >> 1; if (seg[mid].start <= s) lo = mid; else hi = mid; }
        const Seg g = seg[lo];
        u64 site = g.sp;
        if (!(g.info >> 31)) {
          int st; const u64 sa = locate_row(ix, g.sp + (u64)(s - g.start), st);
          site = 2 * ix.N - sa - (u64)(g.info & 0xFFFFu); ++rows; steps += st;
        }
        b.cand[s] = site;
      }
    }
    __syncwarp();
    lo_lane = hi_lane;
  }
  atomicAdd(&s_cnt[0], rows); atomicAdd(&s_cnt[1], steps);
  __syncthreads();
  if (threadIdx.x == 0) { atomicAdd(b.counters + CNT_ROWS, s_cnt[0]); atomicAdd(b.counters + CNT_LOCATE_LF, s_cnt[1]); }
}

// ------------------------------------------------------------------------------------------- votes
// What a read's candidates turn into (Schema.cpp:27527-27612, :19885-19915):
//   conclusive second seed with a single distinct candidate -> ONE_MISMATCH;
//   otherwise sort + run-length encode into windows {max(c-k,0), votes}  (generate_candidate_votes_shift, :4687-4773).
// Returns true when the segment still has to be sorted/encoded.
__device__ __forceinline__ bool classify_read(BatchView& b, int r, u32 beg, u32 n, bool lane0) {
  if (b.round == 1) { if (n == 0) { if (lane0) b.nv[r] = 0; return false; } return true; }   // re-seeded mates: always sort + encode
  const int st = b.state[r];
  if (st == BMBS_EXACT_UNIQUE) { if (lane0) { b.nv[r] = b.pe ? 1u : 0u; if (n) b.vcnt[beg] = 0; } return false; }
  if (st == BMBS_MULTI_EXACT) {
    if (!b.pe) {      // single end: nothing to verify; with --ambiguous_out the located rows stay as they are (row order)
      if (lane0) { const u32 keep = b.amb_out ? n : 0u; for (u32 i = 0; i < keep; ++i) b.vcnt[beg + i] = 0; b.nv[r] = keep; }
      return false;
    }
    return true;
  }
  if (n == 0) { if (lane0) b.nv[r] = 0; return false; }
  if ((b.flags[r] & 2) && (n == 1 || (n == 2 && b.cand[beg] == b.cand[beg + 1]))) {
    if (lane0) { b.state[r] = BMBS_ONE_MISMATCH; b.site0[r] = b.cand[beg]; b.nv[r] = b.pe ? 1u : 0u; b.vcnt[beg] = 0; }
    return false;
  }
  if (lane0) b.state[r] = BMBS_VERIFY;
  return true;
}

__device__ __forceinline__ u64 window_start(u64 c, u64 k) { return c < k ? 0ull : c - k; }

// Sorting network over N registers (bitonic; every index is a compile-time constant after unrolling), ascending.
template <int N>
__device__ __forceinline__ void sort_regs(u64 (&v)[N]) {
#pragma unroll
  for (int k = 2; k <= N; k <<= 1)
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1)
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const int l = i ^ j;
        if (l > i) {
          const u64 a = v[i], c = v[l];
          const bool sw = ((i & k) == 0) ? (a > c) : (a < c);
          v[i] = sw ? c : a; v[l] = sw ? a : c;
        }
      }
}

// sort + run-length encode a segment of n <= N candidates held by one thread, in place (generate_candidate_votes_shift,
// Schema.cpp:4687-4773: equal sites merge into {max(site - k, 0), votes}; distinct small sites that clamp to 0 stay apart)
template <int N>
__device__ __forceinline__ void sort_encode_small(BatchView& b, int r, u32 beg, u32 n, bool live, bool multi) {
  u64 v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = (live && (u32)i < n) ? b.cand[beg + i] : ~0ull;   // padding ~0 sorts last (a real ~0 is equal to it)
  sort_regs<N>(v);
  if (!live) return;
  if (multi) {
#pragma unroll
    for (int i = 0; i < N; ++i) if ((u32)i < n) { b.cand[beg + i] = v[i]; b.vcnt[beg + i] = 0; }
    b.nv[r] = n;
    return;
  }
  const u64 k = b.kk[r];
  u32 out = 0, run = 0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if ((u32)i < n) {
      ++run;
      const bool last = (u32)(i + 1) == n || (i + 1 < N && v[i + 1] != v[i]);
      if (last) { b.cand[beg + out] = window_start(v[i], k); b.vcnt[beg + out] = run; ++out; run = 0; }
    }
  }
  b.nv[r] = out;
}

// One thread per read decides what the candidates turn into and, for the usual short segment (<= 16 candidates), sorts and
// encodes it on the spot with a sorting network in registers (8 wide when the whole warp fits); longer segments go to the
// warp kernel (<= 32) or the CTA kernel.
__global__ void __launch_bounds__(128) votes_classify(BatchView b) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  int which = -1; u32 beg = 0, n = 0;
  if (r < b.n_reads && !*b.status) {
    beg = b.coff[r]; n = b.coff[r + 1] - beg;
    if (classify_read(b, r, beg, n, true)) which = n <= 16 ? 0 : n <= 32 ? 1 : n <= 256 ? 2 : n <= 1024 ? 3 : 4;
  }
  const bool small = which == 0;
  if (__any_sync(0xffffffffu, small)) {
    const bool multi = small && b.round == 0 && b.state[r] == BMBS_MULTI_EXACT;
    if (__all_sync(0xffffffffu, !small || n <= 8)) sort_encode_small<8>(b, r, beg, n, small, multi);
    else sort_encode_small<16>(b, r, beg, n, small, multi);
  }
  list_append(b.sort32, b.sort_count + 1, which == 1, (u32)r);
  list_append(b.mid_list, b.sort_count + 2, which == 2, (u32)r);
  list_append(b.big1k_list, b.sort_count + 3, which == 3, (u32)r);
  list_append(b.big_list, b.big_count, which == 4, (u32)r);
}

// W lanes per read (32; segments up to 16 are sorted by their own thread in votes_classify): bitonic sort in registers over shuffles, run-length encode with a ballot, written back in
// place.  Padding is ~0: a real candidate equal to it sorts next to the padding, so the first n entries are still right.
template <int W>
__global__ void __launch_bounds__(128) votes_sort(BatchView b) {
  const u32 nlist = *b.status ? 0u : b.sort_count[1];
  const u32* list = b.sort32;
  const int lane = threadIdx.x & 31, sub = lane & (W - 1), half_shift = lane & ~(W - 1);
  const u32 groups = gridDim.x * blockDim.x / W;
  for (u32 g0 = 0; g0 < nlist; g0 += groups) {
    const u32 g = g0 + (blockIdx.x * blockDim.x + threadIdx.x) / W;
    const bool live = g < nlist;
    int r = 0; u32 beg = 0, n = 0;
    if (live) { r = (int)list[g]; beg = b.coff[r]; n = b.coff[r + 1] - beg; }
    u64 v = sub < (int)n ? b.cand[beg + sub] : ~0ull;
#pragma unroll
    for (int k = 2; k <= W; k <<= 1)
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        const u64 o = __shfl_xor_sync(0xffffffffu, v, j);
        const bool take_min = ((sub & k) == 0) == ((sub & j) == 0);
        v = take_min ? (o < v ? o : v) : (o > v ? o : v);
      }
    const bool multi = live && b.round == 0 && b.state[r] == BMBS_MULTI_EXACT;
    const u64 prev = __shfl_up_sync(0xffffffffu, v, 1);
    const bool head = live && !multi && sub < (int)n && (sub == 0 || prev != v);
    const u32 heads = (__ballot_sync(0xffffffffu, head) >> half_shift) & (W == 32 ? 0xffffffffu : 0xffffu);
    if (multi) { if (sub < (int)n) { b.cand[beg + sub] = v; b.vcnt[beg + sub] = 0; } if (sub == 0) b.nv[r] = n; }
    else if (live) {
      if (head) {
        const u32 idx = __popc(heads & ((1u << sub) - 1u));
        const u32 later = heads & ~((2u << sub) - 1u);       // run length = distance to the next head (or to n)
        const u32 next = later ? (u32)(__ffs(later) - 1) : n;
        b.cand[beg + idx] = window_start(v, (u64)b.kk[r]);
        b.vcnt[beg + idx] = next - sub;
      }
      if (sub == 0) b.nv[r] = __popc(heads);
    }
  }
}

// ---- segments of 33..1024 candidates: bitonic sort with E consecutive keys per thread in registers.  Element e = tid * E + i.
// A compare-exchange stage with partner distance j < E stays inside the thread (compile-time register indices), E <= j < 32 E
// is one shuffle per key inside the warp, and only j >= 32 E (CTA form, two warps or more) goes through shared memory -- three
// exchanges for 1024 keys where a plain shared-memory network needs 55 block-wide barriers.  Padding is ~0 (sorts last).
template <int E, int T>
__device__ __forceinline__ void bitonic_regs(u64 (&v)[E], const int tid, u64* xch) {
#pragma unroll
  for (int k = 2; k <= E * T; k <<= 1) {
    const bool up = ((tid * E) & k) == 0;                       // for k < E the direction depends on i: handled below
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32 * E) {                                        // partner in another warp
        __syncthreads();
#pragma unroll
        for (int i = 0; i < E; ++i) xch[i * T + tid] = v[i];
        __syncthreads();
        const int pt = tid ^ (j / E);
        const bool take_min = up == ((tid & (j / E)) == 0);
#pragma unroll
        for (int i = 0; i < E; ++i) { const u64 o = xch[i * T + pt]; v[i] = take_min ? (o < v[i] ? o : v[i]) : (o > v[i] ? o : v[i]); }
      } else if (j >= E) {                                      // partner lane in the same warp
        const bool take_min = up == ((tid & (j / E)) == 0);
#pragma unroll
        for (int i = 0; i < E; ++i) { const u64 o = __shfl_xor_sync(0xffffffffu, v[i], j / E); v[i] = take_min ? (o < v[i] ? o : v[i]) : (o > v[i] ? o : v[i]); }
      } else {                                                  // both keys in this thread
#pragma unroll
        for (int i = 0; i < E; ++i) {
          if ((i & j) == 0) {
            const bool asc = k < E ? ((i & k) == 0) : up;
            const u64 a = v[i], c = v[i | j];
            const bool sw = asc ? (a > c) : (a < c);
            v[i] = sw ? c : a; v[i | j] = sw ? a : c;
          }
        }
      }
    }
  }
}

// run-length encode the sorted keys a[0..n) (shared memory) of read r into cand[] / vcnt[] by the 32 lanes of a warp
__device__ __forceinline__ void warp_encode_runs(BatchView& b, int r, u32 beg, u32 n, const u64* a, int lane) {
  const u64 k = b.kk[r];
  u32 base = 0;
  for (u32 c0 = 0; c0 < n; c0 += 32) {
    const u32 i = c0 + lane;
    const bool head = i < n && (i == 0 || a[i - 1] != a[i]);
    const u32 bal = __ballot_sync(0xffffffffu, head);
    if (head) {
      u32 e = i + 1; while (e < n && a[e] == a[i]) ++e;
      const u32 idx = base + __popc(bal & ((1u << lane) - 1u));
      b.cand[beg + idx] = window_start(a[i], k);                // idx <= i and a[] is a copy: in place is safe
      b.vcnt[beg + idx] = e - i;
    }
    base += __popc(bal);
  }
  if (lane == 0) b.nv[r] = base;
}

// a warp sorts the n <= 32 E keys of a segment (E consecutive keys per lane) and leaves them, ascending, in a[0 .. 32 E)
template <int E>
__device__ __forceinline__ void warp_sort_keys(const u64* __restrict__ src, u32 n, u64* a, int lane) {
  u64 v[E];
#pragma unroll
  for (int i = 0; i < E; ++i) { const u32 e = (u32)lane * E + i; v[i] = e < n ? src[e] : ~0ull; }
  bitonic_regs<E, 32>(v, lane, nullptr);
  __syncwarp();
#pragma unroll
  for (int i = 0; i < E; ++i) a[lane * E + i] = v[i];
  __syncwarp();
}

// one warp per segment of 33..256 candidates: two, four or eight keys per lane -- the network over 64 keys is a seventh of the
// work of the one over 256, and most of these segments are short
__global__ void __launch_bounds__(128) votes_mid(BatchView b) {
  __shared__ u64 s_keys[4][32 * 8];
  const u32 nlist = *b.status ? 0u : b.sort_count[2];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const u32 warps = gridDim.x * (blockDim.x >> 5);
  u64* a = s_keys[wid];
  for (u32 g = blockIdx.x * (blockDim.x >> 5) + wid; g < nlist; g += warps) {
    const int r = (int)b.mid_list[g];
    const u32 beg = b.coff[r], n = b.coff[r + 1] - beg;
    if (n <= 64) warp_sort_keys<2>(b.cand + beg, n, a, lane);
    else if (n <= 128) warp_sort_keys<4>(b.cand + beg, n, a, lane);
    else warp_sort_keys<8>(b.cand + beg, n, a, lane);
    if (b.round == 0 && b.state[r] == BMBS_MULTI_EXACT) {
      for (u32 i = lane; i < n; i += 32) { b.cand[beg + i] = a[i]; b.vcnt[beg + i] = 0; }
      if (lane == 0) b.nv[r] = n;
    } else warp_encode_runs(b, r, beg, n, a, lane);
    __syncwarp();
  }
}

// a CTA of T threads sorts the n <= T E keys of a segment and leaves them, ascending, in keys[0 .. T E)
template <int E, int T>
__device__ __forceinline__ void block_sort_keys(const u64* __restrict__ src, u32 n, u64* keys, int tid) {
  u64 v[E];
#pragma unroll
  for (int i = 0; i < E; ++i) { const u32 e = (u32)tid * E + i; v[i] = e < n ? src[e] : ~0ull; }
  bitonic_regs<E, T>(v, tid, keys);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < E; ++i) keys[tid * E + i] = v[i];
  __syncthreads();
}

// one CTA of 128 threads per segment of 257..1024 candidates (four keys per thread up to 512, eight beyond)
__global__ void __launch_bounds__(128) votes_big1k(BatchView b) {
  constexpr int T = 128;
  __shared__ u64 s_keys[8 * T];
  const u32 nlist = *b.status ? 0u : b.sort_count[3];
  const int tid = threadIdx.x, lane = tid & 31;
  for (u32 g = blockIdx.x; g < nlist; g += gridDim.x) {
    const int r = (int)b.big1k_list[g];
    const u32 beg = b.coff[r], n = b.coff[r + 1] - beg;
    if (n <= 4 * T) block_sort_keys<4, T>(b.cand + beg, n, s_keys, tid);
    else block_sort_keys<8, T>(b.cand + beg, n, s_keys, tid);
    if (b.round == 0 && b.state[r] == BMBS_MULTI_EXACT) {
      for (u32 i = tid; i < n; i += T) { b.cand[beg + i] = s_keys[i]; b.vcnt[beg + i] = 0; }
      if (tid == 0) b.nv[r] = n;
    } else if (tid < 32) warp_encode_runs(b, r, beg, n, s_keys, lane);     // <= 32 passes of a warp; the sort dominates
    __syncthreads();
  }
}

// one CTA per long segment: bitonic sort on a power-of-two padded copy (shared memory when it fits,
// global scratch otherwise), then a block-wide run-length encode.
constexpr int BIG_SMEM_ELEMS = 16384;             // 128 KB of dynamic shared memory: segments of up to 16 k candidates never touch global scratch
constexpr int BIG_THREADS = 512;
// Launched twice: 256 threads and 32 KB for segments that pad to at most 4096 keys (several CTAs per SM), 512 threads and
// 128 KB for the longer ones; a CTA skips the segments of the other launch.  cap = keys that fit its shared memory.
__global__ void __launch_bounds__(BIG_THREADS) votes_big(BatchView b, u32 cap, u32 min_p, u32 max_p) {
  extern __shared__ u64 s_buf[];                  // [cap]
  __shared__ u32 s_warp[BIG_THREADS / 32];
  __shared__ u32 s_base, s_soff;
  const u32 nbig = *b.status ? 0u : *b.big_count;
  for (u32 bi = blockIdx.x; bi < nbig; bi += gridDim.x) {
    const int r = (int)b.big_list[bi];
    const u32 beg = b.coff[r], n = b.coff[r + 1] - beg;
    u32 P = 64; while (P < n) P <<= 1;
    if (P < min_p || P > max_p) continue;
    u64* a = s_buf;
    if (P > cap) {
      if (threadIdx.x == 0) s_soff = atomicAdd(b.scratch_used, P);
      __syncthreads();
      if ((u64)s_soff + P > b.scratch_cap) { if (threadIdx.x == 0) { b.nv[r] = 0; atomicOr(b.status, 8u); } __syncthreads(); continue; }
      a = b.scratch + s_soff;
    }
    for (u32 i = threadIdx.x; i < P; i += blockDim.x) a[i] = i < n ? b.cand[beg + i] : ~0ull;
    __syncthreads();
    for (u32 k = 2; k <= P; k <<= 1)
      for (u32 j = k >> 1; j > 0; j >>= 1) {
        for (u32 i = threadIdx.x; i < P; i += blockDim.x) {
          const u32 x = i ^ j;
          if (x > i) {
            const u64 vi = a[i], vx = a[x];
            const bool up = (i & k) == 0;
            if (up ? vi > vx : vi < vx) { a[i] = vx; a[x] = vi; }
          }
        }
        __syncthreads();
      }
    // a real key equal to ~0 is indistinguishable from padding but also equal to it, so the first n entries are right
    if (b.round == 0 && b.state[r] == BMBS_MULTI_EXACT) {
      for (u32 i = threadIdx.x; i < n; i += blockDim.x) { b.cand[beg + i] = a[i]; b.vcnt[beg + i] = 0; }
      if (threadIdx.x == 0) b.nv[r] = n;
      __syncthreads();
      continue;
    }
    const u64 k = b.kk[r];
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (u32 c0 = 0; c0 < n; c0 += blockDim.x) {
      const u32 i = c0 + threadIdx.x;
      const bool head = i < n && (i == 0 || a[i - 1] != a[i]);
      const u32 bal = __ballot_sync(0xffffffffu, head);
      const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
      if (lane == 0) s_warp[wid] = __popc(bal);
      __syncthreads();
      u32 before = 0, total = 0;
      for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) { if (w2 < wid) before += s_warp[w2]; total += s_warp[w2]; }
      if (head) {
        u32 e = i + 1; while (e < n && a[e] == a[i]) ++e;      // run length
        const u32 idx = s_base + before + __popc(bal & ((1u << lane) - 1u));
        b.cand[beg + idx] = window_start(a[i], k);             // idx <= i and a[] is a copy: in place is safe
        b.vcnt[beg + idx] = e - i;
      }
      __syncthreads();
      if (threadIdx.x == 0) s_base += total;
      __syncthreads();
    }
    if (threadIdx.x == 0) b.nv[r] = s_base;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------- pair filter
// The pair rules every pair walk shares.  Is b within [dmin, dmax] of a?  `first` skips entries (index j) that are too far
// below a; stop: b is too far above a, and so is every later entry of an ascending list (Schema.cpp:15800-15840).
__device__ __forceinline__ bool in_range(u64 a, u64 b, int dmax, int dmin, long long j, long long& first, bool& stop) {
  stop = false;
  if (a > b) { const long long d = (long long)(a - b); if (d > dmax) { first = j + 1; return false; } return d >= dmin; }
  const long long d = (long long)(b - a);
  if (d > dmax) { stop = true; return false; }
  return d >= dmin;
}

// the distance bounds of pair (r1, r2): dmax_base + 2k and dmin_base - 2k - L, with k and L the larger of the two mates'
__device__ __forceinline__ void pair_bounds(const BatchView& b, int r1, int r2, int& dmax, int& dmin) {
  const u64 k1 = b.kk[r1], k2 = b.kk[r2], kl = k1 > k2 ? k1 : k2;
  const u32 L1 = b.len[r1], L2 = b.len[r2];
  dmax = (int)((u64)(long long)b.dmax_base + kl * 2);
  dmin = (int)((u64)(long long)b.dmin_base - kl * 2 - (u64)(L1 > L2 ? L1 : L2));
}

// seeding resolved this read: its record is final, its windows are not verified
__device__ __forceinline__ bool is_resolved(int st) { return st == BMBS_EXACT_UNIQUE || st == BMBS_MULTI_EXACT || st == BMBS_ONE_MISMATCH; }

// filter_pairs, Schema.cpp:16052-16180, one thread per pair, literal two-pointer walk.
__global__ void filter_pairs_kernel(BatchView b) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p * 2 + 1 >= b.n_reads || *b.status) return;
  const int r1 = 2 * p, r2 = r1 + 1;
  const bool res1 = is_resolved(b.state[r1]), res2 = is_resolved(b.state[r2]);
  u32 n1 = b.nv[r1], n2 = b.nv[r2];
  if (res1 && res2) return;
  if (n1 == 0 || n2 == 0) { b.nv[r1] = 0; b.nv[r2] = 0; return; }
  const u32 b1 = b.coff[r1], b2 = b.coff[r2];
  int dmax, dmin; pair_bounds(b, r1, r2, dmax, dmin);
  for (u32 i = 0; i < n1; ++i) b.keep[b1 + i] = 0;
  for (u32 j = 0; j < n2; ++j) b.keep[b2 + j] = 0;
  long long first = 0;
  bool any1 = false, any2 = false; u64 last1 = 0, last2 = 0;
  for (long long i = 0; i < (long long)n1; ++i) {
    const u64 a = b.cand[b1 + i];
    for (long long j = first; j < (long long)n2; ++j) {
      const u64 c = b.cand[b2 + j];
      bool stop; const bool in = in_range(a, c, dmax, dmin, j, first, stop);
      if (stop) break;
      if (in) {
        if (!any1 || a > last1) { b.keep[b1 + i] = 1; any1 = true; last1 = a; }
        if (!any2 || c > last2) { b.keep[b2 + j] = 1; any2 = true; last2 = c; }
      }
    }
  }
  u32 k = 0;
  for (u32 i = 0; i < n1; ++i) if (b.keep[b1 + i]) { b.cand[b1 + k] = b.cand[b1 + i]; b.vcnt[b1 + k] = b.vcnt[b1 + i]; ++k; }
  u32 m = 0;
  for (u32 j = 0; j < n2; ++j) if (b.keep[b2 + j]) { b.cand[b2 + m] = b.cand[b2 + j]; b.vcnt[b2 + m] = b.vcnt[b2 + j]; ++m; }
  if (k == 0 || m == 0) { k = 0; m = 0; }
  b.nv[r1] = k; b.nv[r2] = m;
}

// ------------------------------------------------------------------------------------------- gather
// Work item w = voff[r] + j for every surviving window j < nv[r] of read r.  Windows of reads that seeding already resolved
// get their record here (end L-1, err 0 or 1); the others become one VerifyItem each in a dense list, so that every lane of
// the bit-vector kernel has a window to verify.  A warp owns 32 consecutive reads: one scan over their window counts, one
// atomic for the warp's share of the list, then consecutive lanes take consecutive windows (owner found by a binary search
// over the scanned counts through shuffles); the list stays grouped by read.
__global__ void __launch_bounds__(128) gather_work(BatchView b) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = !*b.status, live = ok && r < b.n_reads;
  const u64 out_base = b.totals[2];
  u32 nvr = 0, c0 = 0, w0 = 0, L = 0, k = 0, code_off = 0; int st = BMBS_NONE;
  if (live) {
    nvr = b.nv[r];
    if (nvr) { c0 = b.coff[r]; w0 = b.voff[r]; L = b.len[r]; k = b.kk[r]; code_off = code_word_offset(b.offsets, r); st = b.round == 0 ? b.state[r] : BMBS_VERIFY; }
  }
  const bool is_ver = st == BMBS_VERIFY || st == BMBS_NONE;
  u32 incl = nvr, vincl = is_ver ? nvr : 0u;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 t = __shfl_up_sync(0xffffffffu, incl, o), tv = __shfl_up_sync(0xffffffffu, vincl, o);
    if (lane >= o) { incl += t; vincl += tv; }
  }
  const u32 total = __shfl_sync(0xffffffffu, incl, 31), vtotal = __shfl_sync(0xffffffffu, vincl, 31);
  const u32 excl = incl - nvr, vexcl = vincl - (is_ver ? nvr : 0u);
  u32 vbase = 0;
  if (lane == 0 && vtotal) vbase = atomicAdd(b.list_count + 3, vtotal);
  vbase = __shfl_sync(0xffffffffu, vbase, 0);
  for (u32 i0 = 0; i0 < total; i0 += 32) {
    const u32 i = i0 + lane;
    int o = 0;                                                    // owner: the lane with excl <= i < incl
#pragma unroll
    for (int step = 16; step; step >>= 1) { const u32 t = __shfl_sync(0xffffffffu, incl, o + step - 1); if (t <= i) o += step; }
    o &= 31;
    const u32 j = i - __shfl_sync(0xffffffffu, excl, o);
    const u32 s = __shfl_sync(0xffffffffu, c0, o) + j, w = __shfl_sync(0xffffffffu, w0, o) + j;
    const u32 oL = __shfl_sync(0xffffffffu, L, o), ok_ = __shfl_sync(0xffffffffu, k, o), ocode = __shfl_sync(0xffffffffu, code_off, o);
    const int ost = __shfl_sync(0xffffffffu, st, o);
    const u32 ovex = __shfl_sync(0xffffffffu, vexcl, o);
    if (i < total) {
      const u64 site = b.cand[s]; const u32 vote = b.vcnt[s];
      if (ost == BMBS_VERIFY || ost == BMBS_NONE) {
        VerifyItem it; it.site = site; it.wi = w; it.vote = vote; it.code_off = ocode; it.L = oL; it.k = ok_; it.pad = 0;
        b.vitems[vbase + ovex + j] = it;
      } else {
        bmbs_cand c; c.site = site; c.vote = vote; c.end_site = (int16_t)(oL - 1); c.err = ost == BMBS_ONE_MISMATCH ? 1 : 0;
        b.out_cand[out_base + w] = c;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------- verify
// BS_Reserve_Banded_BPM (Levenshtein_Cal.h:351-567): Hyyro banded Myers, band 2k+1, "pattern" = reference window of
// L+2k bases, "text" = read; read T matches reference C or T, N matches nothing, an all-zero (out-of-genome)
// window matches nothing.  One thread per window; the window's four match bit-planes (A, C, G, T|C) plus a zero
// plane live in shared memory as overlapping 64-bit chunks (chunk c = window bits [32c, 32c+64)), so a column's
// Eq word is one LDS.64 + one shift; band state is one W-bit word per thread (W = 32 for k <= 15, 64 for k <= 31;
// any width >= 2k+2 gives identical results, DESIGN.md §5).
// One column of the band (Levenshtein_Cal.h:436-445).  Bit 0 of D0 (1 = the diagonal cell matched) is shifted into `dbits`,
// newest on top, so that the diagonal error count costs one funnel shift per column and one POPC per eight columns.
template <typename W>
__device__ __forceinline__ void bpm_step(W eq, W& VP, W& VN, u32& dbits) {
  W X = eq | VN;
  const W D0 = ((VP + (X & VP)) ^ VP) | X;
  const W HN = VP & D0, HP = VN | ~(VP | D0);
  X = D0 >> 1;
  VN = X & HP; VP = HN | ~(X | HP);
  dbits = __funnelshift_r(dbits, (u32)D0, 1);
}

// Eq word of column 32*ch + t for read symbol `code`: bits [t, t + band) of the window's match plane.  cb points at the
// thread's chunk ch of plane 0; planes are `pstride` words apart, chunks `stride` words.
template <typename W>
__device__ __forceinline__ W eq_word(const u64* __restrict__ cb, u32 pstride, int stride, u32 code, int t, W mask) {
  const u64 e0 = cb[code * pstride];
  if (sizeof(W) == 4) return (W)(e0 >> t) & mask;
  const u32 e1hi = (u32)(cb[code * pstride + stride] >> 32);
  const u32 lo = __funnelshift_r((u32)e0, (u32)(e0 >> 32), t), hi = __funnelshift_r((u32)(e0 >> 32), e1hi, t);
  return (W)(((u64)hi << 32) | lo) & mask;
}

template <typename W>
__device__ __forceinline__ void bpm_columns(const u64* __restrict__ sm, int stride, int nch2, const u32* __restrict__ rw,
                                            int L, int k, int& end_out, u32& err_out) {
  const int band = 2 * k + 1;
  const W mask = band >= (int)(8 * sizeof(W)) ? ~(W)0 : (((W)1 << band) - 1);
  const u32 pstride = (u32)(nch2 * stride);
  W VP = 0, VN = 0;
  int err = 0;
  const int limit = 3 * k;   // err - 2k > k can never recover (Levenshtein_Cal.h:455); checked every eight columns
  bool dead = false;
  u32 dbits = 0;
  u32 next_word = L > 0 ? __ldg(rw) : 0u;     // the read's code words are fetched one group of eight columns ahead
  for (int ch = 0; ch * 32 < L && !dead; ++ch) {
    const u64* cb = sm + ch * stride;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int i0 = ch * 32 + g * 8;
      if (i0 < L && !dead) {
        const u32 word = next_word;
        if (i0 + 8 < L) next_word = __ldg(rw + (i0 >> 3) + 1);
        if (i0 + 8 <= L) {
#pragma unroll
          for (int j = 0; j < 8; ++j) bpm_step<W>(eq_word<W>(cb, pstride, stride, (word >> (4 * j)) & 0xFu, g * 8 + j, mask), VP, VN, dbits);
          err += 8 - __popc(dbits >> 24);
        } else {
          const int n = L - i0;
          for (int j = 0; j < n; ++j) bpm_step<W>(eq_word<W>(cb, pstride, stride, (word >> (4 * j)) & 0xFu, g * 8 + j, mask), VP, VN, dbits);
          err += n - __popc(dbits >> (32 - n));
        }
        if (err > limit) dead = true;
      }
    }
  }
  end_out = -1; err_out = 0xFFFFFFFFu;
  if (dead) return;
  band_last_column<W>(VP, VN, err, k, L, end_out, err_out);     // the last column, from VN run to VN run (bmbs_band_walk.h)
}

// ---- 32-bit band (k <= 15): the form the ALU pipe is budgeted for.  Per column: one PRMT takes the read's code out of a
// byte-spread copy of its nibble word, one IMAD turns it into the shared-memory address of that symbol's match plane, one
// funnel shift aligns the 64-bit chunk to the column, and the band mask rides in the LOP3 that forms X = (Eq & mask) | VN
// (written as inline lop3 so that the compiler keeps VN in a register instead of recomputing it inside a second LOP3):
// 7 LOP3 + 3 SHF + 1 PRMT on the ALU pipe, IMAD + IADD on the FMA pipe, one LDS.64.
__device__ __forceinline__ void bpm_step32(u32 eq_raw, u32 mask, u32& VP, u32& VN, u32& dbits) {
  u32 X;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(X) : "r"(eq_raw), "r"(mask), "r"(VN));    // (eq_raw & mask) | VN
  const u32 D0 = ((VP + (X & VP)) ^ VP) | X;
  const u32 HN = VP & D0, HP = VN | ~(VP | D0);
  const u32 X2 = D0 >> 1;
  VN = X2 & HP; VP = HN | ~(X2 | HP);
  dbits = __funnelshift_r(dbits, D0, 1);
}
// eight columns of group G (window bits 8G .. 8G+7 of the chunk) on one word of read codes
template <int G, int J>
__device__ __forceinline__ void bpm_col32(const char* __restrict__ cbytes, u32 pstride8, u32 ev, u32 od, u32 mask, u32& VP, u32& VN, u32& dbits) {
  const u32 code = __byte_perm((J & 1) ? od : ev, 0u, 0x4440u | (u32)(J >> 1));          // nibble J of the word, as a number
  const u64 e0 = *reinterpret_cast<const u64*>(cbytes + code * pstride8);
  bpm_step32((u32)(e0 >> (G * 8 + J)), mask, VP, VN, dbits);
}
template <int G>
__device__ __forceinline__ void bpm_group32(const char* __restrict__ cbytes, u32 pstride8, u32 word, u32 mask, u32& VP, u32& VN, u32& dbits) {
  const u32 ev = word & 0x0F0F0F0Fu, od = (word >> 4) & 0x0F0F0F0Fu;
  bpm_col32<G, 0>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 1>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 2>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 3>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 4>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 5>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 6>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
  bpm_col32<G, 7>(cbytes, pstride8, ev, od, mask, VP, VN, dbits);
}
// the last n < 8 columns of a read, in group G of the chunk
template <int G>
__device__ __forceinline__ void bpm_tail32(const char* __restrict__ cbytes, u32 pstride8, u32 word, int n, u32 mask, u32& VP, u32& VN, u32& dbits) {
  for (int j = 0; j < n; ++j) {
    const u32 code = (word >> (4 * j)) & 0xFu;
    const u64 e0 = *reinterpret_cast<const u64*>(cbytes + code * pstride8);
    bpm_step32((u32)(e0 >> (G * 8 + j)), mask, VP, VN, dbits);
  }
}
// What was measured and left out (profiles/r02X_verify_variant*.jsonl): the band shift D0 >> 1 and the diagonal bit from one
// IMAD.WIDE.U32 by 2^31 (high word / bit 31 of the low word), the diagonal count by IMAD.HI.U32, the Eq alignment as IMAD.HI.U32 +
// IMAD by 2^(32-c), the code extraction as a chain of IMAD.WIDE.U32 by 16 -- 8.6 / 7.7 instead of 11.5 ALU-pipe instructions per
// column, every result identical, and 3 / 3 / 6 % SLOWER at L = 150: the kernel's time follows its instruction count
// (15.1 -> 15.4 / 16.7 / 16.6 per column), not the ALU pipe's share of it.
__device__ __forceinline__ void bpm_columns32(const u64* __restrict__ sm, int stride, int nch2, const u32* __restrict__ rw,
                                              int L, int k, int& end_out, u32& err_out) {
  const int band = 2 * k + 1;
  const u32 mask = band >= 32 ? ~0u : ((1u << band) - 1u);
  const u32 pstride8 = (u32)(nch2 * stride) * 8u;
  u32 VP = 0, VN = 0;
  int err = 0;
  const int limit = 3 * k;   // err - 2k > k can never recover (Levenshtein_Cal.h:455); checked every 32 columns
  u32 dbits = 0;             // the diagonal bits of the last 32 columns
  end_out = -1; err_out = 0xFFFFFFFFu;
  // a read's code words start on a 16-byte boundary (code_word_offset): the 32 columns of a chunk are one 128-bit load, fetched
  // one chunk ahead (a read's words are followed by the next read's or by slack: the look-ahead past the last chunk reads
  // something that is never used)
  const uint4* rq = reinterpret_cast<const uint4*>(rw);
  uint4 nextq = __ldg(rq++);
  int rem = L;                                              // columns left
  const char* cbytes = reinterpret_cast<const char*>(sm);
  const u32 chunk_bytes = (u32)stride * 8u;
  for (; rem >= 32; rem -= 32, cbytes += chunk_bytes) {
    const uint4 q = nextq; nextq = __ldg(rq++);
    bpm_group32<0>(cbytes, pstride8, q.x, mask, VP, VN, dbits);
    bpm_group32<1>(cbytes, pstride8, q.y, mask, VP, VN, dbits);
    bpm_group32<2>(cbytes, pstride8, q.z, mask, VP, VN, dbits);
    bpm_group32<3>(cbytes, pstride8, q.w, mask, VP, VN, dbits);
    err += 32 - __popc(dbits);
    if (err > limit) return;
  }
  if (rem > 0) {                                            // the last, partial chunk
    const uint4 q = nextq;
    if (rem >= 8) bpm_group32<0>(cbytes, pstride8, q.x, mask, VP, VN, dbits); else bpm_tail32<0>(cbytes, pstride8, q.x, rem, mask, VP, VN, dbits);
    if (rem >= 16) bpm_group32<1>(cbytes, pstride8, q.y, mask, VP, VN, dbits); else if (rem > 8) bpm_tail32<1>(cbytes, pstride8, q.y, rem - 8, mask, VP, VN, dbits);
    if (rem >= 24) bpm_group32<2>(cbytes, pstride8, q.z, mask, VP, VN, dbits); else if (rem > 16) bpm_tail32<2>(cbytes, pstride8, q.z, rem - 16, mask, VP, VN, dbits);
    if (rem > 24) bpm_tail32<3>(cbytes, pstride8, q.w, rem - 24, mask, VP, VN, dbits);
    err += rem - __popc(dbits >> (32 - rem));
    if (err > limit) return;
  }
  band_last_column<u32>(VP, VN, err, k, L, end_out, err_out);   // the last column, from VN run to VN run (bmbs_band_walk.h)
}

__global__ void __launch_bounds__(128, 7) verify_windows(DevIndex ix, BatchView b, int nch2) {
  extern __shared__ u64 sm_all[];
  __shared__ u64 s_cnt[3];
  if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const u32 total_work = *b.status ? 0u : b.list_count[3];
  const u64 out_base = b.totals[2];
  const int stride = blockDim.x;
  u64* sm = sm_all + threadIdx.x;
  u64 cells = 0, wbytes = 0, verified = 0;
  for (u32 vi = blockIdx.x * blockDim.x + threadIdx.x; vi < total_work; vi += gridDim.x * blockDim.x) {
    const uint4* ip = (const uint4*)(b.vitems + vi);
    const uint4 i0 = __ldg(ip), i1 = __ldg(ip + 1);
    const u64 site = (u64)i0.x | ((u64)i0.y << 32);
    const u32 wi = i0.z, vote = i0.w;
    const int L = (int)i1.y, k = (int)i1.z;
    int end = -1; u32 err = 0xFFFFFFFFu;
    {
      const int plen = L + 2 * k;
      const int nch = (L + 31) >> 5;           // chunks addressed by the column loop
      const int nst = k <= 15 ? nch : nch + 1;  // chunks staged: the 64-bit band also reads the chunk after the column's (nst <= nch2, see launch_verify)
      const bool inside = window_inside(ix, site, (u64)plen);
      if (inside) {
        // window words gp[0 .. nch+2]: eight chunks per pass, their ten words loaded back to back (independent loads in
        // flight together instead of one dependent round trip per chunk)
        const uint2* gp = ix.planes + (site >> 5);
        const unsigned sh = (unsigned)site & 31u;
        for (int c0 = 0; c0 < nst; c0 += 8) {
          uint2 w[10];
#pragma unroll
          for (int j = 0; j < 10; ++j) w[j] = c0 + j <= nch + 2 ? __ldg(gp + c0 + j) : make_uint2(0u, 0u);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int c = c0 + j;
            if (c < nst) {
              const u32 lo0 = __funnelshift_r(w[j].x, w[j + 1].x, sh), hi0 = __funnelshift_r(w[j].y, w[j + 1].y, sh);
              const u32 lo1 = __funnelshift_r(w[j + 1].x, w[j + 2].x, sh), hi1 = __funnelshift_r(w[j + 1].y, w[j + 2].y, sh);
              const u64 lo = (u64)lo0 | ((u64)lo1 << 32), hi = (u64)hi0 | ((u64)hi1 << 32);
              sm[(0 * nch2 + c) * stride] = ~hi & ~lo;   // A
              sm[(1 * nch2 + c) * stride] = ~hi & lo;    // C
              sm[(2 * nch2 + c) * stride] = hi & ~lo;    // G
              sm[(3 * nch2 + c) * stride] = lo;          // T (matches reference C or T)
              sm[(4 * nch2 + c) * stride] = 0;           // N / other
            }
          }
        }
        wbytes += (u64)(nch + 3) * 8;
      } else {
        for (int c = 0; c < nst; ++c) for (int p = 0; p < 5; ++p) sm[(p * nch2 + c) * stride] = 0;
      }
      const u32* rw = b.codes + i1.x;
      if (k <= 15) bpm_columns32(sm, stride, nch2, rw, L, k, end, err);
      else bpm_columns<u64>(sm, stride, nch2, rw, L, k, end, err);
      ++verified; cells += (u64)L * (u64)(2 * k + 1);
    }
    bmbs_cand o; o.site = site; o.vote = vote; o.end_site = (int16_t)end; o.err = err == 0xFFFFFFFFu ? (uint16_t)0xFFFF : (uint16_t)err;
    b.out_cand[out_base + wi] = o;
  }
  atomicAdd(&s_cnt[0], verified); atomicAdd(&s_cnt[1], cells); atomicAdd(&s_cnt[2], wbytes);
  __syncthreads();
  if (threadIdx.x == 0) { atomicAdd(b.counters + CNT_VERIFIED, s_cnt[0]); atomicAdd(b.counters + CNT_CELLS, s_cnt[1]); atomicAdd(b.counters + CNT_WINBYTES, s_cnt[2]); }
}


// ------------------------------------------------------------------------------------------- CIGAR refinement
// fast_recalculate_bs_Cigar (ksw.cpp:2578-3148) for alignments with indels: ksw_semi_global_quality_back (:1850-2045), the
// semi-global banded (2k+1) affine-gap alignment of the read against its window with traceback, then the end fix-ups
// (leading / trailing insertions become matches, :2894-2990) and the NM recount over the final operations (:2990-3143).
// Values and tie-breaks are the reference's, cell by cell (every comparison below is written as it is there).
//   refine_warp<C>   one warp per alignment, C band cells per lane: lane l holds cells l and l + 32 (C = 1 for bands of up to
//                    32 cells, k <= 15; C = 2 for up to 63 cells, k 16..31).  Within a row the match score m and the vertical
//                    gap e only depend on the row above (m: the cell's own h, e: the next cell's), and the horizontal gap opens
//                    from m alone, f[j+1] = max(f[j] - ext, m[j] - open - ext): a max-plus prefix scan over the lanes, one
//                    half after the other.  The four direction bits of a row are four ballots per half, kept in shared memory
//                    (C x 16 bytes per row), so the DP touches global memory only for the read, its qualities and the window.
//                    The end fix-ups are refine_fix_ends (bmbs_refine_ends.h), the same code the CPU refinement runs.
struct RefineScoring { int mp_max, mp_min, n_pen, gap_open, gap_ext, q_base; };

// read character against the window base at double-strand position pos (an out-of-strand window matches nothing)
__device__ __forceinline__ u32 refine_mismatch(const DevIndex& ix, bool inside, u64 pos, char rc) {
  if (!inside) return 1u;
  const int g = strand_base(ix, pos);
  return (u32)!(rc == "ACGT"[g] || (g == 1 && rc == 'T'));
}

__device__ __forceinline__ int refine_nt4(char c) {
  switch (c) { case 'A': case 'a': return 0; case 'C': case 'c': return 1; case 'G': case 'g': return 2; case 'T': case 't': return 3; default: return 4; }
}

constexpr int RW_WARPS = 4;
template <int C>
__global__ void __launch_bounds__(32 * RW_WARPS) refine_warp(DevIndex ix, const bmbs_refine_item* __restrict__ items, u32 n, const char* __restrict__ seqs,
                                                             const char* __restrict__ quals, RefineScoring sc, u32* __restrict__ ops_scratch, const u64* __restrict__ ops_off,
                                                             bmbs_refine_result* __restrict__ res, u32* __restrict__ ops_out, unsigned long long* ops_total, u64 ops_cap, u32 max_len) {
  // [RW_WARPS][max_len][C]: bit l of .x/.y = h source of cell l + 32c, .z = e extended, .w = f extended
  extern __shared__ uint4 s_dirs[];
  __shared__ int s_fin[RW_WARPS][8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint4* dir = s_dirs + (size_t)w * max_len * C;
  const u32 warps = gridDim.x * RW_WARPS;
  const int NEG = -0x40000000, goe = sc.gap_open + sc.gap_ext, ge = sc.gap_ext;
  for (u32 it = blockIdx.x * RW_WARPS + w; it < n; it += warps) {
    const bmbs_refine_item q = items[it];
    const int rlen = q.len, k = q.k, band = 2 * k + 1, wlen = rlen + 2 * k;
    if ((band > 32) != (C > 1)) continue;               // the other instance's
    const char* read = seqs + q.seq_off; const char* qual = quals + q.seq_off;
    const bool inside = window_inside(ix, q.site, (u64)wlen);
    bool act[C]; int hd[C], e_prev[C]; u32 wlo[C], whi[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { act[c] = lane + 32 * c < band; hd[c] = 0; e_prev[c] = -goe; wlo[c] = whi[c] = 0; }   // row 0: H = 0, E = -(open + ext)
    int my_t = 4, my_mism = 0;
    for (int i = 0; i < rlen; ++i) {
      const int ph = i & 31;
      if (ph == 0) {
        // every 32 rows: lane l prepares row i + l (base code, quality-scaled mismatch penalty) and the next 32 window bases of
        // each of its diagonals (window position i + lane + 32c + 0..31)
        const int ri = i + lane;
        my_t = 4; my_mism = 0;
        if (ri < rlen) {
          my_t = refine_nt4(read[ri]);
          double phred = (double)((int)qual[ri] - sc.q_base);
          if (phred > 40) phred = 40;
          phred = phred / 40;
          my_mism = -sc.mp_min - (int)((double)(signed char)(sc.mp_max - sc.mp_min) * phred);
        }
        if (inside) {
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const u64 p = q.site + (u64)(i + lane + 32 * c);
            const uint2 g0 = __ldg(ix.planes + (p >> 5)), g1 = __ldg(ix.planes + (p >> 5) + 1);
            const unsigned sh = (unsigned)p & 31u;
            wlo[c] = __funnelshift_r(g0.x, g1.x, sh); whi[c] = __funnelshift_r(g0.y, g1.y, sh);
          }
        }
      }
      const int t = __shfl_sync(0xffffffffu, my_t, ph), mism = __shfl_sync(0xffffffffu, my_mism, ph);
      int carry = 0;                                    // the low half's scan maximum (lane 31), where the high half's scan starts
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const int jj = lane + 32 * c;
        const int qb = inside ? (int)(((wlo[c] >> ph) & 1u) | (((whi[c] >> ph) & 1u) << 1)) : 4;
        int sco;
        if (t == 4 || qb == 4) sco = -sc.n_pen;
        else if (t == qb || (t == 3 && qb == 1)) sco = 0;
        else sco = mism;
        const int m = hd[c] + sco;
        // e entering cell jj comes from cell jj + 1 of the row above: lane 31 of the low half reads lane 0 of the high half, whose
        // e_prev still holds the row above
        int e = c + 1 < C ? __shfl_sync(0xffffffffu, lane == 0 ? e_prev[(c + 1) % C] : e_prev[c], lane + 1) : __shfl_down_sync(0xffffffffu, e_prev[c], 1);
        if (i == 0) e = -goe; else if (jj == band - 1) e = NEG;
        u32 d = m >= e ? 0u : 1u;
        int h = m >= e ? m : e;
        const int open = m - goe;
        // f entering cell jj: NEG at the band start, then f[jj+1] = max(f[jj] - ge, open[jj]) -- a prefix maximum of open[q] + q ge
        int a = act[c] ? open + jj * ge : (int)0x80000000;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, a, o); if (lane >= o) a = max(a, v); }
        if (c > 0) a = max(a, carry);
        int ex = __shfl_up_sync(0xffffffffu, a, 1);
        if (c > 0 && lane == 0) ex = carry;
        if (c + 1 < C) carry = __shfl_sync(0xffffffffu, a, 31);
        const int f = jj == 0 ? NEG : max(NEG - jj * ge, ex - (jj - 1) * ge);
        d = h >= f ? d : 2u;
        h = h >= f ? h : f;
        e -= ge;
        const bool e_ext = e > open;
        if (!e_ext) e = open;
        const bool f_ext = f - ge > open;
        const u32 b0 = __ballot_sync(0xffffffffu, act[c] && (d & 1u)), b1 = __ballot_sync(0xffffffffu, act[c] && (d & 2u));
        const u32 be = __ballot_sync(0xffffffffu, act[c] && e_ext), bf = __ballot_sync(0xffffffffu, act[c] && f_ext);
        if (lane == 0) dir[i * C + c] = make_uint4(b0, b1, be, bf);
        hd[c] = h; e_prev[c] = e;
      }
    }
    // best end in the last row: the middle of the band unless another cell is strictly better, then the rightmost best one
    int hv = (int)0x80000000;
#pragma unroll
    for (int c = 0; c < C; ++c) if (act[c]) hv = max(hv, hd[c]);
    const int vmax = __reduce_max_sync(0xffffffffu, hv);
    u64 at_max = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) at_max |= (u64)__ballot_sync(0xffffffffu, act[c] && hd[c] == vmax) << (32 * c);
    const int best = C == 1 ? (((u32)at_max >> k) & 1u ? k : 31 - __clz((int)at_max))
                            : ((at_max >> k) & 1u ? k : 63 - __clzll((long long)at_max));
    __syncwarp();
    if (lane == 0) {
      u32* ops = ops_scratch + ops_off[it];
      const u32 cap = (u32)(ops_off[it + 1] - ops_off[it]);
      u32 n_ops = 0, cur = 0;
      auto push = [&](u32 op, u32 len) {
        if (n_ops == 0 || (cur & 0xfu) != op) { if (n_ops) ops[cap - n_ops] = cur; cur = len << 4 | op; ++n_ops; } else cur += len << 4;
      };
      int i = rlen - 1, j = rlen - 1 + best, state = 0;
      while (i >= 0 && j >= 0) {
        const uint4 dd = dir[C == 1 ? i : i * C + ((j - i) >> 5)]; const int jj = C == 1 ? j - i : (j - i) & 31;   // cell j - i's word and bit
        if (state == 0) state = (int)(((dd.x >> jj) & 1u) | (((dd.y >> jj) & 1u) << 1));
        else if (state == 1) state = (int)((dd.z >> jj) & 1u);
        else state = (int)(((dd.w >> jj) & 1u) << 1);
        if (state == 0) { push(0, 1); --i; --j; }
        else if (state == 1) { push(2, 1); --i; }
        else { push(1, 1); --j; }
      }
      if (i >= 0) push(2, (u32)(i + 1));
      if (n_ops) ops[cap - n_ops] = cur;
      int qb = j + 1, qe = rlen - 1 + best, cb = 0, ce = -1;
      if (n_ops) refine_fix_ends(ops + (cap - n_ops), (int)n_ops, qb, qe, cb, ce);
      s_fin[w][0] = qb; s_fin[w][1] = qe; s_fin[w][2] = (int)(cap - n_ops) + cb; s_fin[w][3] = ce - cb + 1;
    }
    __syncwarp();
    const int qb = s_fin[w][0], qe = s_fin[w][1], first = s_fin[w][2], n_fin = max(s_fin[w][3], 0);
    const u32* fo = ops_scratch + ops_off[it] + first;
    // NM over the final operations: the lanes share the bases of every match run
    u32 nm = 0;
    {
      int wi = qb, ri = 0;
      for (int x = 0; x < n_fin; ++x) {
        const u32 op = fo[x] & 0xfu, len = fo[x] >> 4;
        if (op == 0) { for (u32 y = lane; y < len; y += 32) nm += refine_mismatch(ix, inside, q.site + (u64)(long long)(wi + (int)y), read[ri + (int)y]); wi += (int)len; ri += (int)len; }
        else if (op == 1) { wi += (int)len; if (lane == 0) nm += len; }
        else { ri += (int)len; if (lane == 0) nm += len; }
      }
      nm = __reduce_add_sync(0xffffffffu, nm);
    }
    unsigned long long at = 0;
    if (lane == 0) at = atomicAdd(ops_total, (unsigned long long)n_fin);
    at = __shfl_sync(0xffffffffu, at, 0);
    if (at + (u64)n_fin <= ops_cap) for (int x = lane; x < n_fin; x += 32) ops_out[at + x] = fo[x];
    if (lane == 0) { bmbs_refine_result r; r.score = vmax; r.qb = qb; r.qe = qe; r.n_ops = (u32)n_fin; r.ops_off = (u32)at; r.nm = nm; res[it] = r; }
    __syncwarp();
  }
}


// ------------------------------------------------------------------------------------------- sensitive pairing
// select_suit_candidates (Schema.cpp:4775-4824): a verified hit of the mate within [dmin, dmax] of `site`?  The reference
// takes a hit at `site` itself through its skip branch, in_range through its stop branch.  The answer is the same: with
// dmax >= 0 both give 0 >= dmin, and with dmax < 0 no hit can ever be in range, so both return false.  Only the skip
// pointer moves differently, and it only saves time.
__device__ __forceinline__ bool mate_in_range(u64 site, const bmbs_cand* hits, int nh, int dmax, int dmin, int& next) {
  long long first = next;
  bool in = false, stop = false;
  for (int i = next; i < nh && !in && !stop; ++i) in = in_range(site, hits[i].site, dmax, dmin, i, first, stop);
  next = (int)first;
  return in;
}

// hits (err <= k) whose absolute end differs from that of the entry verified just before them, compacted to the
// front of the slice (map_candidate_votes_mutiple_cut_end_to_end_*_for_paired_end, Schema.cpp:7502-7512); with
// `mate` set only entries within range of a mate hit take part (the reference verifies only those,
// generate_candidate_votes_shift_filter, :4884-4992)
__device__ __forceinline__ u32 keep_hits_inplace(bmbs_cand* c, u32 n, u32 k, const bmbs_cand* mate, int nmate, int dmax, int dmin) {
  u32 kept = 0; u64 prev_end = ~0ull; int next = 0;
  for (u32 i = 0; i < n; ++i) {
    const bmbs_cand x = c[i];
    if (mate && !mate_in_range(x.site, mate, nmate, dmax, dmin, next)) continue;
    const u64 end_abs = x.site + (u64)(long long)x.end_site;
    const u32 err = x.err == 0xFFFF ? 0xFFFFFFFFu : x.err;
    if (err <= k && prev_end != end_abs) c[kept++] = x;
    prev_end = end_abs;
  }
  return kept;
}

// ---- warp-cooperative forms of the two walks above (one warp per pair: the lists of a pair in a repeat are thousands of
// entries long, and a single thread pays an L2 round trip per entry).  Both walks are pure per entry once "the previous
// entry that passed the mate filter" is known, as long as no coordinate has wrapped: with every site below 2^62,
// mate_in_range(site) == "a hit h with dmin <= |h - site| <= dmax exists" (the skip pointer only saves time on ascending
// sites), answered by binary searches over the site-sorted hits.  Lists with a wrapped coordinate (windows that start
// before the text; never hits) take the literal single-thread walk.
constexpr u64 SITE_SANE = 1ull << 62;
__device__ __forceinline__ int lower_bound_site(const bmbs_cand* hits, int nh, u64 v) {   // first i with hits[i].site >= v
  int lo = 0, hi = nh;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (hits[mid].site < v) lo = mid + 1; else hi = mid; }
  return lo;
}
__device__ __forceinline__ bool hit_between(const bmbs_cand* hits, int nh, long long lo, long long hi) {   // a hit with lo <= site <= hi
  if (hi < 0 || lo > hi) return false;
  const int i = lower_bound_site(hits, nh, (u64)(lo < 0 ? 0 : lo));
  return i < nh && hits[i].site <= (u64)hi;
}
__device__ __forceinline__ bool in_range_pure(u64 site, const bmbs_cand* hits, int nh, int dmax, int dmin) {
  const long long s = (long long)site;
  if (dmax < 0) return false;
  const long long lo0 = dmin > 0 ? dmin : 0;                          // h <= s: dmin <= s - h <= dmax
  if (hit_between(hits, nh, s - dmax, s - lo0)) return true;
  const long long lo1 = dmin > 1 ? dmin : 1;                          // h > s: dmin <= h - s <= dmax
  return hit_between(hits, nh, s + lo1, s + dmax);
}
// are all coordinates of c[0..n) sane?  (warp-wide answer)
__device__ __forceinline__ bool warp_all_sane(const bmbs_cand* c, u32 n, int lane) {
  bool ok = true;
  for (u32 i = lane; i < n; i += 32) ok = ok && c[i].site < SITE_SANE;
  return __all_sync(0xffffffffu, ok);
}
// keep_hits_inplace by a warp; every lane returns the count
__device__ __forceinline__ u32 warp_keep_hits(bmbs_cand* c, u32 n, u32 k, const bmbs_cand* mate, int nmate, int dmax, int dmin, int lane) {
  const bool sane = warp_all_sane(c, n, lane) && (!mate || warp_all_sane(mate, (u32)nmate, lane));
  if (!sane) {
    u32 kept = 0;
    if (lane == 0) kept = keep_hits_inplace(c, n, k, mate, nmate, dmax, dmin);
    __syncwarp();
    return __shfl_sync(0xffffffffu, kept, 0);
  }
  u32 kept = 0; u64 carry_end = ~0ull;                                  // absolute end of the last entry that passed the mate filter
  for (u32 base = 0; base < n; base += 32) {
    const u32 i = base + lane;
    const bool valid = i < n;
    bmbs_cand x; x.site = 0; x.vote = 0; x.end_site = 0; x.err = 0;
    if (valid) x = c[i];
    const bool pass = valid && (!mate || in_range_pure(x.site, mate, nmate, dmax, dmin));
    const u64 end_abs = x.site + (u64)(long long)x.end_site;
    const u32 pm = __ballot_sync(0xffffffffu, pass);
    const u32 below = pm & ((1u << lane) - 1u);
    const int src = below ? 31 - __clz(below) : 0;
    const u64 prev_in_chunk = __shfl_sync(0xffffffffu, end_abs, src);
    const u64 prev_end = below ? prev_in_chunk : carry_end;
    const u32 err = x.err == 0xFFFF ? 0xFFFFFFFFu : x.err;
    const bool keep = pass && err <= k && prev_end != end_abs;
    const u32 km = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) c[kept + __popc(km & ((1u << lane) - 1u))] = x;           // kept + rank <= i: never ahead of the entries still to be read
    kept += __popc(km);
    if (pm) carry_end = __shfl_sync(0xffffffffu, end_abs, 31 - __clz(pm));
    __syncwarp();
  }
  return kept;
}

// After every window of both mates has been verified: the mate with fewer first-seed candidates is the primary
// (Schema.cpp:23326); its hits are final; the other mate keeps only windows near a primary hit; a secondary left
// without a hit goes to the re-seeding list (:23562-23640).  One thread per pair, literal walks.
__global__ void __launch_bounds__(128) sens_pair(BatchView b) {
  const int lane = threadIdx.x & 31;
  const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;           // one warp per pair
  bool reseed = false; u32 rs = 0;
  if (p * 2 + 1 < b.n_reads && !*b.status) {
    const int r1 = 2 * p, r2 = r1 + 1;
    const bool first_is_1 = b.first_cands[r1] <= b.first_cands[r2];
    const int pri = first_is_1 ? r1 : r2, sec = first_is_1 ? r2 : r1;
    int dmax, dmin; pair_bounds(b, r1, r2, dmax, dmin);
    bmbs_cand* cp = b.out_cand + b.voff[pri]; bmbs_cand* cs = b.out_cand + b.voff[sec];
    u32 occp = b.nv[pri], occs = 0;
    if (!is_resolved(b.state[pri])) occp = warp_keep_hits(cp, occp, b.kk[pri], nullptr, 0, 0, 0, lane);
    __syncwarp();
    if (occp) {
      occs = b.nv[sec];
      if (!is_resolved(b.state[sec])) {
        occs = warp_keep_hits(cs, occs, b.kk[sec], cp, (int)occp, dmax, dmin, lane);
        if (occs == 0) { reseed = true; rs = (u32)sec; }
      }
    }
    if (lane == 0) {
      b.res_first[pri] = b.voff[pri]; b.res_n[pri] = occp;
      b.res_first[sec] = b.voff[sec]; b.res_n[sec] = occs;
    }
  }
  list_append(b.list4, b.list_count + 2, reseed && lane == 0, rs);
}

__global__ void reseed_clear(BatchView b) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < b.n_reads) { b.ntask[r] = 0; b.ncand[r] = 0; b.nv[r] = 0; }
  if (r == 0) { b.totals[2] = b.totals[1]; b.list_count[3] = 0; b.sort_count[0] = 0; b.sort_count[1] = 0; b.sort_count[2] = 0; b.sort_count[3] = 0; b.big_count[0] = 0; b.scratch_used[0] = 0; }      // the re-seeding round appends to out_cand
}

// reseed_filter_muti_thread, Schema.cpp:16998-17240: up to three exact seeds chosen from the gaps of the seeds used so
// far (select_best_seeds, :16630-16670), then a greedy seed every 8 bases; a multi-hit seed counts from 20 bases.
// One warp per read.  Where a seed starts does not depend on the seeds before it (fixed positions, then a fixed step of 8),
// only whether it is still looked at does (the seed budget, and the loops stop at an unusable seed that reaches the read
// end).  So the lanes compute the seeds side by side -- each one a chain of dependent table / occ lookups, long in
// repeats -- and lane 0 then replays the reference's loop over the finished results.
struct ReseedResult { u64 sp, val; u32 hits, mlen; u32 off, flags; };   // flags bit0: val is a site, bit1: val is a suffix-array value
__global__ void __launch_bounds__(128) seed_reseed(DevIndex ix, BatchView b, u32 plane_cap) {
  extern __shared__ uint4 s_planes[];      // [plane_cap][SEED_BLOCK]: column (warp's first thread) holds the warp's read
  __shared__ u64 s_cnt[4];
  __shared__ unsigned char s_lut[256];
  __shared__ ReseedResult s_res[4][32];
  if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
  build_key_lut(s_lut);
  __syncthreads();
  const u32 n4 = *b.status ? 0u : b.list_count[2];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const u32 warps = gridDim.x * (blockDim.x >> 5);
  SeedCounters cn;
  for (u32 i = blockIdx.x * (blockDim.x >> 5) + wid; i < n4; i += warps) {
    const u32 r = b.list4[i];
    const u32 L = b.len[r];
    // the read's chunks, staged once for the warp
    ReadPlanes rp; rp.p = b.rplanes + plane_chunk_offset(b.offsets, (int)r); rp.s = s_planes + (threadIdx.x & ~31u);
    rp.ns = (L >> 5) + 2; if (rp.ns > plane_cap) rp.ns = plane_cap;
    __syncwarp();
    for (u32 c = lane; c < rp.ns; c += 32) s_planes[c * SEED_BLOCK + (threadIdx.x & ~31u)] = __ldg(rp.p + c);
    __syncwarp();
    u64 max_seeds = (u64)L / 10 - 1; if (max_seeds > 25) max_seeds = 25;
    const unsigned short* k5 = b.bk + (size_t)r * 5;
    const u32 bn = k5[0], s0 = k5[1], s1 = k5[2], e_prev = k5[3], e_last = k5[4];
    u32 rs[3], rl[3]; u32 nsel = 0;
    if (bn >= 2) { rs[0] = s0; rl[0] = s1 - s0; rs[1] = e_prev; rl[1] = L - e_prev; nsel = 2; }
    else if (bn == 1) { rs[0] = s0; rl[0] = L / 2; rs[1] = s0 + L / 2; rl[1] = L - rs[1]; nsel = 2; }
    // with no seed used the reference reads element [-1] of two malloc'ed int arrays: 0 with glibc -> the whole read
    const u32 last_end = bn ? e_last : 0;
    if (last_end < L) { rs[nsel] = last_end; rl[nsel] = L - last_end; ++nsel; }
    const u32 goff0 = bn > 1 ? (s0 + s1) / 2 : 4u;
    // lane j < nsel: exact seed j; lane nsel + g: greedy seed at goff0 + 8 g (at most 25 of them are ever looked at)
    ReseedResult me; me.sp = 0; me.val = 0; me.hits = 0; me.mlen = 0; me.off = 0; me.flags = 0;
    if ((u32)lane < nsel) {
      const u32 off = lane == 0 ? rs[0] : lane == 1 ? rs[1] : rs[2], mlen = lane == 0 ? rl[0] : lane == 1 ? rl[1] : rl[2];
      u64 sp = 0, ep = 0, site = 0; bool have_site = false;
      const u64 hits = count_exact(ix, rp, s_lut, off, mlen, sp, ep, have_site, site, cn.n_occ, cn.n_hash, cn.n_rows, cn.n_llf);
      me.sp = sp; me.val = site; me.hits = (u32)(hits > 0xFFFFFFFFull ? 0xFFFFFFFFull : hits); me.mlen = mlen; me.off = off; me.flags = have_site ? 1u : 0u;
    } else {
      const u32 off = goff0 + 8u * ((u32)lane - nsel);
      if (off < L && (u64)((u32)lane - nsel) < max_seeds) {
        const SeedHit h = seed_until_unique(ix, rp, s_lut, off, L - off, cn.n_occ, cn.n_hash);
        me.sp = h.sp; me.val = h.sa; me.hits = (u32)(h.hits > 0xFFFFFFFFull ? 0xFFFFFFFFull : h.hits); me.mlen = h.mlen; me.off = off; me.flags = h.has_sa ? 2u : 0u;
      }
    }
    s_res[wid][lane] = me;
    __syncwarp();
    if (lane == 0) {
      u32 nt = 0, nc = 0;
      TaskWriter tw{b, r, nt, nc};
      u64 seed_id = 0;
      for (; seed_id < nsel; ++seed_id) {
        const ReseedResult& q = s_res[wid][seed_id];
        const u32 cur = L - q.off;
        if (q.hits == 1) { if (q.flags & 1u) tw.emit(q.val, 0, 0, 0); else tw.emit(q.sp, 1, q.mlen, q.off); }
        else if (q.mlen >= 20 && q.hits <= MAX_SEED_HITS) { if (q.hits) tw.emit(q.sp, q.hits, q.mlen, q.off); }
        else if (cur == q.mlen) break;
      }
      u32 g = 0;
      for (u32 off = goff0; seed_id < max_seeds && off < L; off += 8, ++seed_id, ++g) {
        const ReseedResult& q = s_res[wid][nsel + g];
        const u32 cur = L - off;
        if (q.hits == 1) { if (q.flags & 2u) tw.emit(2 * ix.N - q.val - q.mlen - off, 0, 0, 0); else tw.emit(q.sp, 1, q.mlen, off); }
        else if (q.mlen >= 20 && q.hits <= MAX_SEED_HITS) { if (q.hits) tw.emit(q.sp, q.hits, q.mlen, off); }
        else if (cur == q.mlen) break;
      }
      tw.store();
    }
    __syncwarp();
  }
  flush_counters(s_cnt, cn, b.counters);
}


// re-seeded mates: keep the windows near a hit of the (final) primary before verifying them
__global__ void __launch_bounds__(128) sens_reseed_filter(BatchView b) {
  const u32 n4 = *b.status ? 0u : b.list_count[2];
  const int lane = threadIdx.x & 31;
  const u32 warps = gridDim.x * (blockDim.x >> 5);
  for (u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n4; i += warps) {      // one warp per re-seeded mate
    const int r = (int)b.list4[i], mate = r ^ 1;
    int dmax, dmin; pair_bounds(b, r & ~1, r | 1, dmax, dmin);
    const bmbs_cand* hits = b.out_cand + b.res_first[mate]; const int nh = (int)b.res_n[mate];
    const u32 beg = b.coff[r], n = b.nv[r];
    bool ok = true;
    for (u32 j = lane; j < n; j += 32) ok = ok && b.cand[beg + j] < SITE_SANE;
    const bool sane = __all_sync(0xffffffffu, ok) && warp_all_sane(hits, (u32)nh, lane);
    u32 kept = 0;
    if (!sane) {
      if (lane == 0) {
        int next = 0;
        for (u32 j = 0; j < n; ++j) {
          const u64 site = b.cand[beg + j];
          if (mate_in_range(site, hits, nh, dmax, dmin, next)) { b.cand[beg + kept] = site; b.vcnt[beg + kept] = b.vcnt[beg + j]; ++kept; }
        }
      }
    } else {
      for (u32 base = 0; base < n; base += 32) {
        const u32 j = base + lane;
        u64 site = 0; u32 vote = 0;
        if (j < n) { site = b.cand[beg + j]; vote = b.vcnt[beg + j]; }
        const bool keep = j < n && in_range_pure(site, hits, nh, dmax, dmin);
        const u32 km = __ballot_sync(0xffffffffu, keep);
        __syncwarp();
        if (keep) { const u32 at = beg + kept + __popc(km & ((1u << lane) - 1u)); b.cand[at] = site; b.vcnt[at] = vote; }
        kept += __popc(km);
        __syncwarp();
      }
    }
    if (lane == 0) b.nv[r] = kept;
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) sens_reseed_finish(BatchView b) {
  const u32 n4 = *b.status ? 0u : b.list_count[2];
  const u64 base = b.totals[2];
  const int lane = threadIdx.x & 31;
  const u32 warps = gridDim.x * (blockDim.x >> 5);
  for (u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n4; i += warps) {
    const int r = (int)b.list4[i];
    const u32 first = (u32)(base + b.voff[r]);
    const u32 kept = warp_keep_hits(b.out_cand + first, b.nv[r], b.kk[r], nullptr, 0, 0, 0, lane);
    if (lane == 0) { b.res_first[r] = first; b.res_n[r] = kept; }
  }
}

// ------------------------------------------------------------------------------------------- finalize
__global__ void finalize_reads(BatchView b) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= b.n_reads) return;
  bmbs_read_result o;
  o.site = b.site0[r]; o.first_cand = b.sensitive ? b.res_first[r] : b.voff[r];
  o.n_cand = b.sensitive ? b.res_n[r] : b.nv[r];
  if (r == 0) b.totals[3] = b.totals[2] + b.totals[1];
  o.one_mismatch_pos = b.one_mm[r]; o.state = b.state[r]; o.is_multiple_map = b.flags[r] & 1; o.reserved = 0;
  b.out_res[r] = o;
}

// ------------------------------------------------------------------------------------------- finishing (single end)
// What the reference's worker does after its verification calls, for every read of a single-end batch (SURVEY 8a V3, 8f-1):
//   * the vote-ordered reduction (Schema.cpp:7847-8056 / :8325-8745): the hit with the smallest err, "ambiguous" when another
//     hit with that err ends elsewhere, second_best_diff = what the running minimum stood at before the best hit was met.
//     The reference walks the windows in the order its unstable std::sort by vote leaves them.  finish_se (a thread per read,
//     two passes over the window list) computes the outcome from order-free quantities whenever the order among equal
//     votes cannot change it, and from the true order when the list has at most 16 windows (libstdc++ then runs a plain,
//     stable insertion sort).  The other reads go to finish_sorted, which replays the introsort step by step
//     (bmbs_sort_replay.h) in shared memory; lists beyond its capacity are handed to the host (BMBS_FIN_HOST).
//   * try_cigar_without_path (ksw.cpp:2515-2570): the best hit's diagonal re-read against the genome; exactly `err` mismatches
//     on it = an ungapped alignment, CIGAR <L>M, and the mismatch positions go back so that the host can price them by quality
//     (MismatchPenaltyByQuality; the quality strings never cross the link for such reads).  Otherwise the read is marked
//     BMBS_FIN_DP: the banded affine DP (refine_warp) decides.
//   * coordinates (Schema.cpp:12596-12650, :9188-9244): strand, chromosome, 1-based POS, and the drop of hits that run over
//     the end of their chromosome.
struct FinCounters { unsigned long long mism_used, fb_used, n_sorted, n_host, n_dp, n_unc_idx, n_unc_sbd, n_long, cursor_long, cursor_sorted, n_huge, cursor_huge, pad[4]; };

// What the finishing kernels write: a record per read, the mismatch positions of ungapped hits, the window lists of the reads
// handed back to the host (BMBS_FIN_HOST), the work lists of the later tiers and their counters.
struct FinishView {
  bmbs_final* fin;
  unsigned short* mism; u32 mism_cap;
  bmbs_cand* fb; u32 fb_cap;
  u32* sort_list; u32* long_list; u32* huge_list;
  FinCounters* fc;
  u32 pe_short;                  // pairs with more hits than this in both lists together go to finish_pe_long
};
// The finishing kernels take the fields of a FinishView as separate parameters and rebuild it on entry: with the struct as
// the parameter, nvcc loads every field at kernel entry and keeps them live (finish_se: 40 registers instead of 32 on sm_100a).
#define FINISH_PARAMS bmbs_final* fin, unsigned short* mism, u32 mism_cap, bmbs_cand* fb, u32 fb_cap, u32* sort_list, u32* long_list, u32* huge_list, FinCounters* fc, u32 pe_short
#define FINISH_VIEW FinishView{fin, mism, mism_cap, fb, fb_cap, sort_list, long_list, huge_list, fc, pe_short}

struct PlacedDev { u32 chrom; u64 pos; u32 reverse; bool off; };
__device__ __forceinline__ PlacedDev place_hit(const DevIndex& ix, u64 site, long long start_site, u64 end_site) {
  PlacedDev p;
  u64 loc = site;
  if (loc >= ix.N) { loc = ix.N * 2 - (loc + end_site) - 1; p.reverse = 1; }
  else { loc = loc + (u64)start_site; p.reverse = 0; }
  // the chromosome whose [start, end] holds loc (the reference scans the table; chromosomes are contiguous, so the last one
  // that starts at or before loc is the only candidate); when nothing holds it: the last entry, where the reference's scan ends
  u32 lo = 0, hi = ix.n_chrom;                   // chrom_start[n_chrom] = N
  while (hi - lo > 1) { const u32 mid = (lo + hi) >> 1; if (__ldg(ix.chrom_start + mid) <= loc) lo = mid; else hi = mid; }
  u64 cs = __ldg(ix.chrom_start + lo), ce = __ldg(ix.chrom_start + lo + 1);
  if (!(loc >= cs && loc < ce)) { lo = ix.n_chrom - 1; cs = __ldg(ix.chrom_start + lo); ce = __ldg(ix.chrom_start + lo + 1); }
  p.chrom = lo;
  p.pos = loc + 1 - cs;
  p.off = p.pos + end_site - (u64)start_site > ce - cs;
  return p;
}

constexpr int FIN_MM = 32;           // mismatch positions kept per read (err <= 31)
constexpr u32 FIN_INF = 0xFFFFu;
constexpr int FIN_SORT_CAP = 2048;   // longest window list finish_sorted replays (one warp, keys in shared memory)
constexpr int FIN_SORT_WARPS = 3;    // warps per block there: 12 KB of shared memory each
constexpr u32 FIN_SHORT = 16;        // window lists up to this long are finished by their own thread (std::sort = stable insertion sort)
constexpr u32 FIN_THREAD_MAX = 64;    // up to here the read's own thread reduces the list (finish_se)
constexpr u32 FIN_WARP_MAX = 1024;   // up to here a warp reduces the list (finish_long), beyond a block (finish_huge)

__device__ __forceinline__ bmbs_final fin_blank(u32 k) {
  bmbs_final o; o.site = 0; o.chrom_pos = 0; o.aux_first = 0; o.end_site = 0; o.nm = 0; o.sbd = 255; o.status = BMBS_FIN_UNMAPPED;
  o.flags = 0; o.mapq_fixed = 0; o.k = (uint8_t)k; o.n_aux = 0;
  return o;
}
__device__ __forceinline__ void fin_set_place(bmbs_final& o, const PlacedDev& p) {
  if (p.off) { o.status = BMBS_FIN_UNMAPPED; return; }
  o.status = BMBS_FIN_UNIQUE;
  o.chrom_pos = ((u64)p.chrom << 40) | (p.pos & 0xFFFFFFFFFFull);
  o.flags |= (uint8_t)p.reverse;
}
__device__ __forceinline__ u64 end_abs(const bmbs_cand& x) { return x.site + (u64)(long long)x.end_site; }

// Mismatches of read bases [32 ch, 32 ch + 32) against the double-strand sequence from `pos` on, one bit per base: the read's
// bit-planes (pack_reads) against two funnel-shifted words of the genome planes; read T on genome C is a match, a read base
// that is not A/C/G/T matches nothing.
__device__ __forceinline__ u32 diagonal_mismatch_bits(const DevIndex& ix, const uint4* __restrict__ rpl, u64 pos, u32 ch, u32 L) {
  const uint4 r = rpl[ch];
  const u64 p = pos + 32ull * ch;
  const uint2 g0 = __ldg(ix.planes + (p >> 5)), g1 = __ldg(ix.planes + (p >> 5) + 1);
  const unsigned sh = (unsigned)p & 31u;
  const u32 glo = __funnelshift_r(g0.x, g1.x, sh), ghi = __funnelshift_r(g0.y, g1.y, sh);
  const u32 same = ~(r.x ^ glo) & ~(r.y ^ ghi), t_on_c = r.x & r.y & glo & ~ghi;
  const u32 left = L - 32u * ch, valid = left >= 32u ? 0xFFFFFFFFu : (1u << left) - 1u;
  return ~((same | t_on_c) & ~r.z) & valid;
}

// The chosen window -> the read's record, by one thread: try_cigar_without_path on the window's diagonal that ends at end_site
// (exactly err mismatches = ungapped, their read positions into mm[]), then the coordinates.  Returns the number of positions.
// A hit that runs over the end of its chromosome leaves the read unmapped; with KEEP_OFF_END (the mates of a pair) it keeps its
// coordinates, because the caller's span check over both mates drops the pair.  A template flag rather than an argument keeps
// finish_pe's register count.
template <bool KEEP_OFF_END>
__device__ __forceinline__ u32 finish_hit(const DevIndex& ix, const BatchView& b, int r, u32 L, u32 k, const bmbs_cand x, unsigned short* mm, bmbs_final& o) {
  o.site = x.site; o.end_site = x.end_site; o.nm = (uint8_t)x.err;
  const int start = (int)x.end_site - (int)L + 1;
  u32 mm_n = 0;
  if (x.err != 0) {
    bool ok = start >= 0 && window_inside(ix, x.site, (u64)L + 2ull * k);
    if (ok) {
      const uint4* rpl = b.rplanes + plane_chunk_offset(b.offsets, r);
      for (u32 ch = 0; ch * 32u < L && mm_n <= x.err; ++ch) {
        u32 mis = diagonal_mismatch_bits(ix, rpl, x.site + (u64)(long long)start, ch, L);
        while (mis) { const u32 bit = (u32)__ffs(mis) - 1u; mis &= mis - 1u; if (mm_n < (u32)FIN_MM) mm[mm_n] = (unsigned short)(32u * ch + bit); ++mm_n; }
      }
      ok = mm_n == x.err;
    }
    if (!ok) { o.status = BMBS_FIN_DP; return 0; }
  }
  PlacedDev p = place_hit(ix, x.site, start, (u64)(long long)x.end_site);
  if (KEEP_OFF_END) p.off = false;
  fin_set_place(o, p);
  return o.status == BMBS_FIN_UNIQUE ? mm_n : 0u;
}

// lane 0 finishes hit x into o and mm[]; every lane returns the number of positions and gets o.status
__device__ __forceinline__ u32 warp_finish_hit(const DevIndex& ix, const BatchView& b, int r, u32 L, u32 k, const bmbs_cand& x, unsigned short* mm, bmbs_final& o, int lane) {
  u32 mm_n = 0;
  if (lane == 0) mm_n = finish_hit<false>(ix, b, r, L, k, x, mm, o);
  o.status = (uint8_t)__shfl_sync(0xffffffffu, (u32)o.status, 0);
  return __shfl_sync(0xffffffffu, mm_n, 0);
}

// n entries for each lane of a full warp from *counter, with one atomicAdd per warp; returns the lane's first entry
__device__ __forceinline__ unsigned long long warp_reserve(unsigned long long* counter, u32 n) {
  const int lane = threadIdx.x & 31;
  u32 inc = n;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  const u32 tot = __shfl_sync(0xffffffffu, inc, 31);
  unsigned long long base = 0;
  if (lane == 0 && tot) base = atomicAdd(counter, (unsigned long long)tot);
  return __shfl_sync(0xffffffffu, base, 0) + inc - n;
}

// the next work item of a persistent warp, from a FinCounters cursor
__device__ __forceinline__ u32 warp_next(unsigned long long* cursor) {
  u32 i = 0;
  if ((threadIdx.x & 31) == 0) i = (u32)atomicAdd(cursor, 1ull);
  return __shfl_sync(0xffffffffu, i, 0);
}

// One thread per read.  Reads that seeding resolved and window lists of up to FIN_THREAD_MAX entries are finished here (two
// passes over the list; up to FIN_SHORT windows in std::sort's stable order, beyond that when the order cannot matter, else
// the read goes to finish_sorted); longer lists go to finish_long / finish_huge.
__global__ void __launch_bounds__(128) finish_se(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  __shared__ unsigned short s_mm[128][FIN_MM + 1];
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = r < b.n_reads;
  bmbs_read_result res; res.state = BMBS_NONE; res.first_cand = 0; res.n_cand = 0; res.site = 0; res.one_mismatch_pos = 0; res.is_multiple_map = 0;
  u32 L = 0, k = 0;
  if (live) { res = b.out_res[r]; L = b.len[r]; k = b.kk[r]; }
  bmbs_final o = fin_blank(k);
  unsigned short* mm = s_mm[threadIdx.x];
  u32 my_mm = 0;
  bool is_long = false, to_sort = false;
  if (live) {
    if (res.state == BMBS_EXACT_UNIQUE) {
      o.site = res.site; o.end_site = (int16_t)(L - 1); o.mapq_fixed = 42;
      fin_set_place(o, place_hit(ix, res.site, 0, L - 1));
    } else if (res.state == BMBS_ONE_MISMATCH) {
      o.site = res.site; o.end_site = (int16_t)(L - 1); o.nm = 1;
      fin_set_place(o, place_hit(ix, res.site, 0, L - 1));
      if (o.status == BMBS_FIN_UNIQUE) { mm[0] = (unsigned short)res.one_mismatch_pos; my_mm = 1; }
    } else if (res.state == BMBS_MULTI_EXACT) {
      if (!b.amb_out) o.status = BMBS_FIN_AMBIGUOUS;
      else {      // the first located row (suffix-array order) that stays inside a chromosome, MAPQ 1 (Schema.cpp:27216-27245)
        for (u32 j = 0; j < res.n_cand; ++j) {
          const u64 site = b.out_cand[res.first_cand + j].site;
          const PlacedDev p = place_hit(ix, site, 0, L - 1);
          if (!p.off) { o.site = site; o.end_site = (int16_t)(L - 1); o.mapq_fixed = 1; o.flags |= BMBS_FINF_AMBIGUOUS; fin_set_place(o, p); break; }
        }
      }
    } else if (res.state == BMBS_VERIFY) {
      const u32 n = res.n_cand;
      if (n > FIN_THREAD_MAX) is_long = true;
      else {
        const bmbs_cand* __restrict__ c = b.out_cand + res.first_cand;
        // pass 1: smallest err and, among the hits that have it, the largest vote -- one minimum over (err, ~vote)
        u32 key = 0xFFFFFFFFu;
        for (u32 j = 0; j < n; ++j) { const bmbs_cand x = c[j]; key = min(key, (u32)x.err << 16 | (0xFFFFu - min(x.vote, 0xFFFFu))); }
        const u32 m = key >> 16, vstar = 0xFFFFu - (key & 0xFFFFu);
        if (n && m != FIN_INF) {
          // pass 2: the first top-voted hit with that err and how many there are, whether all hits with that err end at the same
          // place, the smallest err voted higher (A), voted the same (B) and voted the same ahead of the hit (Bs)
          u32 i_top = 0xFFFFFFFFu, cnt_top = 0, A = FIN_INF, B = FIN_INF, Bs = FIN_INF;
          u64 e_min = ~0ull, e_max = 0;
          for (u32 j = 0; j < n; ++j) {
            const bmbs_cand y = c[j];
            if (y.err == m) { const u64 e = end_abs(y); e_min = min(e_min, e); e_max = max(e_max, e); if (y.vote == vstar) { ++cnt_top; if (i_top == 0xFFFFFFFFu) i_top = j; } }
            else if (y.vote > vstar) A = min(A, (u32)y.err);
            else if (y.vote == vstar) { B = min(B, (u32)y.err); if (i_top == 0xFFFFFFFFu) Bs = min(Bs, (u32)y.err); }
          }
          const bool amb = e_min != e_max;
          if (amb && !b.amb_out) o.status = BMBS_FIN_AMBIGUOUS;
          else {
            u32 before = A;
            bool sort_it = false;
            if (n <= FIN_SHORT) before = min(A, Bs);          // std::sort is a stable insertion sort: equal votes stay in site order
            else if (cnt_top > 1 && (m != 0 || amb)) { sort_it = true; atomicAdd(&f.fc->n_unc_idx, 1ull); }
            else if (!amb && B < A) { sort_it = true; atomicAdd(&f.fc->n_unc_sbd, 1ull); }
            if (sort_it) to_sort = true;
            else {
              if (amb) { o.sbd = 0; o.flags |= BMBS_FINF_AMBIGUOUS; }
              else o.sbd = (uint8_t)(before == FIN_INF ? 255u : min(before - m, 255u));
              my_mm = finish_hit<false>(ix, b, r, L, k, c[i_top], mm, o);
            }
          }
        }
      }
    }
  }
  // window lists whose order decides go to finish_sorted; longer lists to finish_long (a warp each) and finish_huge (a block each)
  const bool is_huge = is_long && res.n_cand > FIN_WARP_MAX;
  list_append(f.sort_list, &f.fc->n_sorted, to_sort, (u32)r);
  list_append(f.long_list, &f.fc->n_long, is_long && !is_huge, (u32)r);
  list_append(f.huge_list, &f.fc->n_huge, is_huge, (u32)r);
  {
    const u32 mdp = __ballot_sync(0xffffffffu, live && o.status == BMBS_FIN_DP);
    if (lane == 0 && mdp) atomicAdd(&f.fc->n_dp, (unsigned long long)__popc(mdp));
  }
  const unsigned long long at = warp_reserve(&f.fc->mism_used, my_mm);
  if (my_mm) {
    o.aux_first = (u32)at; o.n_aux = my_mm;
    if (at + my_mm <= f.mism_cap) for (u32 j = 0; j < my_mm; ++j) f.mism[at + j] = mm[j];
  }
  if (live && !is_long && !to_sort) f.fin[r] = o;
}

// what a warp leaves behind for its read: the record, its mismatch positions, or the whole window list for the host
__device__ __forceinline__ void fin_store(const FinishView& f, int r, bmbs_final o, u32 mm_n, const unsigned short* mm, const bmbs_cand* __restrict__ c, u32 n, int lane) {
  unsigned long long at = 0;
  if (o.status == BMBS_FIN_HOST) {
    if (lane == 0) { at = atomicAdd(&f.fc->fb_used, (unsigned long long)n); atomicAdd(&f.fc->n_host, 1ull); }
    at = __shfl_sync(0xffffffffu, at, 0);
    o.aux_first = (u32)at; o.n_aux = n;
    if (at + n <= f.fb_cap) for (u32 j = lane; j < n; j += 32) f.fb[at + j] = c[j];
  } else if (mm_n) {
    if (lane == 0) at = atomicAdd(&f.fc->mism_used, (unsigned long long)mm_n);
    at = __shfl_sync(0xffffffffu, at, 0);
    o.aux_first = (u32)at; o.n_aux = mm_n;
    if (at + mm_n <= f.mism_cap && (u32)lane < mm_n) f.mism[at + lane] = mm[lane];
  }
  if (lane == 0) { if (o.status == BMBS_FIN_DP) atomicAdd(&f.fc->n_dp, 1ull); f.fin[r] = o; }
}

// The group of threads that works on one long window list: a warp (lists of up to FIN_WARP_MAX windows) or a whole block.
struct WarpGroup {
  static constexpr u32 SIZE = 32;
  __device__ __forceinline__ static u32 id() { return threadIdx.x & 31u; }
  __device__ __forceinline__ static u32 rmin(u32 v, u32*) { return __reduce_min_sync(0xffffffffu, v); }
  __device__ __forceinline__ static u32 rmax(u32 v, u32*) { return __reduce_max_sync(0xffffffffu, v); }
  __device__ __forceinline__ static u32 radd(u32 v, u32*) { return __reduce_add_sync(0xffffffffu, v); }
  __device__ __forceinline__ static void sync() { __syncwarp(); }
};
struct BlockGroup {      // 256 threads
  static constexpr u32 SIZE = 256;
  __device__ __forceinline__ static u32 id() { return threadIdx.x; }
  template <int OP> __device__ __forceinline__ static u32 red(u32 v, u32* sh) {
    v = OP == 0 ? __reduce_min_sync(0xffffffffu, v) : OP == 1 ? __reduce_max_sync(0xffffffffu, v) : __reduce_add_sync(0xffffffffu, v);
    __syncthreads();
    if ((threadIdx.x & 31u) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    u32 t = sh[threadIdx.x & 7u];
    t = OP == 0 ? __reduce_min_sync(0xffffffffu, t) : OP == 1 ? __reduce_max_sync(0xffffffffu, t) : __reduce_add_sync(0xffffffffu, (threadIdx.x & 31u) < 8u ? t : 0u);
    return t;
  }
  __device__ __forceinline__ static u32 rmin(u32 v, u32* sh) { return red<0>(v, sh); }
  __device__ __forceinline__ static u32 rmax(u32 v, u32* sh) { return red<1>(v, sh); }
  __device__ __forceinline__ static u32 radd(u32 v, u32* sh) { return red<2>(v, sh); }
  __device__ __forceinline__ static void sync() { __syncthreads(); }
};

// Order-free part of the reduction over one window list, by a group of threads: four passes of reductions say what the
// outcome is whenever the order among equal votes cannot change it -- it cannot when the best hit is the only top-voted one
// with its err (or err 0: every such window is the same alignment) and no hit of the same vote has an err below everything
// voted higher.  Returns 0: o is the read's record up to the chosen window `xt` (caller finishes the hit when o.status is
// BMBS_FIN_UNIQUE), 1: the order decides.
template <class G>
__device__ __forceinline__ int reduce_order_free(const BatchView& b, const bmbs_cand* __restrict__ c, u32 n, bmbs_final& o, bmbs_cand& xt, u32* sh, FinCounters* fc) {
  const u32 id = G::id();
  u32 m = FIN_INF;
  for (u32 j = id; j < n; j += G::SIZE) m = min(m, (u32)c[j].err);
  m = G::rmin(m, sh);
  if (m == FIN_INF) return 0;                                      // nothing within k: unmapped
  u32 vstar = 0;
  for (u32 j = id; j < n; j += G::SIZE) { const bmbs_cand x = c[j]; if (x.err == m) vstar = max(vstar, x.vote); }
  vstar = G::rmax(vstar, sh);
  // the top-voted hits with that err and the first of them; the smallest err voted higher (A) and voted the same (B)
  u32 cnt_top = 0, i_top = 0xFFFFFFFFu, A = FIN_INF, B = FIN_INF;
  for (u32 j = id; j < n; j += G::SIZE) {
    const bmbs_cand x = c[j];
    if (x.err == m) { if (x.vote == vstar) { ++cnt_top; i_top = min(i_top, j); } }
    else if (x.vote > vstar) A = min(A, (u32)x.err);
    else if (x.vote == vstar) B = min(B, (u32)x.err);
  }
  cnt_top = G::radd(cnt_top, sh); i_top = G::rmin(i_top, sh); A = G::rmin(A, sh); B = G::rmin(B, sh);
  xt = c[i_top];
  const u64 e0 = end_abs(xt);
  u32 amb = 0;
  for (u32 j = id; j < n; j += G::SIZE) { const bmbs_cand x = c[j]; if (x.err == m) amb |= (u32)(end_abs(x) != e0); }
  amb = G::rmax(amb, sh);
  if (amb && !b.amb_out) { o.status = BMBS_FIN_AMBIGUOUS; return 0; }
  if (cnt_top > 1 && (m != 0 || amb)) { if (id == 0) atomicAdd(&fc->n_unc_idx, 1ull); return 1; }   // which of the equal hits comes first decides the window
  if (!amb && B < A) { if (id == 0) atomicAdd(&fc->n_unc_sbd, 1ull); return 1; }                    // a worse hit with the same vote may or may not come first
  if (amb) { o.sbd = 0; o.flags |= BMBS_FINF_AMBIGUOUS; }
  else o.sbd = (uint8_t)(A == FIN_INF ? 255u : min(A - m, 255u));
  o.status = BMBS_FIN_UNIQUE;                                      // provisional: finish_hit decides
  return 0;
}

// One warp per read of long_list (window lists of FIN_THREAD_MAX+1 .. FIN_WARP_MAX entries; reads taken from a shared
// cursor).  Reads whose outcome the order cannot change are finished here, the others go to finish_sorted.
__global__ void __launch_bounds__(128) finish_long(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  __shared__ unsigned short s_mm[4][FIN_MM + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const u32 n_list = (u32)f.fc->n_long;
  for (;;) {
    const u32 i = warp_next(&f.fc->cursor_long);
    if (i >= n_list) break;
    const int r = (int)f.long_list[i];
    const bmbs_read_result res = b.out_res[r];
    const u32 n = res.n_cand, L = b.len[r], k = b.kk[r];
    const bmbs_cand* __restrict__ c = b.out_cand + res.first_cand;
    bmbs_final o = fin_blank(k);
    bmbs_cand xt; xt.site = 0; xt.vote = 0; xt.end_site = 0; xt.err = 0;
    u32 mm_n = 0;
    const int sort_it = reduce_order_free<WarpGroup>(b, c, n, o, xt, nullptr, f.fc);
    if (sort_it) {
      if (lane == 0) f.sort_list[atomicAdd(&f.fc->n_sorted, 1ull)] = (u32)r;     // n <= FIN_WARP_MAX <= FIN_SORT_CAP
    } else {
      if (o.status == BMBS_FIN_UNIQUE) mm_n = warp_finish_hit(ix, b, r, L, k, xt, s_mm[w], o, lane);   // lane 0 holds the record; the others help with the copies
      __syncwarp();
      fin_store(f, r, o, mm_n, s_mm[w], c, n, lane);
    }
    __syncwarp();
  }
}

// One block per read of huge_list (more than FIN_WARP_MAX windows -- reads out of high-copy repeats, up to 25 x 1000).  Such a
// list is beyond the sort replay: when the order decides, the read goes back to the host with its list.
__global__ void __launch_bounds__(256) finish_huge(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  __shared__ unsigned short s_mm[FIN_MM + 1];
  __shared__ u32 s_red[8];
  __shared__ u32 s_i;
  const u32 n_list = (u32)f.fc->n_huge;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_i = (u32)atomicAdd(&f.fc->cursor_huge, 1ull);
    __syncthreads();
    const u32 i = s_i;
    if (i >= n_list) break;
    const int r = (int)f.huge_list[i];
    const bmbs_read_result res = b.out_res[r];
    const u32 n = res.n_cand, L = b.len[r], k = b.kk[r];
    const bmbs_cand* __restrict__ c = b.out_cand + res.first_cand;
    bmbs_final o = fin_blank(k);
    bmbs_cand xt; xt.site = 0; xt.vote = 0; xt.end_site = 0; xt.err = 0;
    const int sort_it = reduce_order_free<BlockGroup>(b, c, n, o, xt, s_red, f.fc);
    if (sort_it && n <= (u32)FIN_SORT_CAP) {
      if (threadIdx.x == 0) f.sort_list[atomicAdd(&f.fc->n_sorted, 1ull)] = (u32)r;
    } else if (threadIdx.x < 32) {      // the first warp writes the record
      const int lane = threadIdx.x;
      u32 mm_n = 0;
      if (sort_it) { o = fin_blank(k); o.status = BMBS_FIN_HOST; o.site = res.is_multiple_map; }
      else if (o.status == BMBS_FIN_UNIQUE) mm_n = warp_finish_hit(ix, b, r, L, k, xt, s_mm, o, lane);
      __syncwarp();
      fin_store(f, r, o, mm_n, s_mm, c, n, lane);
    }
  }
}

// std::sort's partition phase on key[0..n) (u16: vote << 11 | position in the list), by a whole warp, step for step what
// bmbs_sort_replay.h does sequentially (that header is checked against std::sort on the CPU; this routine against std::sort
// through bmbs_debug_sort_order on the GPU).  One unguarded Hoare partition = the t-th element from the left that is not
// before the pivot swaps with the t-th element from the right that is not after it, for as long as the two have not met
// (positions untouched by earlier swaps are all the scan ever stops at, so the pairs can be formed up front): both stopper
// lists are compacted with ballots, the number of swaps T is where the lists cross, the T swaps are independent, and the cut is
// the first stopper the left scan would meet next.  Ranges of <= 16 are left as they are: the final insertion sort is stable,
// i.e. equal votes stay in the order the partitions left them, which is all the callers need.
__device__ __forceinline__ u32 key_vote(unsigned short k) { return (u32)k >> 11; }
__device__ bool warp_replay_partitions(unsigned short* key, int n, unsigned short* posL, unsigned short* posR, u32* stack, int lane) {
  if (n <= 16) return true;
  const u32 lt = (1u << lane) - 1u;
  int sp = 1;
  if (lane == 0) stack[0] = (u32)n << 12 | (u32)(2 * (31 - __clz(n))) << 24;
  __syncwarp();
  while (sp) {
    --sp;
    const u32 e = stack[sp];
    int first = (int)(e & 0xFFFu), last = (int)((e >> 12) & 0xFFFu), depth = (int)(e >> 24);
    __syncwarp();
    while (last - first > 16) {
      if (depth == 0 || sp >= 31) return false;
      --depth;
      const int ia = first + 1, ib = first + (last - first) / 2, ic = last - 1;       // __move_median_to_first
      const u32 va = key_vote(key[ia]), vb = key_vote(key[ib]), vc = key_vote(key[ic]);
      int pick;
      if (va > vb) { if (vb > vc) pick = ib; else if (va > vc) pick = ic; else pick = ia; }
      else if (va > vc) pick = ia;
      else if (vb > vc) pick = ic;
      else pick = ib;
      __syncwarp();
      if (lane == 0) { const unsigned short t = key[first]; key[first] = key[pick]; key[pick] = t; }
      __syncwarp();
      const u32 vp = key_vote(key[first]);
      const int lo0 = first + 1, s = last - lo0;
      int nL = 0, nR = 0;
      for (int base = 0; base < s; base += 32) {
        const int o = base + lane;
        bool isL = false, isR = false;
        if (o < s) { isL = key_vote(key[lo0 + o]) <= vp; isR = key_vote(key[last - 1 - o]) >= vp; }
        const u32 mL = __ballot_sync(0xffffffffu, isL), mR = __ballot_sync(0xffffffffu, isR);
        if (isL) posL[nL + __popc(mL & lt)] = (unsigned short)(lo0 + o);
        if (isR) posR[nR + __popc(mR & lt)] = (unsigned short)(last - 1 - o);
        nL += __popc(mL); nR += __popc(mR);
      }
      __syncwarp();
      int T = 0; const int nmin = min(nL, nR);
      for (int base = 0; base < nmin; base += 32) {
        const int t = base + lane;
        const u32 m = __ballot_sync(0xffffffffu, t < nmin && posL[t] < posR[t]);
        T += __popc(m);
        if (m != 0xffffffffu) break;
      }
      for (int t = lane; t < T; t += 32) { const int i = posL[t], j = posR[t]; const unsigned short x = key[i]; key[i] = key[j]; key[j] = x; }
      const int cut = min(T < nL ? (int)posL[T] : 0x7fffffff, T >= 1 ? (int)posR[T - 1] : 0x7fffffff);
      __syncwarp();
      if (lane == 0) stack[sp] = (u32)cut | (u32)last << 12 | (u32)depth << 24;
      ++sp;
      last = cut;
      __syncwarp();
    }
  }
  return true;
}

// One warp per read of sort_list: the window list as (vote << 11 | position) keys in shared memory, the partition phase of
// std::sort replayed, then the reference's walk in the resulting order -- among the hits with the smallest err the one that
// comes first (largest vote, then earliest place after the partitions) is the hit, the smallest err in front of it is where
// the running minimum stood (second_best_diff), a hit with the same err and another end makes it ambiguous.
__global__ void __launch_bounds__(32 * FIN_SORT_WARPS) finish_sorted(DevIndex ix, BatchView b, FINISH_PARAMS) {
  const FinishView f = FINISH_VIEW;
  __shared__ unsigned short s_key[FIN_SORT_WARPS][FIN_SORT_CAP], s_posL[FIN_SORT_WARPS][FIN_SORT_CAP], s_posR[FIN_SORT_WARPS][FIN_SORT_CAP];
  __shared__ u32 s_stack[FIN_SORT_WARPS][32];
  __shared__ unsigned short s_mm[FIN_SORT_WARPS][FIN_MM + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const u32 n_list = (u32)f.fc->n_sorted;
  for (;;) {
    const u32 i = warp_next(&f.fc->cursor_sorted);
    if (i >= n_list) break;
    const int r = (int)f.sort_list[i];
    const bmbs_read_result res = b.out_res[r];
    const u32 n = res.n_cand, L = b.len[r], k = b.kk[r];
    const bmbs_cand* __restrict__ c = b.out_cand + res.first_cand;
    unsigned short* key = s_key[w];
    u32 m = FIN_INF, vmax = 0;
    for (u32 j = lane; j < n; j += 32) { const bmbs_cand x = c[j]; key[j] = (unsigned short)((x.vote & 31u) << 11 | j); m = min(m, (u32)x.err); vmax = max(vmax, x.vote); }
    m = __reduce_min_sync(0xffffffffu, m); vmax = __reduce_max_sync(0xffffffffu, vmax);
    __syncwarp();
    const bool ok = vmax < 32u && warp_replay_partitions(key, (int)n, s_posL[w], s_posR[w], s_stack[w], lane);
    __syncwarp();
    bmbs_final o = fin_blank(k);
    u32 mm_n = 0;
    if (!ok) { o.status = BMBS_FIN_HOST; o.site = res.is_multiple_map; }
    else {
      // the hit: smallest err, largest vote, earliest place; ahead of it: every larger vote, and the equal votes placed before it
      u32 vstar = 0;
      for (u32 j = lane; j < n; j += 32) { const bmbs_cand x = c[j]; if (x.err == m) vstar = max(vstar, x.vote); }
      vstar = __reduce_max_sync(0xffffffffu, vstar);
      u32 p_hit = 0xFFFFFFFFu;
      for (u32 p = lane; p < n; p += 32) { const bmbs_cand x = c[key[p] & 0x7FFu]; if (x.err == m && x.vote == vstar) p_hit = min(p_hit, p); }
      p_hit = __reduce_min_sync(0xffffffffu, p_hit);
      const bmbs_cand x = c[key[p_hit] & 0x7FFu];
      const u64 e0 = end_abs(x);
      u32 before = FIN_INF, amb = 0;
      for (u32 p = lane; p < n; p += 32) {
        const bmbs_cand y = c[key[p] & 0x7FFu];
        if (y.err == m) amb |= (u32)(end_abs(y) != e0);
        else if (y.vote > vstar || (y.vote == vstar && p < p_hit)) before = min(before, (u32)y.err);
      }
      before = __reduce_min_sync(0xffffffffu, before);
      amb = __any_sync(0xffffffffu, amb != 0) ? 1u : 0u;
      if (amb && !b.amb_out) o.status = BMBS_FIN_AMBIGUOUS;
      else {
        if (amb) { o.sbd = 0; o.flags |= BMBS_FINF_AMBIGUOUS; }
        else o.sbd = (uint8_t)(before == FIN_INF ? 255u : min(before - m, 255u));
        mm_n = warp_finish_hit(ix, b, r, L, k, x, s_mm[w], o, lane);
      }
    }
    __syncwarp();
    fin_store(f, r, o, mm_n, s_mm[w], c, n, lane);
    __syncwarp();
  }
}

#include "bmbs_finish_pe.cuh"

// Test entry (bmbs_debug_sort_order): the order std::sort by vote leaves each list in, through the same warp routine -- the
// partition phase, then the stable final pass as a counting sort by vote (rank = larger votes + equal votes placed earlier).
__global__ void __launch_bounds__(32 * FIN_SORT_WARPS) debug_sort_order(const u32* __restrict__ votes, const u32* __restrict__ offsets, u32 n_lists, unsigned short* __restrict__ order, int* __restrict__ okflag) {
  __shared__ unsigned short s_key[FIN_SORT_WARPS][FIN_SORT_CAP], s_posL[FIN_SORT_WARPS][FIN_SORT_CAP], s_posR[FIN_SORT_WARPS][FIN_SORT_CAP];
  __shared__ u32 s_stack[FIN_SORT_WARPS][32];
  __shared__ u32 s_base[FIN_SORT_WARPS][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const u32 warps = gridDim.x * (blockDim.x >> 5);
  for (u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_lists; i += warps) {
    const u32 off = offsets[i], n = offsets[i + 1] - off;
    unsigned short* key = s_key[w];
    for (u32 j = lane; j < n; j += 32) key[j] = (unsigned short)((votes[off + j] & 31u) << 11 | j);
    __syncwarp();
    const bool ok = warp_replay_partitions(key, (int)n, s_posL[w], s_posR[w], s_stack[w], lane);
    if (lane == 0) okflag[i] = ok ? 1 : 0;
    // histogram of the votes, first rank of every vote (descending)
    u32 cnt = 0;
    for (u32 p = 0; p < n; ++p) cnt += key_vote(key[p]) == (u32)lane;
    u32 above = 0;
    for (int v = 31; v >= 0; --v) { const u32 t = __shfl_sync(0xffffffffu, cnt, v); if (v > lane) above += t; }
    s_base[w][lane] = above;
    __syncwarp();
    for (u32 base = 0; base < n; base += 32) {
      const u32 p = base + lane;
      const bool live = p < n;
      const u32 v = live ? key_vote(key[p]) : 32u + (u32)lane;
      const u32 peers = __match_any_sync(0xffffffffu, v);
      if (live) {
        const u32 dest = s_base[w][v] + __popc(peers & ((1u << lane) - 1u));
        order[off + dest] = key[p] & 0x7FFu;
      }
      __syncwarp();
      if (live && (peers & ((1u << lane) - 1u)) == 0) s_base[w][v] += __popc(peers);
      __syncwarp();
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------- scan
// exclusive scan of u32 counts into u32 offsets (out[n] = total); 0xFFFFFFFF inputs count as 0 and set *overflow.
constexpr int SCAN_TILE = 1024;
__global__ void scan_tiles(const u32* in, u32 n, u64* tile_sum, u32* overflow) {
  __shared__ u64 s_w[32];
  const u32 i = blockIdx.x * SCAN_TILE + threadIdx.x;
  u32 v = i < n ? in[i] : 0u;
  if (v == 0xFFFFFFFFu) { v = 0; atomicOr(overflow, 1u); }
  u64 x = v;
  for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = x;
  __syncthreads();
  if (threadIdx.x < 32) {
    u64 y = s_w[threadIdx.x];
    for (int o = 16; o; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = y;
  }
}
__global__ void scan_tile_sums(u64* tile_sum, u32 ntiles, u64* total, u64 cap, u32* status, u32 cap_bit, const u64* base) {
  // single block, serial over chunks of blockDim
  __shared__ u64 s_carry; __shared__ u64 s_w[32];
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (u32 base = 0; base < ntiles; base += blockDim.x) {
    const u32 i = base + threadIdx.x;
    const u64 v = i < ntiles ? tile_sum[i] : 0ull;
    u64 x = v;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) { const u64 y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_w[wid] = x;
    __syncthreads();
    u64 wbase = 0; for (int w2 = 0; w2 < wid; ++w2) wbase += s_w[w2];
    const u64 incl = s_carry + wbase + x;
    if (i < ntiles) tile_sum[i] = incl - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) s_carry = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) { *total = s_carry; if (s_carry + (base ? *base : 0ull) > cap) atomicOr(status, cap_bit); }
}
__global__ void scan_apply(const u32* in, u32 n, const u64* tile_sum, u32* out) {
  __shared__ u32 s_w[32];
  const u32 i = blockIdx.x * SCAN_TILE + threadIdx.x;
  u32 v = i < n ? in[i] : 0u;
  if (v == 0xFFFFFFFFu) v = 0;
  u32 x = v;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) s_w[wid] = x;
  __syncthreads();
  u32 wbase = 0; for (int w2 = 0; w2 < wid; ++w2) wbase += s_w[w2];
  const u64 excl = tile_sum[blockIdx.x] + wbase + x - v;
  if (i < n) out[i] = (u32)(excl > 0xFFFFFFFFull ? 0xFFFFFFFFull : excl);
  if (i == n - 1) { const u64 t = excl + v; out[n] = (u32)(t > 0xFFFFFFFFull ? 0xFFFFFFFFull : t); }
}

}  // namespace bmbs
