/* bmbs.h -- C ABI of libbmbs_gpu.so: BitMapperBS's seed-and-verify hot path on B200.
 *
 * The reference has no plugin/FFI interface; its worker threads call the hot
 * functions inline over process globals.  Each entry point below names the
 * reference seam it replaces (file:line into chhylp123/BitMapperBS v1.0.2.3):
 *
 *   bmbs_index_load / _free      Start_Load_Index + Load_Index (Index.cpp:1048, :940) and
 *                                load_index (bwt.cpp:2458): same six on-disk files, read as-is.
 *   bmbs_map_batch_se            per-read body of Map_Single_Seq_split (Schema.cpp:27077-27752)
 *                                up to, not including, the vote-ordered reduction and CIGAR:
 *                                C_to_T_forward (Schema.h:1534), count_backward_as_much_1_terminate
 *                                (bwt.h:2081), count_hash_table (bwt.h:1848), locate_muti_thread
 *                                (bwt.cpp:4986) / locate_one_position_direct (bwt.h:2585),
 *                                try_process_unique_mismatch_end_to_end_output_buffer
 *                                (Schema.cpp:15410), std::sort + generate_candidate_votes_shift
 *                                (Schema.cpp:27599, :4687), get_actuall_genome/_rc_genome
 *                                (Schema.cpp:4998, :5061) + BS_Reserve_Banded_BPM{,_4_SSE,_8_SSE}
 *                                (Levenshtein_Cal.h:351, :1678, :2093).
 *   bmbs_map_batch_pe            the same for Map_Pair_Seq_split_fast (Schema.cpp:21856-22382):
 *                                get_candidates_muti_thread (:19550) for both mates, filter_pairs
 *                                (:16052) and verification of every surviving candidate.
 *   bmbs_verify                  BS_Reserve_Banded_BPM over caller-supplied (read, site) pairs.
 *
 * Conventions: plain pointers and sizes, caller-owned in/out buffers (pinned
 * host memory makes the copies faster but is not required), library-owned device
 * memory and streams.  Every function returns 0 on success and a negative code
 * on failure with a message in bmbs_last_error(); nothing calls exit().  The
 * index handle is immutable after load and may be shared by any number of host
 * threads; a bmbs_batch / bmbs_refiner (own stream, own device buffers) belongs to
 * one thread at a time, and the one-call forms keep one such context per calling
 * thread -- the reference's -t N workers can all be inside the library at once.
 */
#ifndef BMBS_H
#define BMBS_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define BMBS_OK 0
#define BMBS_ERR_IO (-1)        /* index file missing / short                      */
#define BMBS_ERR_CUDA (-2)      /* CUDA runtime error                              */
#define BMBS_ERR_ARG (-3)       /* bad argument                                    */
#define BMBS_ERR_CAPACITY (-4)  /* caller's output buffer too small; see *_used    */

typedef struct bmbs_index bmbs_index; /* opaque: host metadata + one device copy per GPU */
typedef struct bmbs_batch bmbs_batch; /* opaque: device + pinned staging for one in-flight batch */

/* index_prefix is "<genome.fa>.index" (the name Load_Index opens); devices==NULL means device 0. */
int bmbs_index_load(const char* index_prefix, const int* devices, int n_dev, bmbs_index** out);
void bmbs_index_free(bmbs_index* idx);
uint64_t bmbs_index_genome_length(const bmbs_index* idx);   /* N, bases               */
uint64_t bmbs_index_device_bytes(const bmbs_index* idx);    /* resident HBM per GPU   */
const char* bmbs_last_error(void);

typedef struct {
  double e_rate;      /* -e, default 0.08 (Process_CommandLines.cpp:40)            */
  int seed_len;       /* --seed, default 30                                        */
  int min_ins;        /* --min, default 0                                          */
  int max_ins;        /* --max, default 500                                        */
  int sensitive;      /* 0 = --fast (default); 1 = --sensitive (paired batches)     */
  int ambiguous_out;  /* --ambiguous_out: single-end reads that match exactly at several places (state 2) also get
                         their rows located, in suffix-array row order, at most 1000 (Schema.cpp:26704-26758)  */
} bmbs_params;
void bmbs_params_default(bmbs_params* p);

/* What seeding decided for one read (one mate). */
enum {
  BMBS_NONE = 0,          /* no candidate at all (unmapped)                                        */
  BMBS_EXACT_UNIQUE = 1,  /* unique first seed + error-free direct compare: site, NM 0, CIGAR <L>M */
  BMBS_MULTI_EXACT = 2,   /* whole read matches >1 rows and has no C: SE counts it ambiguous;
                             PE lists all sites as finished hits in cand[]                         */
  BMBS_ONE_MISMATCH = 3,  /* unique hit with exactly one mismatch: site, NM 1, CIGAR <L>M          */
  BMBS_VERIFY = 4         /* cand[] holds the site-sorted windows, each verified                   */
};
typedef struct {
  uint64_t site;            /* states 1 and 3: double-strand coordinate of the read start        */
  uint32_t first_cand;      /* slice of cand[]                                                   */
  uint32_t n_cand;
  int16_t one_mismatch_pos; /* state 3: read index of the mismatch (Schema.cpp:27203)            */
  uint8_t state;
  uint8_t is_multiple_map;  /* first seed was a full-length multi-hit (selects the reduction
                               variant, Schema.cpp:27617-27672)                                   */
  uint32_t reserved;
} bmbs_read_result;         /* 24 bytes */

/* One candidate window [site, site+L+2k) and its verification. */
typedef struct {
  uint64_t site;      /* window start, double-strand coordinate ([0,N) fwd, [N,2N) rc); wraps mod 2^64 like the reference */
  uint32_t vote;      /* number of seeds that voted for it                                           */
  int16_t end_site;   /* last window position of the best alignment, -1 if none within k              */
  uint16_t err;       /* edit distance, 0xFFFF if none within k                                       */
} bmbs_cand;          /* 16 bytes */

/* ---- one-call form (host buffers in, host buffers out) -------------------------------------------
 * seqs: concatenated upper-case ASCII reads; read i is seqs[offsets[i] .. offsets[i+1]).
 * For pairs, reads 2p and 2p+1 are the mates, mate 2 already reverse-complemented
 * (what Process_Reads.cpp:359-369 stores in Read::seq).
 * res[n_reads]; cand[cand_cap]; *cand_used receives the number of entries written (or needed,
 * with BMBS_ERR_CAPACITY). */
int bmbs_map_batch_se(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_reads,
                      const bmbs_params* prm, bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap,
                      size_t* cand_used);
int bmbs_map_batch_pe(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_pairs,
                      const bmbs_params* prm, bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap,
                      size_t* cand_used);

/* Kernel-3 only: verify n (read, site) pairs.  read_idx[i] selects the read, sites[i] the window
 * start; k = min(31, (uint64)(e_rate*L)) per read.  Writes end_site[i], err[i] (0xFFFFFFFF = none). */
int bmbs_verify(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_reads,
                const uint32_t* read_idx, const uint64_t* sites, size_t n, double e_rate,
                int32_t* end_site, uint32_t* err);

/* ---- staged form (what the mapper and bench.py drive; lets copies overlap kernels) --------------- */
int bmbs_batch_create(bmbs_index* idx, int dev, size_t max_reads, size_t max_bases, size_t cand_cap, bmbs_batch** out);
void bmbs_batch_free(bmbs_batch* b);
/* async H2D of the reads into the batch's device buffers (pe: reads come in mate pairs) */
int bmbs_batch_upload(bmbs_batch* b, const char* seqs, const uint64_t* offsets, int n_reads, int pe);
/* enqueue the device pipeline on the batch stream; inputs must have been uploaded */
int bmbs_batch_run(bmbs_batch* b, const bmbs_params* prm);
/* async D2H of results into the caller's buffers, then wait; returns BMBS_ERR_CAPACITY like above */
int bmbs_batch_download(bmbs_batch* b, bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap, size_t* cand_used);
int bmbs_batch_sync(bmbs_batch* b);
/* Wait for the batch, then say how many entries the download call will write, so that the caller can size its buffers first:
 * *n_cand entries of cand[] (bmbs_batch_download: the verified windows of every read; bmbs_batch_download_final after
 * bmbs_batch_finish: the window lists of handed-back reads) and *n_mism mismatch positions (0 unless finished).  Returns what
 * the download would return for the batch itself (BMBS_ERR_CAPACITY with the candidate slots needed in *n_cand). */
int bmbs_batch_output_sizes(bmbs_batch* b, size_t* n_cand, size_t* n_mism);
/* device time of the last bmbs_batch_run in ms (CUDA events on the batch stream), per stage:
 * [0] total [1] pack [2] seed [3] locate [4] votes [5] pair filter [6] verify [7] sensitive pairing + re-seeding round */
int bmbs_batch_timings(bmbs_batch* b, float ms[8]);
/* work counters of the last run, for roofline accounting (SURVEY.md §8d):
 * [0] hash queries [1] occ-block lookups (one interval end, one LF step) [2] located rows
 * [3] locate LF steps [4] verified candidates [5] verified cell updates L*(2k+1) [6] candidates
 * [7] genome-window bytes fetched */
int bmbs_batch_counters(bmbs_batch* b, uint64_t c[8]);
/* Kernel 3 alone (what bmbs_verify does, staged; BASELINE.json config 5): verify n (read, site) items over the
 * reads of the last bmbs_batch_upload; results stay on the device until bmbs_batch_download_verify.
 * bmbs_batch_timings()[6] is the verify_windows launch, bmbs_batch_counters()[5] its cell updates. */
int bmbs_batch_verify(bmbs_batch* b, const uint32_t* read_idx, const uint64_t* sites, size_t n, double e_rate);
int bmbs_batch_download_verify(bmbs_batch* b, int32_t* end_site, uint32_t* err, size_t n);
/* measured peak of the integer ALU pipe on `dev` (LOP3 + IADD3, no dependencies between chains), 32-bit ops/s:
 * the roofline kernel 3 is reported against (SURVEY.md §8d asks for it to be measured, not assumed) */
int bmbs_ubench_int_pipe(int dev, double* ops_per_second);
/* page-locked host memory for the caller's in/out buffers (copies from and to it are asynchronous and run at link speed) */
void* bmbs_pinned_alloc(size_t bytes);
void bmbs_pinned_free(void* p);
/* measured rate of independent 32-byte sector loads at random addresses over `bytes` of device memory, sectors/s: the
 * bound of the seeding kernels, whose work is one table entry / occ block / suffix-array entry per dependent step */
int bmbs_ubench_random_sectors(int dev, size_t bytes, double* sectors_per_second);
/* number of kernels launched by the last bmbs_batch_run */
int bmbs_batch_launches(bmbs_batch* b);
/* test entry: the grids as launched (host values): [0] SMs the persistent and grid-stride launches are sized for (the device's
 * count, or fewer with BMBS_GRID_SMS=n at index load) [1] seed_reads blocks of the last bmbs_batch_run [2] verify_windows blocks
 * of its last launch [3] their block size */
int bmbs_batch_grid(bmbs_batch* b, uint32_t g[4]);


/* ---- finished single-end records (SURVEY.md 8a V3 + 8f-1): reduction, ungapped CIGAR, coordinates on the device -----
 * Replaces, for a single-end batch, what Map_Single_Seq_split does after its verification calls: the vote-ordered reduction
 * (Schema.cpp:27612 std::sort + :7847-8056 / :8325-8745; second_best_diff and the choice among equal hits in exactly the
 * order libstdc++'s std::sort leaves), try_cigar_without_path (ksw.cpp:2515-2570) and the coordinate conversion with the
 * end-of-chromosome drop (Schema.cpp:12596-12650).  One 32-byte record per read comes back instead of the read's whole
 * verified window list.  What stays with the caller: the alignment score of an ungapped hit = sum of
 * MismatchPenaltyByQuality (ksw.h:148-162) over the returned mismatch positions (the quality strings never go to the
 * device), MAP_Calculation on (sbd, k, score), the banded DP of BMBS_FIN_DP reads through bmbs_refine, SAM text. */
enum {
  BMBS_FIN_UNMAPPED = 0,   /* no hit within k, or the hit runs over the end of its chromosome: no record, not counted   */
  BMBS_FIN_UNIQUE = 1,     /* hit without indels, CIGAR <L>M: chrom_pos, strand, nm, mismatch positions, sbd            */
  BMBS_FIN_AMBIGUOUS = 2,  /* equally good hits at different places: counted, no record (without --ambiguous_out)       */
  BMBS_FIN_DP = 3,         /* the chosen window (site, end_site, nm = the verifier's err, sbd) needs the banded DP      */
  BMBS_FIN_HOST = 4        /* handed back: cand[aux_first .. +n_aux) is the read's verified window list, site = is_multiple_map */
};
#define BMBS_FINF_REVERSE 1u    /* SAM flag 16                                                                          */
#define BMBS_FINF_AMBIGUOUS 2u  /* --ambiguous_out: the first of several equally good hits; counted as ambiguous        */
typedef struct {
  uint64_t site;        /* double-strand coordinate of the chosen window (states 1 / 3: of the read)                    */
  uint64_t chrom_pos;   /* BMBS_FIN_UNIQUE: chromosome index << 40 | 1-based POS                                        */
  uint32_t aux_first;   /* BMBS_FIN_UNIQUE: first of n_aux = nm mismatch read positions in mism[]; BMBS_FIN_HOST: in cand[] */
  int16_t end_site;     /* last window position of the alignment (the verifier's)                                       */
  uint8_t nm;           /* mismatches (BMBS_FIN_UNIQUE) / the verifier's err (BMBS_FIN_DP)                              */
  uint8_t sbd;          /* second_best_diff, 255 = none or more (MAP_Calculation only asks whether it exceeds k <= 31)  */
  uint8_t status;       /* BMBS_FIN_*                                                                                    */
  uint8_t flags;        /* BMBS_FINF_*                                                                                   */
  uint8_t mapq_fixed;   /* non-zero: MAPQ is this (42: unique exact first seed, 1: multi-exact with --ambiguous_out)    */
  uint8_t k;            /* the read's error threshold                                                                    */
  uint32_t n_aux;
} bmbs_final;           /* 32 bytes */
/* Enqueue the finishing kernels behind bmbs_batch_run on the batch's stream.
 * Paired batches (SURVEY.md 8a V4 / V5): what Map_Pair_Seq_split_fast / Map_Pair_Seq_split do after their verification calls --
 * hit compaction (Schema.cpp:7502-7608), filter_pairs_single_side (:16186-16288), the pair pick new_faster_verify_pairs
 * (:15773-15959: smallest err sum, the first such pair, how many, second_best_diff), then try_cigar_without_path and the
 * coordinates of the two chosen hits.  fin[2p], fin[2p+1] are the mates of pair p: fin[2p].status = BMBS_FIN_UNMAPPED (no pair),
 * BMBS_FIN_AMBIGUOUS (several equally good pairs, not reported), else each mate is BMBS_FIN_UNIQUE (ungapped: chrom_pos,
 * strand, nm, mismatch positions) or BMBS_FIN_DP (site, end_site, nm = the verifier's err); sbd = the pair's second_best_diff
 * (255 = more); BMBS_FINF_AMBIGUOUS = reported although several pairs tie (--ambiguous_out).  A mate that runs over the end of
 * its chromosome keeps its coordinates (the caller's span check drops the pair, Schema.cpp:22310-22330).  The window lists of
 * the batch are compacted in place: bmbs_batch_download is not meaningful after this call.  No window lists come back. */
int bmbs_batch_finish(bmbs_batch* b);
/* Wait, then copy back fin[n_reads], the mismatch positions and the window lists of handed-back reads.
 * BMBS_ERR_CAPACITY with the needed sizes in *mism_used / *cand_used when a caller buffer is too small. */
int bmbs_batch_download_final(bmbs_batch* b, bmbs_final* fin, uint16_t* mism, size_t mism_cap, size_t* mism_used,
                              bmbs_cand* cand, size_t cand_cap, size_t* cand_used);
/* counters of the last bmbs_batch_finish: [0] mismatch positions [1] handed-back windows [2] reads whose window order was
 * replayed on the device [3] reads handed back [4] reads marked BMBS_FIN_DP [5] / [6] replayed because the chosen window /
 * second_best_diff depended on the order [7] device time of the finishing kernels, us */
int bmbs_batch_finish_counters(bmbs_batch* b, uint64_t c[8]);
/* test entry: the order libstdc++'s std::sort by vote (descending, Schema.cpp:27612) leaves each list
 * votes[offsets[i] .. offsets[i+1]) in (<= 2048 votes per list, each < 32), computed by the warp routine the finishing uses;
 * order[] receives original positions, ok[i] = 0 when the replay declined (introsort depth limit) */
int bmbs_debug_sort_order(int dev, const uint32_t* votes, const uint32_t* offsets, uint32_t n_lists, uint16_t* order, int* ok);

/* ---- CIGAR refinement (SURVEY.md 8f-1): the banded affine-gap DP with traceback, end fix-ups and NM recount ----------
 * Replaces fast_recalculate_bs_Cigar (ksw.cpp:2578-3148) for the alignments whose ungapped re-check (try_cigar_without_path,
 * :2515-2570 -- done by bmbs_batch_finish for single-end reads, by the caller otherwise) failed, i.e. alignments with indels:
 * ksw_semi_global_quality_back (:1850-2045), then the leading / trailing insertions turned into matches (:2894-2990) and the NM
 * recount over the final operations (:2990-3143).  One call refines a whole sub-block's worth of alignments.
 * The window is read from the index on the device (get_actuall_genome / _rc_genome, Schema.cpp:4998-5115: L + 2k bases
 * at `site`, all-N when it leaves the strand); the caller sends the read as aligned and its qualities in the order the
 * reference's DP sees them (reversed for mate 2, calculate_best_map_cigar_end_to_end_return need_reverse_quality=1).
 * Scores: read T on reference C is a match; mismatch = -(mp_min + (int)((mp_max - mp_min) * min(q - q_base, 40) / 40));
 * N on either side = -n_pen; gap of length g = -(gap_open + g * gap_ext)  (ksw.h:148-162, ksw.cpp:1917-1950).
 * Result: best score in the last row, first / last window position of the final alignment (qb, qe), NM, and the final
 * operations as run-length ops in read order, (len << 4) | op with op 0 = M, 1 = D (window only), 2 = I (read only); the
 * CIGAR string is these ops printed first to last for a forward-strand hit and last to first for a reverse-strand one. */
typedef struct bmbs_refiner bmbs_refiner;              /* one per host thread: own stream and device buffers          */
typedef struct { int mp_max, mp_min, n_pen, gap_open, gap_ext, q_base; } bmbs_scoring;   /* defaults 6 2 1 5 3 33 */
typedef struct {
  uint64_t site;        /* window start, double-strand coordinate (as bmbs_cand.site)                                  */
  uint32_t seq_off;     /* offset of the read (and of its qualities) in seqs[] / quals[]                               */
  uint16_t len;         /* read length L                                                                               */
  uint8_t  k;           /* error threshold: band = 2k + 1, window = L + 2k                                             */
  uint8_t  pad;
} bmbs_refine_item;
typedef struct { int32_t score, qb, qe; uint32_t n_ops; uint32_t ops_off; uint32_t nm; } bmbs_refine_result;   /* ops[ops_off .. +n_ops) */
int bmbs_refiner_create(bmbs_index* idx, int dev, bmbs_refiner** out);
void bmbs_refiner_free(bmbs_refiner* r);
/* seqs / quals: `bytes` bytes each; res[n]; ops[ops_cap] receives every item's ops back to back (*ops_used entries);
 * BMBS_ERR_CAPACITY with the needed size in *ops_used when ops_cap is too small (2 * len + 2 * k + 2 per item always fits). */
int bmbs_refine(bmbs_refiner* r, const char* seqs, const char* quals, size_t bytes, const bmbs_refine_item* items, size_t n,
                const bmbs_scoring* sc, bmbs_refine_result* res, uint32_t* ops, size_t ops_cap, size_t* ops_used);
/* device time of the kernels of the last bmbs_refine call (CUDA events on the refiner's stream), ms */
int bmbs_refiner_kernel_ms(bmbs_refiner* r, float* ms);

#ifdef __cplusplus
}
#endif
#endif
