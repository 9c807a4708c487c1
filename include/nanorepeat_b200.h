/*
 * nanorepeat_b200.h -- C ABI of libnanorepeat_b200.so, the B200 (sm_100a) drop-in for NanoRepeat's
 * repeat-size estimation hot path (rounds 2 and 3).
 *
 * What it replaces in the reference (paths relative to the reference tree, src/NanoRepeat/):
 *   - the alignment engine call `pymm2.main(cmd)` at nanoRepeat_bam.py:362 (round 2: every read core
 *     against ONE template  left_anchor + motif*T)            -> nr_round2_region()
 *   - the per-read engine call at nanoRepeat_bam.py:497 (round 3: one core against the ladder
 *     left_anchor + motif*k + right_anchor, k = kmin..kmax) together with the PAF parse / top-score /
 *     span-predicate selection of nanoRepeat_bam.py:408-434     -> nr_round3_region()
 *   - the generic engine shape (any query against any target, PAF fields AS/tstart/tend of
 *     paf.py:39-64)                                             -> nr_score_tasks()
 *   - the data-type -> preset table tk.py:502-517               -> nr_get_preset()
 *
 * Plain pointers and sizes only; the caller owns every buffer; the library keeps device / pinned pools
 * between calls and never calls exit()/abort().  Every function returns NR_OK (0) or a negative error code;
 * nr_last_error() describes the last failure on the calling thread.  CUDA is initialised lazily on the first
 * compute call (never at load time), so the library is safe to load before the reference's fork()
 * (nanoRepeat_bam.py:719-724); each worker process then owns its own context.
 *
 * Sequences.  Reads may hold any character: ACGT / acgt are bases, anything else is an ambiguous base (minimap2's code 4,
 * scored -ambiguous against every template base, as the reference's engine does with N); white space around a read is
 * dropped, as the reference's FASTQ / FASTA round trip does (nanoRepeat_bam.py:311-321, :487-493).  Templates (anchors,
 * motif, generic targets) must be ACGT: a region whose anchor holds another character is NOT SCORED -- its reads come back
 * with score 0, i.e. "the aligner printed nothing" (round 2 leaves the size unset, nanoRepeat_bam.py:373; round 3 leaves
 * it untouched, :421) -- and so is a single task beyond nr_limits (match * min(|query|, |template|) > 32767, or a template
 * over 65471 bases).  Neither fails the call: nr_stats_t.n_skipped counts them, every other read is scored as usual.
 *
 * Alignment contract (bit-exact with oracle/nr_oracle.c): exact local alignment, match +a, mismatch -b,
 * gap of length l costs min(q + l*e, q2 + l*e2);
 *   score  = best local score (0: nothing aligns),
 *   tend   = smallest target end (0-based exclusive) among alignments reaching score,
 *   tstart = largest target start (0-based) among alignments reaching score and ending at tend.
 */
#ifndef NANOREPEAT_B200_H
#define NANOREPEAT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NR_OK                0
#define NR_ERR_CUDA         -1   /* CUDA runtime failure (no device, launch error, out of memory on device) */
#define NR_ERR_ARG          -2   /* null pointer / negative size / inconsistent arguments */
#define NR_ERR_BAD_BASE     -3   /* malformed read buffer (e.g. a line count that does not match n_reads) */
#define NR_ERR_TOO_LARGE    -4   /* a batch exceeds an index range (2^31 rungs, 2^32 pool words, 2^24 tasks) */
#define NR_ERR_NOMEM        -5   /* host allocation failure */
#define NR_ERR_UNKNOWN_TYPE -6   /* nr_get_preset: data type not in the reference's table */

typedef struct nr_scoring_t {
    int32_t match;        /* minimap2 -A  (map-ont: 2)  */
    int32_t mismatch;     /* minimap2 -B  (4), charged as -mismatch */
    int32_t gap_open1;    /* minimap2 -O first value (4) */
    int32_t gap_ext1;     /* minimap2 -E first value (2) */
    int32_t gap_open2;    /* minimap2 -O second value (24) */
    int32_t gap_ext2;     /* minimap2 -E second value (1) */
    int32_t ambiguous;    /* minimap2 --score-N (1): a read base other than ACGT scores -ambiguous against any base */
    int32_t min_dp_score; /* minimap2 -s (80): alignments scoring below it are "not printed" by the selection */
} nr_scoring_t;

/* One alignment record: the three PAF fields rounds 2-3 read (paf.py:47-52,57-58). */
typedef struct nr_aln_t { int32_t score, tstart, tend; } nr_aln_t;

/* Per-rung summary produced by the round-3 ladder kernel: everything nanoRepeat_bam.py:423-431 looks at. */
typedef struct nr_rung_t {
    int32_t score;        /* AS:i of core vs left + motif*k + right */
    uint8_t starts_in_left;  /* ends_in_right && tstart < |left|: the reference only ever tests the conjunction (:427) */
    uint8_t ends_in_right;   /* tlen - tend < |right|                      (nanoRepeat_bam.py:427, strict) */
    uint8_t pad[2];
} nr_rung_t;

/* Work counters of the last completed call on this thread's context (for bench.py / roofline). */
typedef struct nr_stats_t {
    int64_t algorithmic_cells;  /* sum over tasks of |query| * |template| (full rectangles, SURVEY.md 8d) */
    int64_t executed_cells;     /* DP cells the kernels actually updated (padding and shared prefixes accounted) */
    int64_t n_tasks;
    int32_t kernel_launches;    /* launches of this library's kernels */
    int32_t n_skipped;          /* tasks / reads left unscored: template with a base other than ACGT, or beyond nr_limits.
                                   Their records are zero ("the aligner printed nothing"); everything else is unaffected */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
} nr_stats_t;

/* How the last nr_batch_run split its work (bench.py: one roofline per kernel). */
typedef struct nr_launch_info_t {
    int64_t paired_cells;   /* DP cells the paired u16x2 launch updates (both halves of every word, padding included);
                               after a run of a round-2 batch: the cells it executed (the dominance exit skips some) */
    int64_t rest_cells;     /* DP cells of the 32-bit launch beside it (long reads, other scorings, ...) */
    int32_t n_pairs;        /* warps' worth of paired tasks */
    int32_t n_rest;         /* tasks of the 32-bit launch */
    int32_t n_redo;         /* paired round 3: reads rescored on 32-bit words because of an undecidable tie */
    int32_t reserved;
    float paired_ms, rest_ms, redo_ms;   /* CUDA-event durations on the launching streams; 0 unless nr_set_timing(1) */
    float reserved2;
    int64_t paired_useful_cells;   /* the same counts without padding: only rows that belong to a read (a warp sweeps */
    int64_t rest_useful_cells;     /* 32 * R rows per pair / stripe whatever the reads' lengths) */
    int64_t planned_paired_cells;          /* paired_cells and paired_useful_cells as planned: every pair sweeps its */
    int64_t planned_paired_useful_cells;   /* whole template */
} nr_launch_info_t;

/* Data-type preset table (reference tk.py:502-517: ont, ont_sup, ont_q20, clr, hifi -- all map-ont). */
int nr_get_preset(const char* data_type, nr_scoring_t* out);

/* Lazy, idempotent. device < 0: use NR_DEVICE env var, else LOCAL_RANK, else device 0. */
int nr_init(int device);
int nr_shutdown(void);
const char* nr_last_error(void);
int nr_device_info(int32_t* device, int32_t* sm_count, int32_t* clock_khz);

/* Largest task the packed kernels score: match * min(qlen, tlen) <= max_score and tlen <= max_tlen (larger ones are
 * skipped, see "Sequences" above). */
int nr_limits(int32_t* max_score, int32_t* max_tlen);

/*
 * How round 3 is computed (scores, predicates and selection are identical, bit for bit; tests run all four):
 *   3 (default)  paired flag ladder: as mode 2, but two reads of a region share a warp, one per 16-bit half of every DP
 *                word (VIADDMNMX.U16x2 / VIMNMX3.U16x2: two cells per DPX instruction).  Reads longer than 384 bases,
 *                regions without a left or right anchor and other scorings than map-ont take mode 2's kernel; so does,
 *                in a second launch, any read whose selection hinges on a tie that 16-bit words cannot order.  No rung
 *                records (nr_batch_fetch_round3 with rungs != NULL fails);
 *   2            flag ladder: one backward sweep over the right anchor and one forward sweep over left + motif*kmax
 *                per read, joined at every junction column |left| + k*|motif| (the rungs share prefix and suffix);
 *                the DP words carry the score and the two span predicates only, no coordinates
 *                (nr_batch_fetch_alns is not available on such a batch; |right| <= 32767);
 *   1            the same two sweeps on (score, span) words: every rung also gets its exact (tstart, tend);
 *   0            every rung left + motif*k + right scored as its own full rectangle (what the reference hands its
 *                aligner, nanoRepeat_bam.py:474-497).
 */
int nr_set_ladder_mode(int mode);

/* Generic engine: n independent (query, target) tasks -> out[i]. Replaces pymm2.main at the PAF level. */
int nr_score_tasks(const nr_scoring_t* sc, int32_t n_tasks,
                   const char* const* queries, const int32_t* qlen,
                   const char* const* targets, const int32_t* tlen,
                   nr_aln_t* out);

/* Round 2 (nanoRepeat_bam.py:349-362): every core vs left + motif*T. out[r] for read r. */
int nr_round2_region(const nr_scoring_t* sc,
                     const char* left, int32_t n_left, const char* motif, int32_t motif_len, int32_t T,
                     int32_t n_reads, const char* const* cores, const int32_t* core_len,
                     nr_aln_t* out);

/*
 * Round 3 (nanoRepeat_bam.py:452-500 + :408-434): read r against left + motif*k + right, k = kmin[r]..kmax[r].
 * Outputs per read: top_score[r] = best AS over reportable rungs (0 when none reaches min_dp_score: the
 * reference then leaves round3_repeat_size untouched), n_k[r] / sum_k[r] = count and sum of the rungs k tied at
 * top_score that start inside left and end inside right (n_k == 0: reference falls back to round 2).
 * The host computes np.mean as sum_k / n_k in float64 exactly like :431.
 * rungs (nullable) receives every rung's summary at rungs[rung_offset[r] + k - kmin[r]]; rung_offset has
 * n_reads + 1 entries and may be NULL when rungs is NULL.
 */
int nr_round3_region(const nr_scoring_t* sc,
                     const char* left, int32_t n_left, const char* right, int32_t n_right,
                     const char* motif, int32_t motif_len,
                     int32_t n_reads, const char* const* cores, const int32_t* core_len,
                     const int32_t* kmin, const int32_t* kmax,
                     const int64_t* rung_offset, nr_rung_t* rungs,
                     int64_t* sum_k, int32_t* n_k, int32_t* top_score);

/*
 * Device-resident batches (bench.py `value`: inputs already in HBM when the timed region starts).
 * create = pack + upload; run = kernel launches only, asynchronous on `stream` (a cudaStream_t, NULL = the
 * library's own stream); fetch = synchronise + device->host copy + selection.
 */
typedef struct nr_batch nr_batch_t;
nr_batch_t* nr_batch_create_tasks(const nr_scoring_t* sc, int32_t n_tasks,
                                  const char* const* queries, const int32_t* qlen,
                                  const char* const* targets, const int32_t* tlen);
nr_batch_t* nr_batch_create_round2(const nr_scoring_t* sc,
                                   const char* left, int32_t n_left, const char* motif, int32_t motif_len, int32_t T,
                                   int32_t n_reads, const char* const* cores, const int32_t* core_len);
nr_batch_t* nr_batch_create_round3(const nr_scoring_t* sc,
                                   const char* left, int32_t n_left, const char* right, int32_t n_right,
                                   const char* motif, int32_t motif_len,
                                   int32_t n_reads, const char* const* cores, const int32_t* core_len,
                                   const int32_t* kmin, const int32_t* kmax);
/*
 * Multi-region batches: one launch covers every region added (the reference walks regions one by one,
 * nanoRepeat_bam.py:604-612; with 30 reads per region a B200 needs hundreds of regions per launch to fill up).
 * begin -> add_round2 / add_round3 once per region -> commit (plan + upload) -> run -> fetch.  Reads are passed as
 * one concatenated buffer with n_reads + 1 offsets.  Outputs are concatenated in the order the regions were added.
 * On any error the batch stays valid only for nr_batch_destroy().
 */
#define NR_KIND_ROUND2 1
#define NR_KIND_ROUND3 2
/* Round 2 with (score, tend, tstart <= |left|) records instead of (score, tstart, tend): all the selection of
 * nanoRepeat_bam.py:364-384 reads.  Lets reads up to 512 bases run on the paired u16x2 kernel; fetch with
 * nr_batch_fetch_round2.  As the source of nr_batch_begin_round3_from it also keeps every pair's DP state at the end of
 * the left anchor on the device, and round 3 resumes from it instead of sweeping the left anchor again. */
#define NR_KIND_ROUND2_FLAGS 3
nr_batch_t* nr_batch_begin(const nr_scoring_t* sc, int32_t kind);
int nr_batch_add_round2(nr_batch_t* b, const char* left, int32_t n_left, const char* motif, int32_t motif_len,
                        int32_t T, int32_t n_reads, const char* cores_concat, const int64_t* core_off);
/* The same with the reads as n_reads lines separated by '\n' (no offsets array: one pass less for a Python caller). */
int nr_batch_add_round2_lines(nr_batch_t* b, const char* left, int32_t n_left, const char* motif, int32_t motif_len,
                              int32_t T, int32_t n_reads, const char* lines, int64_t lines_len);
int nr_batch_add_round3(nr_batch_t* b, const char* left, int32_t n_left, const char* right, int32_t n_right,
                        const char* motif, int32_t motif_len, int32_t n_reads, const char* cores_concat,
                        const int64_t* core_off, const int32_t* kmin, const int32_t* kmax);
/*
 * Round 3 over the reads of a committed round-2 batch: the reads stay packed in HBM, only templates and per-read ladder
 * bounds are uploaded (the reference writes every core to disk twice, nanoRepeat_bam.py:311-321 and :487-493).
 * region_index = position of the region among the round-2 batch's nr_batch_add_round2 calls; kmin / kmax cover all
 * reads of that region in order, kmax < kmin skips a read (round 2 gave it no size, :460).  The round-2 batch may be
 * destroyed at any time; its device buffers live until the last batch that reads them is destroyed.
 */
nr_batch_t* nr_batch_begin_round3_from(nr_batch_t* round2);
int nr_batch_add_round3_reuse(nr_batch_t* b, int32_t region_index, const char* right, int32_t n_right,
                              const int32_t* kmin, const int32_t* kmax);
int nr_batch_commit(nr_batch_t* b);
int nr_batch_run(nr_batch_t* b, void* stream);
int nr_batch_fetch_alns(nr_batch_t* b, nr_aln_t* out);                      /* tasks / round2 batches */
/* round-2 batches of either kind: per read AS, tend and the predicate tstart <= |left| (nanoRepeat_bam.py:373).
 * NR_KIND_ROUND2_FLAGS: tend and the predicate are exact whenever tend >= |left| (the other half of the span test);
 * an alignment that ends before the repeat is reported with some tend < |left| -- the reference drops such reads. */
int nr_batch_fetch_round2(nr_batch_t* b, int32_t* score, int32_t* tend, uint8_t* starts_by_left);
int nr_batch_fetch_round3(nr_batch_t* b, const int64_t* rung_offset, nr_rung_t* rungs,
                          int64_t* sum_k, int32_t* n_k, int32_t* top_score);  /* round3 batches */
int nr_batch_stats(const nr_batch_t* b, nr_stats_t* out);
/* nr_set_timing(1): nr_batch_run brackets every kernel with CUDA events; nr_batch_launch_info waits for the run. */
int nr_set_timing(int on);
int nr_batch_launch_info(nr_batch_t* b, nr_launch_info_t* out);
void nr_batch_destroy(nr_batch_t* b);

/*
 * Rounds 1-3 of any number of regions in ONE call: what quantify1repeat_from_bam does per region with
 * round1_and_round2_estimation + round3_estimation (nanoRepeat_bam.py:675-679), with no trip back to the caller between
 * the rounds.  Host buffers in, per-read results out (concatenated in region order):
 *   r1[i]       = float(dist_between_anchors) / len(motif)                               (:341)
 *   r2[i]       = round-2 size, valid only where r2_valid[i] (Read.round2_repeat_size stays None otherwise, :373-384)
 *   r3[i]       = round-3 size; r3_state[i]: 0 = untouched (None), 1 = mean of the tied top rungs (an np.float64 in the
 *                 reference, :431), 2 = fell back to r2 (:433)
 *   T_out[g]    = region g's round-2 template size (:344-347); may be NULL
 * All deciding arithmetic (r1, T, r2, ladder bounds with their truncations, the mean) is done in IEEE doubles exactly as
 * the reference's Python evaluates it.  Regions are grouped and software-pipelined so that packing, uploads and
 * selection of one group overlap the kernels of another.  The reads of a region arrive as n_reads lines separated by
 * '\n' (no trailing newline needed).  has_round1_max_dist: this "region" is one piece of a split region and
 * round1_max_dist is the whole region's longest dist_between_anchors (T is region-wide, :344).
 * Needs map-ont scoring (every preset of the reference) and nr_set_ladder_mode != 0.
 * Threads: the call may be made from several host threads at once (the Python layer sends a long region list as a few
 * chunks on a few threads).  Launches without cooperating stripes run on a stream of the calling thread's own, so two
 * calls' kernels share the GPU block by block; launches with long reads' cooperating stripes stay on the library's one
 * stream (two half-resident grids of waiting blocks must never meet).  A thread's stream lives as long as the process.
 */
typedef struct nr_region_t {
    const char* left;  int32_t n_left;      /* RepeatRegion.left_anchor_seq  */
    const char* right; int32_t n_right;     /* RepeatRegion.right_anchor_seq */
    const char* motif; int32_t motif_len;   /* RepeatRegion.repeat_unit_seq  */
    int32_t n_reads;
    const char* reads; int64_t reads_len;   /* read_core_seq_dict values, in read_dict order */
    const int32_t* dist_between_anchors;    /* Read.dist_between_anchors */
    int32_t has_round1_max_dist;
    int64_t round1_max_dist;
} nr_region_t;
int nr_estimate_regions(const nr_scoring_t* sc, int32_t fast_mode, int32_t n_regions, const nr_region_t* regions,
                        double* r1, double* r2, uint8_t* r2_valid, double* r3, uint8_t* r3_state, int32_t* T_out,
                        nr_stats_t* stats /* nullable: summed over the batches of the call */);

/*
 * Step 1 of any number of regions in ONE call: both anchors in every raw read and the core / middle positions
 * (nanoRepeat_bam.py:165-234), what find_anchor_locations_in_reads does per region with minimap2 (:260-286).
 * Per read the four exact alignments (left / right anchor x read / its reverse complement; the anchor is the query, the
 * read strand the template); a hit is an alignment scoring >= min_dp_score; per anchor the hits sorted by score, '+'
 * first on a tie; an anchor is good with one hit, or with two when AS0 > 1.5 * AS1 (:165-179); a read is accepted when
 * both anchors are good and dist = right.qstart - left.qend (0 when the strands differ) > -10 (:195-211); the core is
 * [left.qend - 100, right.qstart + 100) clamped to the read, the middle [left.qend, right.qstart) (:221-234), both in
 * the orientation of the left anchor's strand.  Two kernel launches per call, whatever the number of regions.
 * A read that is empty, longer than nr_limits' template limit or holds a character other than ACGTacgt is not scored
 * (no hit; nr_stats_t.n_skipped counts the last two); an anchor may hold any character (N scores -ambiguous).  An anchor
 * whose score can exceed nr_limits' score limit on a read (match * min(|anchor|, |read|) > 32767) is not scored on that
 * read: it has no hit there, and n_skipped counts each such (read, anchor) once.
 * Needs map-ont scoring with min_dp_score >= 10 * match (every preset): a hit then spans >= 10 read bases, so the
 * reference's align_len < 10 test (:173) never decides.
 */
typedef struct nr_anchor_region_t {
    const char* left;  int32_t n_left;      /* RepeatRegion.left_anchor_seq  */
    const char* right; int32_t n_right;     /* RepeatRegion.right_anchor_seq */
    int32_t n_reads;
    const char* reads; int64_t reads_len;   /* the region's raw reads: n_reads lines separated by '\n' */
} nr_anchor_region_t;
typedef struct nr_anchor_read_t {           /* one per read, concatenated in region order */
    uint8_t accepted;                       /* the read enters read_dict (both anchors good, dist > -10) */
    uint8_t left_good, right_good;          /* left_anchor_is_good / right_anchor_is_good */
    uint8_t strand;                         /* accepted reads: '+' or '-' (the left anchor's strand); else 0 */
    uint8_t left_strand, right_strand;      /* strand of each anchor's best hit: '+', '-', 0 = no hit */
    uint8_t pad[2];
    int32_t read_len;
    int32_t dist_between_anchors;           /* both anchors good: right.qstart - left.qend, or 0 across strands */
    int32_t core_start, core_end, mid_start, mid_end, left_buffer, right_buffer;   /* accepted reads */
    nr_aln_t left, right;                   /* best hit of each anchor as (AS, qstart, qend) on its strand; score 0: none;
                                               qstart is recovered for good anchors only (-1 otherwise) */
} nr_anchor_read_t;
int nr_anchor_regions(const nr_scoring_t* sc, int32_t n_regions, const nr_anchor_region_t* regions, nr_anchor_read_t* out,
                      nr_stats_t* stats /* nullable: algorithmic cells = sum of 2 * (|left| + |right|) * |read| over the
                                           scored reads */);

/*
 * Joint path (nanoRepeat-joint: two neighbouring repeats quantified together).  The reference aligns every read against
 * a grid of templates left + motif1*k1 + mid + motif2*k2 + right with `minimap2 -c --eqx` (nanoRepeat_joint.py:315-343,
 * :397-419) and re-scores each alignment's CIGAR inside the window [|left| - 10, |left| + m1 k1 + |mid| + m2 k2 + 10)
 * with tk.target_region_alignment_stats_from_cigar (tk.py:435-500); per read the grid point with the best window score
 * wins (nanoRepeat_joint.py:457-476).  Here one DP returns both numbers per (read, template): the alignment score and the
 * window score of the optimal alignment, carried through the DP as a payload -- no CIGAR, no text.  Among alignments of
 * equal score the one with the highest window score is the alignment (the CPU checker under oracle/ states the same rule; its
 * traceback's CIGAR re-scored by the reference's own function gives the same number: tests/golden/make_golden_window.py).
 * A read is aligned as given and as its reverse complement when asked (the joint CLI feeds raw reads of either strand).
 */
typedef struct nr_window_t { int32_t score, window_score; } nr_window_t;
/* n independent (query, target, window [a, b)) tasks; reverse (nullable): 1 = align the query's reverse complement. */
int nr_window_tasks(const nr_scoring_t* sc, int32_t n_tasks, const char* const* queries, const int32_t* qlen,
                    const char* const* targets, const int32_t* tlen, const int32_t* win_a, const int32_t* win_b,
                    const uint8_t* reverse, nr_window_t* out);
/* Grid points of one locus: point i = read point_read[i] against the template of (point_k1[i], point_k2[i]); every
 * distinct template is built and packed once.  out[i] = the better strand's (score, window score), strand[i] (nullable)
 * 0 for '+', 1 for '-'.  score 0: no alignment (the reference would have no PAF line). */
int nr_joint_grid(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* mid, int32_t n_mid,
                  const char* right, int32_t n_right, const char* motif1, int32_t m1, const char* motif2, int32_t m2,
                  int32_t n_reads, const char* const* reads, const int32_t* read_len, int32_t n_points,
                  const int32_t* point_read, const int32_t* point_k1, const int32_t* point_k2, nr_window_t* out,
                  uint8_t* strand);

/* ---- Allele phasing in one dimension (SURVEY.md 8(f) row f3) ------------------------------------------------------
 * What the reference does per region after round 3 (nanoRepeat_bam.py:515-575 split_allele_using_gmm_1d): drop sizes
 * outside mean +- 3 sd (split_alleles.py:98-154), bootstrap every kept size 100 times with Gaussian noise of
 * sd = error_rate * (10 + size) (:82-88), fit sklearn GaussianMixture(n, 'diag', n_init = 10) for n = 2, 3, ... and stop
 * at the first n where two components' [isf(1 - o), isf(o)] intervals (sd floored at 1.0) overlap, keeping n - 1
 * (:171-200); label the kept sizes with that mixture (:258-279).  Here: all regions of a call at once, one thread
 * block per (region, start) running scikit-learn's EM (same E / M steps, reg_covar, tolerance and choice among starts)
 * in fp64.  The reference's random draws are unseeded (random.gauss, k-means inside sklearn), so it does not reproduce
 * itself; this library draws from a counter-based generator keyed by (seed, region_id_base + region index), so a region's
 * result is reproducible and does not depend on which other regions share the call.  Parity is therefore statistical
 * (same number of alleles and labels, means within the bootstrap's standard error), bit-level only against the CPU
 * checker that shares the generator.  Starts: k-means from evenly spread means (start 0) or hashed samples (others).
 */
#define NR_GMM_MAX_COMPONENTS 32
typedef struct nr_gmm_params_t {
    int32_t max_components;      /* --max_num_components (default ploidy + 20, nanoRepeat.py:159-160); <= NR_GMM_MAX_COMPONENTS */
    int32_t n_init;              /* starts per fit: 10 (split_alleles.py:174) */
    int32_t max_iter;            /* 100 (sklearn default) */
    int32_t reserved;
    double  error_rate;          /* 0.07 for every data type as the reference is written (nanoRepeat_bam.py:692-701) */
    double  max_mutual_overlap;  /* --max_mutual_overlap, 0.15 (nanoRepeat.py:123) */
    double  tol;                 /* 1e-3 (sklearn default) */
    double  reg_covar;           /* 1e-6 (sklearn default) */
    uint64_t seed;
} nr_gmm_params_t;
/* sizes[offsets[g] .. offsets[g + 1]) = the round-3 sizes of region g.  Per region: n_components[g] (0: fewer than two
 * sizes, not phased, nanoRepeat_bam.py:533-539) and weights / means / variances [g * max_components + j]; per size:
 * label (component index; -1: trimmed as an outlier or region not phased) and proba (the label's responsibility).
 * Components come in ascending order of their means. */
int nr_phase_1d(const nr_gmm_params_t* p, int32_t n_regions, const int64_t* offsets, const double* sizes,
                int64_t region_id_base, int32_t* n_components, double* weights, double* means, double* variances,
                int32_t* label, double* proba);
/* The two device steps on their own (test seams): the bootstrap (out: 100 * offsets[n_regions] samples, region g's at
 * 100 * offsets[g], sample rep * n + i from size i) and the best-of-n_init fit of n_components[i] components to explicit
 * samples data[offsets[i] .. offsets[i + 1]) (region_id nullable: problem index). lower / iters nullable. */
int nr_gmm_bootstrap(const nr_gmm_params_t* p, int32_t n_regions, const int64_t* offsets, const double* sizes,
                     int64_t region_id_base, double* out);
int nr_gmm1d_fit(const nr_gmm_params_t* p, int32_t n_problems, const int64_t* offsets, const double* data,
                 const int32_t* n_components, const int64_t* region_id, double* lower, int32_t* iters,
                 double* weights, double* means, double* variances);

/* Counters of the last nr_score_tasks / nr_round2_region / nr_round3_region call on this thread. */
int nr_last_stats(nr_stats_t* out);

#ifdef __cplusplus
}
#endif
#endif /* NANOREPEAT_B200_H */
