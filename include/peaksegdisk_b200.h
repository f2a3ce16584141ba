/* peaksegdisk_b200.h -- C ABI of the B200-native PeakSegFPOP solver (libpeaksegdisk_b200.so).
 *
 * Drop-in boundary: the reference's only native entry for this path is
 *     int PeakSegFPOP_disk(char *bedGraph_file_name, char *penalty_str, char *db_file_name);
 * declared in tdhock/PeakSegDisk src/PeakSegFPOPLog.h:15 and called from src/interface.cpp:15
 * (the .C routine "PeakSegFPOP_interface" that R/PeakSegFPOP_file.R:66-71 invokes).
 * This library exports that exact C++-mangled symbol (_Z16PeakSegFPOP_diskPcS_S_) so an unchanged
 * interface.cpp links against it, plus the plain-C entry points below.  No torch types, only
 * pointers and sizes.  All entry points are thread-safe for distinct plans / distinct file names.
 *
 * There is no CPU fallback: every solve runs the sm_100a kernels and fails with PSD_ERR_CUDA
 * when no usable GPU / driver is present.
 */
#ifndef PEAKSEGDISK_B200_H
#define PEAKSEGDISK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ---------------------------------------------------------------------------
 * 0..11 are the reference's (src/PeakSegFPOPLog.h:3-13), same meaning, same order of checks. */
#define PSD_OK 0
#define PSD_ERR_PENALTY_NOT_FINITE 1
#define PSD_ERR_PENALTY_NEGATIVE 2
#define PSD_ERR_UNABLE_TO_OPEN_BEDGRAPH 3
#define PSD_ERR_NOT_ENOUGH_COLUMNS 4
#define PSD_ERR_NON_INTEGER_DATA 5
#define PSD_ERR_INCONSISTENT_CHROMSTART_CHROMEND 6
#define PSD_ERR_WRITING_COST_FUNCTIONS 7
#define PSD_ERR_WRITING_LOSS_OUTPUT 8
#define PSD_ERR_NO_DATA 9
#define PSD_ERR_PENALTY_NOT_NUMERIC 10
#define PSD_ERR_WRITING_SEGMENTS_OUTPUT 11
/* ours (never produced by the reference) */
#define PSD_ERR_PIECE_OVERFLOW 101   /* a cost function outgrew the largest piece-list tier */
#define PSD_ERR_STORE_EXHAUSTED 102  /* the HBM cost-function store cannot hold this problem */
#define PSD_ERR_BACKTRACK 103
#define PSD_ERR_INTERNAL 104
#define PSD_ERR_CUDA 110             /* no device, driver error or kernel fault: see psd_last_error() */
#define PSD_ERR_ARG 111

/* Replaces PeakSegFPOP_disk (src/PeakSegFPOPLog.cpp:143-463): reads the 4-column bedGraph, solves
 * on the GPU, writes <bedGraph>_penalty=<penalty_str>_segments.bed and _loss.tsv byte-identical to
 * the reference's.  db_file is created/truncated on the non-trivial branch exactly as the
 * reference does (error 7 if that fails) and receives a small header; the cost functions
 * themselves live in HBM.  Returns a status code. */
int psd_fpop_disk(const char *bedGraph_file_name, const char *penalty_str, const char *db_file_name);

/* The same for n (bedGraph, penalty, db) triples in ONE batched launch: one warp per problem.
 * status_out[i] receives problem i's code.  Returns 0, or PSD_ERR_CUDA if the device failed. */
int psd_fpop_disk_batch(int n, const char *const *bedGraph_file_names, const char *const *penalty_strs,
                        const char *const *db_file_names, int *status_out);

/* Message for a status code; the 1..11 texts are interface.cpp:16-52's format strings. */
const char *psd_status_message(int status);
const char *psd_last_error(void);

/* ---- in-memory batch ("plan"): rows in, segments out, explicit H2D / solve / D2H steps ------ */
typedef struct psd_plan psd_plan;

typedef struct psd_result {
  int32_t status;
  int32_t trivial;           /* 1: one-segment model (penalty Inf or constant coverage), solved on the host */
  int32_t n_rows;            /* bedGraph.lines */
  int32_t n_segments;
  int32_t n_peaks;
  int32_t n_equality;        /* equality.constraints */
  double penalty;
  double bases;
  double mean_pen_cost;
  double total_loss;
  double mean_intervals;
  double max_intervals;
} psd_result;

typedef struct psd_stats {
  double dp_ms;              /* device time of the DP kernel(s), CUDA events on the plan's stream */
  double backtrack_ms;       /* device time of the backtrack kernel(s) */
  double h2d_ms, d2h_ms;
  int64_t rows_solved;       /* rows of the non-trivial problems */
  int64_t store_bytes_algorithmic;  /* sum over problems of N*24 + 20*total_intervals (SURVEY 8d) */
  int64_t store_bytes_written;      /* bytes of records + index actually written to HBM */
  int64_t store_bytes_spilled_host; /* record bytes that overflowed into pinned host memory */
  int64_t backtrack_bytes_read;
  int64_t h2d_bytes, d2h_bytes;
  int32_t n_launches;        /* kernels launched by the last solve */
  int32_t n_waves;           /* store waves */
  int32_t n_overflow_tier;   /* problems that needed the global-memory piece-list tier */
  int32_t piece_cap;         /* shared-memory tier capacity (pieces per function) */
  int32_t warps_per_sm;
  int32_t n_sm;
  /* count-vector problems (psd_plan_add_counts): the device run-length encoding done at upload */
  int32_t n_rle_launches;
  double rle_ms;                    /* device time of the four RLE kernels */
  int64_t rle_positions;            /* count positions encoded */
  int64_t rle_bytes_algorithmic;    /* 4 B per position read + 12 B per row written */
  int32_t n_latency_waves;          /* waves of the last solve that ran the latency kernel (one problem per block) */
  int32_t pad_;
  int64_t store_bytes_drained_dma;  /* of the spilled bytes: copied HBM ring -> pinned host by cudaMemcpyAsync on the side stream */
} psd_stats;

/* device < 0 selects the current CUDA device. */
psd_plan *psd_plan_create(int device);
void psd_plan_destroy(psd_plan *plan);
/* Adds one problem; rows are copied.  penalty_is_inf != 0 selects the no-peaks model.
 * Rows must be contiguous (chromStart[i] == chromEnd[i-1], else -6 like the file path,
 * src/PeakSegFPOPLog.cpp:180-186), of positive width and non-negative coverage (else -PSD_ERR_ARG).
 * Returns the problem id (>= 0) or a negative PSD_ERR_*. */
int psd_plan_add(psd_plan *plan, int64_t n_rows, const int32_t *chromStart, const int32_t *chromEnd,
                 const int32_t *coverage, double penalty, int penalty_is_inf);
/* In-memory front end for a count vector (replaces R/PeakSegFPOP_vec.R:18-25 + PeakSegFPOP_df's
 * bedGraph round trip): counts[i] >= 0 is the coverage of base [i, i+1).  The run-length encoding
 * into bedGraph rows happens on the device at upload.  Results are the same as psd_plan_add() on the
 * rows (chromStart 0-based, chromEnd = cumulative run lengths).  Returns the problem id or -PSD_ERR_*. */
int psd_plan_add_counts(psd_plan *plan, int64_t n_positions, const int32_t *counts, double penalty,
                        int penalty_is_inf);
int psd_plan_size(const psd_plan *plan);
/* stream: a cudaStream_t (0 = default stream).  upload/solve/download enqueue work on it;
 * download synchronizes the stream before returning. */
int psd_plan_upload(psd_plan *plan, void *stream);
int psd_plan_solve(psd_plan *plan, void *stream);
int psd_plan_download(psd_plan *plan, void *stream);
/* upload + solve + download */
int psd_plan_run(psd_plan *plan, void *stream);
int psd_plan_result(const psd_plan *plan, int id, psd_result *out);
/* Segments of problem id, last segment first (the order of _segments.bed).  Arrays need
 * n_segments entries; is_peak is 0 (background) / 1 (peak). */
int psd_plan_segments(const psd_plan *plan, int id, int32_t *chromStart, int32_t *chromEnd,
                      int32_t *is_peak, double *mean);
int psd_plan_get_stats(const psd_plan *plan, psd_stats *out);
/* Replaces problem id's penalty (used by the sequential search to re-solve the same rows). */
int psd_plan_set_penalty(psd_plan *plan, int id, double penalty, int penalty_is_inf);

/* ---- label errors (PeakError semantics, 0-based half-open coordinates) ------------------------
 * A label [chromStart, chromEnd) of kind 0 noPeaks, 1 peaks, 2 peakStart, 3 peakEnd is scored on the
 * peak segments [ps, pe) of a problem's segmentation: o = peaks with ps < chromEnd and chromStart < pe,
 * a = peak starts in [chromStart, chromEnd), b = peak ends in (chromStart, chromEnd].
 *   noPeaks: fp = o > 0, fn = 0;  peaks: fp = 0, fn = o == 0;  peakStart: fp = a > 1, fn = a == 0;
 *   peakEnd: fp = b > 1, fn = b == 0.  possible_fp = kind != 1, possible_fn = kind != 0.
 * Labels are scored on the device right after the backtrack, only for plans that have labels. */
typedef struct psd_label_errors {
  int32_t fp, fn, possible_fp, possible_fn, errors;   /* sums over the problem's labels; errors = fp + fn */
} psd_label_errors;
/* Copies n labels of problem id (n = 0 removes them).  Each needs chromStart < chromEnd inside the
 * problem's [first chromStart, last chromEnd) and kind 0..3; they may be unsorted and overlap.  Returns
 * 0, or PSD_ERR_ARG with the problem and label named in psd_last_error(). */
int psd_plan_set_labels(psd_plan *plan, int id, int64_t n, const int32_t *chromStart, const int32_t *chromEnd,
                        const int32_t *kind);
/* After psd_plan_solve: the totals of problem id and, if the arrays are not null, fp / fn per label in
 * the order they were set.  Returns 0, the problem's solver status, or PSD_ERR_ARG (no labels, not solved). */
int psd_plan_label_errors(const psd_plan *plan, int id, psd_label_errors *total, int32_t *fp, int32_t *fn);

/* ---- exact model-selection path (CROPS) ------------------------------------------------------
 * Every model that is optimal for some penalty in [pen_min, pen_max], found by solving at the crossing
 * penalty of each pair of neighbouring models (Haynes, Eckley and Fearnhead 2017); every pending pair of
 * every problem is solved in one batched plan solve per round.  With labels, each model's label errors
 * are counted on the device and the target interval is the widest (in log penalty) run of consecutive
 * models with the fewest errors. */
typedef struct psd_path_problem {
  int64_t n_rows;                                    /* rows as for psd_plan_add */
  const int32_t *chromStart, *chromEnd, *coverage;
  int64_t n_labels;                                  /* labels as for psd_plan_set_labels (0: none) */
  const int32_t *label_start, *label_end, *label_kind;
} psd_path_problem;
typedef struct psd_path_model {
  double min_lambda, max_lambda;   /* the penalties for which this model is optimal */
  double penalty;                  /* the penalty of the solve that found it */
  double total_loss;
  int32_t peaks, segments;
  int32_t fp, fn, possible_fp, possible_fn, errors;   /* zero without labels */
  int32_t pad_;
} psd_path_model;
typedef struct psd_path psd_path;
typedef struct psd_path_stats {
  double dp_ms, backtrack_ms, label_ms;   /* device time summed over rounds */
  int64_t rows_solved;                     /* rows x solves of the non-trivial solves */
  int64_t h2d_bytes, d2h_bytes;
  int32_t rounds, solves, models, n_problems;
} psd_path_stats;
/* Solves the path of n_problems problems on [pen_min, pen_max] (pen_max may be INFINITY).  Inputs are
 * checked on the host before any device work: NaN or negative pen_min, pen_min > pen_max, an infinite
 * pen_min with a finite pen_max, n_problems < 0 and bad rows or labels return PSD_ERR_ARG, naming the
 * problem in psd_last_error().  A problem whose solve fails keeps that status and no models; the others
 * finish.  device < 0: the current device.  Returns 0 and *out (free with psd_path_free), or an error. */
int psd_model_path(int device, int n_problems, const psd_path_problem *problems, double pen_min, double pen_max,
                   psd_path **out);
int psd_path_status(const psd_path *path, int i);        /* problem i's status (PSD_ERR_ARG if i is out of range) */
int psd_path_n_models(const psd_path *path, int i);      /* -1 if i is out of range */
/* Copies problem i's models, sorted by peaks ascending; the array needs psd_path_n_models entries. */
int psd_path_models(const psd_path *path, int i, psd_path_model *models);
/* Problem i's target interval: *errors = -1 (and NaN penalties) when it has no labels or no models. */
int psd_path_target(const psd_path *path, int i, double *min_lambda, double *max_lambda, int32_t *errors);
int psd_path_get_stats(const psd_path *path, psd_path_stats *out);
void psd_path_free(psd_path *path);

/* Where the wall time of the process's last psd_fpop_disk / psd_fpop_disk_batch call went. */
typedef struct psd_batch_stats {
  double parse_ms;           /* bedGraph text -> rows (distinct files on all host cores) + penalty parsing */
  double build_ms;           /* pass-1 totals, output files created, scratch db files */
  double run_ms;             /* upload + DP + backtrack + download (wall) */
  double write_ms;           /* _segments.bed / _loss.tsv rendered and written */
  double release_ms;
  double dp_ms, backtrack_ms;      /* device time inside run_ms (max over the GPUs used) */
  int64_t rows_parsed, rows_solved;
  int64_t h2d_bytes, d2h_bytes, store_bytes_algorithmic;
  int32_t n_problems, n_files_parsed, n_devices, n_launches, n_waves, n_latency_waves;
} psd_batch_stats;
int psd_last_batch_stats(psd_batch_stats *out);

/* Writes rows as the 4-column bedGraph text R/writeBedGraph.R:35-37 produces (tab separated, no
 * header, one "chrom\tchromStart\tchromEnd\tcount" line per row).  Returns 0 or PSD_ERR_ARG when the
 * file cannot be written. */
int psd_write_bedgraph(const char *path, const char *chrom, int64_t n_rows, const int32_t *chromStart,
                       const int32_t *chromEnd, const int32_t *count);

/* ---- coverage from aligned reads --------------------------------------------------------------
 * One problem is the reads of one region of one sample.  The coverage of base b is the number of
 * reads with start <= b < end (bedtools genomecov -bga, clipped to the region); the rows are the
 * maximal runs of equal coverage, zero runs included, and tile [region_start, region_end) exactly, so
 * they are valid psd_plan_add / psd_write_bedgraph input.  Reads partly outside the region are
 * clipped, reads wholly outside are ignored; a region without reads gives one zero row. */
typedef struct psd_reads {
  int64_t n_reads;
  const int32_t *read_start, *read_end;    /* half-open [start, end), any order */
  int32_t region_start, region_end;        /* rows tile [region_start, region_end) */
} psd_reads;
typedef struct psd_coverage psd_coverage;  /* rows of every problem, on the host */
typedef struct psd_coverage_stats {
  double device_ms;                        /* CUDA events around H2D + zero-fill + scatter + scan + RLE + D2H, summed over waves */
  double kernel_ms;                        /* zero-fill + scatter + scan + RLE only */
  int64_t reads, bases, rows, h2d_bytes, d2h_bytes;   /* reads and bases of the problems that went to the device */
  int32_t n_problems, n_waves;
} psd_coverage_stats;
/* Computes the rows of n_problems problems on the device, in waves whose dense per-base buffers fit
 * the "coverage_gb" budget (psd_set_option).  Inputs are checked on the host before any device work:
 * start < 0, end <= start, region_start < 0, region_end <= region_start, a region longer than
 * 0x3fffffff bases, a null read array with n_reads > 0 and n_reads outside [0, 2^31) return PSD_ERR_ARG
 * and psd_last_error() names the problem and read.  device < 0: the current device.  Returns 0 and
 * *out (free it with psd_coverage_free), or PSD_ERR_ARG / PSD_ERR_CUDA and no handle. */
int psd_coverage_from_reads(int device, int n_problems, const psd_reads *problems, psd_coverage **out);
/* Rows of problem i (-1 if i is out of range). */
int64_t psd_coverage_n_rows(const psd_coverage *cov, int i);
/* Copies problem i's rows; the arrays need psd_coverage_n_rows(cov, i) entries. */
int psd_coverage_rows(const psd_coverage *cov, int i, int32_t *chromStart, int32_t *chromEnd, int32_t *count);
int psd_coverage_get_stats(const psd_coverage *cov, psd_coverage_stats *out);
void psd_coverage_free(psd_coverage *cov);

/* ---- per-problem coverage statistics (penalty-learning features) -------------------------------
 * For one problem the rows give weights w_i = chromEnd_i - chromStart_i and counts c_i; the per-base
 * vector has B = sum w_i entries (w_i copies of c_i).  The statistics are those of that vector, computed
 * on the device without expanding it: the quartiles at p = 0, .25, .5, .75, 1 by R's type 7 (h = (B-1) p,
 * lo = floor(h), g = h - lo; x[lo] when g == 0 or x[lo+1] == x[lo], else (1-g) x[lo] + g x[lo+1] on the
 * sorted vector x), mean = S1 / B and sd = sqrt((B S2 - S1^2) / (B (B-1))) with S1 = sum w c and
 * S2 = sum w c^2 in exact integer arithmetic (NaN when B == 1), bases = B and rows = the row count. */
typedef struct psd_rows {
  int64_t n_rows;
  const int32_t *chromStart, *chromEnd, *coverage;   /* rows as for psd_plan_add */
} psd_rows;
typedef struct psd_problem_features {
  double quartile[5];   /* p = 0, .25, .5, .75, 1 (R type 7) */
  double mean, sd;      /* sd NaN when bases == 1 */
  int64_t bases, rows;
} psd_problem_features;
typedef struct psd_features_stats {
  double device_ms;     /* CUDA events around H2D + kernels + D2H, summed over waves */
  double kernel_ms;     /* the histogram and select kernels only */
  int64_t rows, h2d_bytes, d2h_bytes;
  int32_t n_problems, n_waves, n_launches;
} psd_features_stats;
/* Fills out[0 .. n_problems-1].  Rows are checked on the host before any device work with the rules of
 * psd_plan_add: a bad problem returns PSD_ERR_ARG (or PSD_ERR_INCONSISTENT_CHROMSTART_CHROMEND for rows
 * that are not contiguous) and is named in psd_last_error(); so do null arrays and n_problems < 0.  Zero
 * problems return 0 without touching the device.  Problems go in waves of consecutive problems whose
 * device buffers fit the "coverage_gb" budget (psd_set_option).  device < 0: the current device.  stats
 * may be null.  Returns 0, or an error (out's contents are then unspecified). */
int psd_features(int device, int n_problems, const psd_rows *problems, psd_problem_features *out,
                 psd_features_stats *stats);

/* ---- joint single-peak models of many samples (the model of PeakSegJoint, solved exactly) -------------
 * A problem is one region [region_start, region_end) with S samples (1 <= S <= 256) whose rows (the rules of
 * psd_plan_add) tile the region exactly, and a bin width bin_bases >= 1.
 *   Grid: g_k = region_start + k bin_bases for k = 0..N-1 and g_N = region_end, N = ceil(length / bin_bases)
 *   (the last bin may be shorter).  N is at most PSD_JOINT_MAX_BINS: a problem's work grows as N^2 S (about
 *   1.4e11 pair x sample evaluations at the cap with 256 samples), and pair indices stay in 32 bits.
 *   Sums: C_s(i, j) = the sum of sample s's counts over the bases of [g_i, g_j) (exact int64), W(i, j) = g_j - g_i.
 *   Segment loss: L_s(i, j) = C - C log(C / W) in double (0 when C = 0); the flat model of s has L1_s = L_s(0, N),
 *   and flat = the sum of L1_s in sample order.
 *   Peak (a, b), 1 <= a < b <= N-1: sample s can carry it only if C_s(a,b) W(0,a) > C_s(0,a) W(a,b) and
 *   C_s(a,b) W(b,N) > C_s(b,N) W(a,b) (exact integers: its peak mean is strictly above both flank means);
 *   then L3_s = (L_s(0,a) + L_s(a,b)) + L_s(b,N) and r_s = L1_s - L3_s.
 *   Model k at (a, b): the first k feasible samples in the order (r desc, sample index asc) carry the peak;
 *   loss_k(a, b) = flat - R_k, R_k their reductions added one after the other in that order (+inf when
 *   fewer than k samples are feasible).
 *   Model k (k = 0..S): the minimum of loss_k over all peaks, ties to the smaller a, then the smaller b.  Model 0
 *   is the flat model without a peak; a k that no peak reaches has no model.
 *   Selection: argmin_k loss_k + lambda k, lambda in [0, inf).  The selectable models are the corners of the
 *   lower convex hull of (k, loss_k), added by increasing k, a corner being dropped unless the breakpoint
 *   (loss_i - loss_j) / (j - i) with the corner before it is strictly larger than with the next one and
 *   strictly positive.  A selectable model gets [min_lambda, max_lambda] from its breakpoints (model 0:
 *   max_lambda = inf; the selectable model with the most peaks: min_lambda = 0); the others get NaN.
 *   Labels (optional, per sample, the kinds and rules of psd_plan_set_labels): in model k each peaked sample has
 *   the one peak [g_a, g_b) and the others none; fp / fn / possible_fp / possible_fn / errors are summed over
 *   all samples' labels, and the target interval is psd_model_path's, over the selectable models.
 * The device computes the minima (joint_gpu.cuh); the host recomputes each winner's samples and loss in the same
 * arithmetic and requires the same bits (PSD_ERR_INTERNAL otherwise).  This is not PeakSegJoint's binned search:
 * it is the exact optimum over every peak of the grid. */
#define PSD_JOINT_MAX_SAMPLES 256
#define PSD_JOINT_MAX_BINS 32768
typedef struct psd_joint_sample {
  int64_t n_rows;                                    /* rows as for psd_plan_add */
  const int32_t *chromStart, *chromEnd, *coverage;
  int64_t n_labels;                                  /* labels as for psd_plan_set_labels (0: none) */
  const int32_t *label_start, *label_end, *label_kind;
} psd_joint_sample;
typedef struct psd_joint_problem {
  int32_t region_start, region_end;                  /* every sample's rows tile exactly this region */
  int32_t bin_bases;                                 /* bin width, >= 1 */
  int32_t n_samples;                                 /* S, 1..PSD_JOINT_MAX_SAMPLES */
  const psd_joint_sample *samples;
} psd_joint_problem;
typedef struct psd_joint_model {
  double total_loss;
  double min_lambda, max_lambda;   /* NaN when not selectable */
  int32_t peaks;                   /* k, the number of samples with the peak */
  int32_t peak_start, peak_end;    /* [g_a, g_b); -1 for k = 0 */
  int32_t selectable;
  int32_t fp, fn, possible_fp, possible_fn, errors;   /* sums over all samples' labels; zero without labels */
  int32_t pad_;
} psd_joint_model;
typedef struct psd_joint psd_joint;
typedef struct psd_joint_stats {
  double device_ms;                /* CUDA events around H2D + kernels + D2H, summed over waves */
  double kernel_ms;                /* the flank, flat, pair and reduce kernels only */
  int64_t samples;                 /* sum of S over the problems */
  int64_t pair_sample_evals;       /* sum of S (N-1)(N-2)/2: the (peak, sample) pairs scored on the device */
  int64_t h2d_bytes, d2h_bytes;
  int32_t n_problems, n_waves, n_launches, pad_;
} psd_joint_stats;
/* Solves n_problems problems.  Inputs are checked on the host before any device work: S outside 1..256, a null
 * sample array, rows that break psd_plan_add's rules or do not tile the problem's region, bin_bases < 1, N over
 * PSD_JOINT_MAX_BINS and bad labels return PSD_ERR_ARG, and psd_last_error() names the problem and the sample.
 * Zero problems never touch the device.  Problems go in waves whose device buffers fit the "coverage_gb" budget
 * (psd_set_option); a problem larger than the budget runs alone.  device < 0: the current device.  Returns 0
 * and *out (free it with psd_joint_free), or an error and no handle. */
int psd_joint_models(int device, int n_problems, const psd_joint_problem *problems, psd_joint **out);
int psd_joint_n_models(const psd_joint *h, int i);   /* models of problem i (k that have one); -1 if i is out of range */
/* Copies problem i's models, k ascending; the array needs psd_joint_n_models entries. */
int psd_joint_model_table(const psd_joint *h, int i, psd_joint_model *models);
/* in_peak[s] = 1 if sample s carries the peak in problem i's model with k peaked samples (S entries); PSD_ERR_ARG
 * if that model does not exist. */
int psd_joint_samples(const psd_joint *h, int i, int k, uint8_t *in_peak);
/* Problem i's target interval: *errors = -1 (and NaN penalties) when no sample of it has labels. */
int psd_joint_target(const psd_joint *h, int i, double *min_lambda, double *max_lambda, int32_t *errors);
int psd_joint_get_stats(const psd_joint *h, psd_joint_stats *out);
void psd_joint_free(psd_joint *h);

/* Inspection of the cost-function store (replaces DiskVector::read, src/PeakSegFPOPLog.cpp:103-117,
 * for tests and tools): the stored function `which` (0 = up, 1 = down) of bedGraph row `row` of
 * problem id, in the reference's record fields (src/PeakSegFPOPLog.cpp:18-34: max_log_mean, data_i,
 * prev_log_mean per piece).  *n_pieces receives the piece count; arrays need `cap` >= that many
 * entries (PSD_ERR_ARG otherwise).  Valid for problems solved in the plan's last store wave (all of them
 * unless the store had to be recycled). */
int psd_plan_store_function(psd_plan *plan, int id, int row, int which, int cap, int *n_pieces, double *max_log_mean,
                            int *data_i, double *prev_log_mean);

/* Tunables (call before psd_plan_create): "piece_cap" (shared-memory tier, default 48),
 * "overflow_cap" (global tier, default 8192), "store_gb" (HBM pool, default 0 = auto),
 * "chunk_kb" (store chunk, default 64), "spill_cap" (per-warp global workspace, default 512),
 * "host_spill_gb" (pinned-host overflow of the store: -1 = automatic, 0 = off),
 * "spill_mode" (how spilled records reach the host: 0 = written into an HBM ring that a host thread drains
 * with cudaMemcpyAsync on a side stream (default), 1 = zero-copy stores through the mapping), "ring_gb",
 * "occupancy_mode" (0 = choose per batch, 1 = one block of 14 warps per SM, 2 = two blocks),
 * "latency_mode" (0 = per wave, whichever of the two kernels a makespan model predicts to finish first:
 * the latency kernel -- one problem per block, one chain per warp -- for few or long problems, never beyond
 * "latency_max_blocks" (16) problems per SM; 1 = always the latency kernel; 2 = never),
 * "devices" (GPUs one psd_fpop_disk_batch call may use: 1 = the current device (default), k = the
 * first k, <= 0 = all; problems are dealt longest-first, one plan and host thread per GPU),
 * "coverage_gb" (device budget of one psd_coverage_from_reads, psd_features or psd_joint_models wave: dense
 * per-base buffer, rows and reads; rows and histograms; or prefix sums, flank losses and per-chunk candidates;
 * 0 = automatic, half of the free HBM; a problem larger than the budget runs in a wave of its own). */
int psd_set_option(const char *name, double value);

int psd_device_count(void);

/* psd_fpop_disk / psd_fpop_disk_batch keep the plan of their last call parked (device buffers, store
 * pool and pinned staging, up to 100 GB of HBM) so that the next call does not allocate again; this
 * frees it.  Safe to call at any time from any thread. */
void psd_release_cache(void);

#ifdef __cplusplus
}
#endif
#endif
