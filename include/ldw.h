/*
 * libldwgpu -- C ABI of the B200-native LDWeaver hot path (encoding -> Hamming-distance weights ->
 * weighted pairwise-MI scan -> short-range / long-range link filter).
 *
 * Pure C, no R / torch / C++ types in any signature.  Inputs are BORROWED, read-only host buffers
 * (R vectors, numpy arrays); fixed-size outputs are caller-allocated; variable-size link lists are
 * library-owned pinned host buffers (owned by the context) that stay valid until the next scan on the
 * same context or until ldw_destroy().  Every entry point returns 0 on success or a nonzero LDW_ERR_* code;
 * ldw_last_error() gives the message (thread-local).  Nothing is ever printed to stdout and no
 * exception or longjmp crosses this boundary, so an R shim can turn a nonzero code into
 * Rf_error(ldw_last_error()) after releasing its own resources (reference convention:
 * BEGIN_RCPP/END_RCPP, src/RcppExports.cpp:17,24).
 *
 * There is NO CPU fallback behind the device entry points (encoding, weights, scan): without a CUDA
 * device they fail with LDW_ERR_CUDA.  The entry points marked "host only" (FASTA / TSV I/O and the
 * steps that follow the scan inside perform_MI_computation) are not fallbacks of device code: they
 * replace parts of the reference that are host code there too, and work on host buffers.
 *
 * Each entry point names the reference interface it replaces (paths relative to the LDWeaver
 * source tree, v1.5.2).
 */
#ifndef LDW_H
#define LDW_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LDW_ABI_VERSION 2

#if defined(__GNUC__)
#define LDW_API __attribute__((visibility("default")))
#else
#define LDW_API
#endif

enum {
  LDW_OK = 0,
  LDW_ERR_ARG = 1,         /* invalid argument (message says which) */
  LDW_ERR_CUDA = 2,        /* CUDA runtime / driver failure, or no device */
  LDW_ERR_NOMEM = 3,       /* host or device allocation failed */
  LDW_ERR_UNSUPPORTED = 4, /* input outside what this round implements (message says what) */
  LDW_ERR_INTERNAL = 5
};

/* flags for ldw_mi_scan */
enum {
  LDW_SCAN_SR_ONLY = 1,   /* perform_SR_analysis_only = TRUE (R/computePairwiseMI.R:179-189, quirk Q12) */
  LDW_SCAN_IDEAL_Q = 2,   /* opt-out of quirk Q1: use 0.25*r_i*r_j on off-diagonal blocks too (NOT reference behaviour) */
  LDW_SCAN_NO_LINKS = 4,  /* compute MI / thresholds only: no link columns are materialised or copied */
  LDW_SCAN_NO_D2H = 8,    /* materialise the link columns in device memory but do not copy them to the host
                             (device-resident throughput measurement); link outputs come back with n rows and NULL pointers */
  LDW_SCAN_SR_EXACT = 16, /* recompute the MI of every short-range link in fp64 (the reference's arithmetic) on the device,
                             block by block, before the rows are copied out (mi_sr_exact_kernel; also valid with
                             LDW_SCAN_SR_ONLY).  Parity-checked on the fixture in both modes (1e-12) */
  LDW_SCAN_SR_ON_DEVICE = 64, /* the short-range rows are materialised in device memory and STAY there (sr_out comes back with n rows
                             and NULL columns); long-range and borderline rows are copied as usual.  For ldw_sr_postprocess_dev,
                             which derives sr_links_red / the ARACNE check set from the device-resident table, so that the
                             2.9 GB (616 x 100k) of short-range columns never cross PCIe */
  LDW_SCAN_LR_ONLY = 32   /* no short-range link table (sr_out->n = 0): only the long-range rows, thresholds and statistics.
                             For inputs whose short-range table would not fit host memory (2000 x 500k SNPs in a 2.2 Mb
                             genome: 2.3e9 short-range links = 72 GB of columns) and for callers that only feed the
                             long-range links on (analyse_long_range_links, R/lr_analyser.R:72-108) */
};

typedef struct ldw_ctx ldw_ctx;         /* one per device; owns stream + scratch */
typedef struct ldw_mi_plan ldw_mi_plan; /* device-resident packed operands for one snp.dat + hdw */

LDW_API int ldw_abi_version(void);
LDW_API const char* ldw_last_error(void);

/* Create / destroy a context on CUDA device `device` (0-based). */
LDW_API int ldw_create(int device, ldw_ctx** out);
LDW_API void ldw_destroy(ldw_ctx* ctx);
/* Number of visible CUDA devices (0 if none / no driver). */
LDW_API int ldw_device_count(void);

/* ------------------------------------------------------------------------------------------------
 * Encoding.
 *
 * ldw_aln_param replaces `.extractAlnParam(file, filter, gap_thresh, maf_thresh)`
 *   (R/RcppExports.R:32-34 -> _LDWeaver_extractAlnParam, src/RcppExports.cpp:109;
 *    body src/getACGTNsites.cpp:13-176) for an alignment already tokenised into a byte matrix.
 *   aln        : nseq x seq_len bytes, row-major (one FASTA record per row, raw characters)
 *   filter     : 0 = "default", 1 = "relaxed" (R/extractSNPs.R:29-36)
 *   pos_out    : capacity seq_len int32; receives the 1-based retained columns (ascending)
 *   n_snp_out  : number retained
 *   counts_out : optional (may be NULL) 5 x seq_len doubles, column-major (A,C,G,T,other per column)
 *
 * ldw_extract_snps replaces `.extractSNPs(file, n_seq, n_snp, POS)`
 *   (R/RcppExports.R:36-38 -> _LDWeaver_extractSNPs, src/RcppExports.cpp:123;
 *    body src/getACGTNsites.cpp:179-291).  The reference's 15 COO vectors partition the
 *   nseq x nsnp grid; they are returned as ONE uint8 class matrix:
 *   codes_out  : nsnp x nseq bytes (codes_out[k*nseq + s] in 0..4 = A,C,G,T,N/other)
 *   table_out  : 5 x nsnp doubles, column-major (ACGTN_table)
 *
 * ldw_read_fasta is the host-side tokeniser (gz or plain multi-FASTA -> byte matrix); it stays on
 *   the CPU like the reference's kseq/zlib reader (src/kseq2.h, src/getACGTNsites.cpp:33-45).
 *   Call with aln_out == NULL to query nseq / seq_len (seq_len = -1 if records differ in length,
 *   as src/getACGTNsites.cpp:54-56), then again with aln_out (capacity aln_cap bytes) and the queried
 *   seq_len left in *seq_len_out (it is the row stride); names_out receives nseq NUL-terminated names
 *   back to back (capacity names_cap bytes; may be NULL).
 */
LDW_API int ldw_aln_param(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, int filter, double gap_thresh,
                  double maf_thresh, int32_t* pos_out, int64_t* n_snp_out, double* counts_out);
LDW_API int ldw_extract_snps(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, const int32_t* pos,
                     int64_t n_snp, uint8_t* codes_out, double* table_out);
/* ldw_encode_alignment = ldw_aln_param + ldw_extract_snps in ONE call (what parse_fasta_alignment needs,
 *   R/extractSNPs.R:39-45): the alignment is uploaded once when it fits one device chunk (8 GiB by default), otherwise
 *   it streams through in row chunks -- device memory stays O(chunk), as the reference's record-by-record passes
 *   (src/getACGTNsites.cpp:49-85) need O(seq_len).  *pos_out (n_snp int32), *codes_out (n_snp x nseq) and *table_out
 *   (5 x n_snp doubles, column-major) are library-allocated and released with ldw_buffer_free; all NULL when
 *   *n_snp_out == 0 ("File does not contain any SNPs", R/extractSNPs.R:43). */
LDW_API int ldw_encode_alignment(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, int filter, double gap_thresh,
                         double maf_thresh, int64_t* n_snp_out, int32_t** pos_out, uint8_t** codes_out, double** table_out);
LDW_API int ldw_read_fasta(const char* path, int64_t* nseq_out, int64_t* seq_len_out, uint8_t* aln_out, int64_t aln_cap,
                   char* names_out, int64_t names_cap);
/* ldw_read_fasta_alloc: the same tokeniser in ONE pass over the file (SURVEY.md 8f row 4: the reference opens the gz
 *   file three times, src/getACGTNsites.cpp:33,44,212): inflate on a reader thread, tokenising on the caller's, the
 *   matrix in a library-allocated buffer.  *aln_out (nseq x seq_len bytes, row-major; NULL when the records differ in
 *   length, *seq_len_out = -1, or when there is no sequence) and *names_out (*names_len_out bytes: NUL-terminated names
 *   back to back) are released with ldw_buffer_free. */
LDW_API int ldw_read_fasta_alloc(const char* path, int64_t* nseq_out, int64_t* seq_len_out, uint8_t** aln_out, char** names_out,
                         int64_t* names_len_out);
LDW_API void ldw_buffer_free(void* p);

/* ldw_acgtn2num replaces `.ACGTN2num(nv, cv, ncores)` (R/RcppExports.R:4-6 -> _LDWeaver_ACGTN2num,
 *   src/RcppExports.cpp:16; body src/ACGTN2num_parallel.cpp:10-43).  In place on nv (5 x n doubles,
 *   column-major); ref holds one character per SNP. */
LDW_API int ldw_acgtn2num(ldw_ctx* ctx, double* nv, const char* ref, int64_t n);

/* ------------------------------------------------------------------------------------------------
 * Population-structure weights.
 * ldw_hdw replaces the body of estimate_Hamming_distance_weights(snp.dat, threshold)
 *   (R/performPopulationStuctureCorrection.R:20-81; the five Matrix::crossprod calls :49-74 and
 *   the threshold/colSums/reciprocal :76).
 *   codes      : nsnp x nseq class matrix (== the five snp.matrix_* slots); a class outside 0..4 is refused with
 *                LDW_ERR_ARG (checked on the device after the upload, as ldw_group_load_codes does)
 *   threshold  : fraction; thresh = (int)(nsnp*threshold) (truncation, :23)
 *   cnt_out    : nseq int32, #sequences (incl. self) with Hamming distance < thresh
 *   hdw_out    : nseq doubles, 1/(cnt+1)
 *   dist_out   : optional (may be NULL) nseq x nseq int32 Hamming distances, column-major
 */
LDW_API int ldw_hdw(ldw_ctx* ctx, const uint8_t* codes, int64_t n_snp, int64_t nseq, double threshold, int32_t* cnt_out,
            double* hdw_out, int32_t* dist_out);

/* ------------------------------------------------------------------------------------------------
 * Weighted pairwise-MI scan + sr/lr link filter.
 * Replaces the scan part of perform_MI_computation (R/computePairwiseMI.R:46-116: make_blocks :147-165,
 *   perform_MI_computation_ACGTN :167-386, computeMI_Sprase :390-398, .fastHadamard
 *   src/computeMI.cpp:11-21, .compareToRow src/computeMI.cpp:25-41).  mergeNsort_sr_links, ARACNE and
 *   the tsv writers stay in R and consume the link columns returned here.
 *
 * ldw_mi_plan_create uploads one snp.dat (codes, uqe-derived allele sets, POS) and the weights, and
 * packs the tensor-core operands on the device.  `blk` is round(max_blk_sz, -3) (R/computePairwiseMI.R:69).
 */
typedef struct ldw_links {
  int64_t n;             /* rows */
  const int32_t* pos1;   /* POS of the column ("to") SNP   (R/computePairwiseMI.R:320) */
  const int32_t* pos2;   /* POS of the row ("from") SNP    (:319) */
  const int32_t* clust1; /* paint of the column SNP        (:323) */
  const int32_t* clust2; /* paint of the row SNP           (:322) */
  const int32_t* len;    /* circular distance              (:330), integer-valued */
  const double* MI;      /* mutual information             (:331) */
  const int32_t* block;  /* 0-based make_blocks row the link came from */
} ldw_links;

typedef struct ldw_scan_stats {
  int64_t n_blocks;
  int64_t n_pairs;       /* pairs evaluated == rows the reference's MI_df would hold, summed over blocks */
  int64_t n_sr;          /* len <= sr_dist */
  int64_t n_lr_total;    /* len > sr_dist (before the quantile filter) */
  int64_t n_lr_kept;
  int64_t n_borderline;  /* LR candidates within borderline_tol of their block threshold (listed in `borderline`) */
  int64_t n_reruns;      /* blocks re-run: candidate threshold guess too high, or measured epilogue error above the margin's head room */
  int64_t n_candidates;  /* long-range candidates collected by the scan kernel (before refinement / selection) */
  double t_pack_ms, t_scan_ms, t_select_ms, t_d2h_ms; /* CUDA-event phase timings of the last scan (library stream) */
  double t_kernel_ms;    /* sum of the scan kernel's own launch durations (CUDA events around each launch) */
  int64_t n_scan_launches; /* launches of the scan kernel */
  int64_t n_launches;    /* all kernels this library launched during the scan */
  int64_t n_tiles;       /* tiles processed */
  double exec_int8_ops;  /* int8 tensor operations actually issued (2 * MACs) */
  double t_host_prep_ms; /* host time spent building and staging the per-block tables (overlaps the device work) */
  double exec_mufu_ops;  /* MUFU (LG2 / RCP) instructions x lanes the epilogue executed */
  double eps_obs_max;    /* largest |fp32 epilogue MI - fp64 MI| the long-range selection observed on its refined candidates
                            (it re-runs a block with wider margins when 4x this exceeds the selection margin, 4e-6) */
} ldw_scan_stats;

LDW_API int ldw_mi_plan_create(ldw_ctx* ctx, const uint8_t* codes, int64_t n_snp, int64_t nseq, const double* hdw,
                       const int32_t* pos, const int32_t* paint, int64_t blk, ldw_mi_plan** out);
LDW_API void ldw_mi_plan_destroy(ldw_mi_plan* plan);

/* Run the scan over this part's share of the make_blocks() blocks (multi-GPU: one plan per device; n_parts = 1,
 * part = 0 for everything).  Blocks are dealt by cost -- pairs, largest first, each to the least-loaded part,
 * lowest part on ties -- so every rank derives the same assignment (ldweaver_b200/api.py:partition_blocks mirrors it).
 *   g               : genome length (snp.dat$g)
 *   sr_dist         : short-range cut-off (len <= sr_dist is SR, R/computePairwiseMI.R:333)
 *   lr_retain_links, lr_links_approx : as R/computePairwiseMI.R:352 (lr_links_approx computed by the
 *                     caller, it depends on R's RNG, :94-97); ignored with LDW_SCAN_SR_ONLY
 *   thr_out / prob_out : optional arrays of n_blocks doubles (NaN where the block had no LR branch)
 * Link lists are in reference order (blocks in make_blocks order; rows inside a block as
 * R/computePairwiseMI.R:306-310), LR rows being those that pass `MI >= disc_thresh` (:358).
 */
LDW_API int ldw_mi_scan(ldw_mi_plan* plan, double g, double sr_dist, double lr_retain_links, double lr_links_approx,
                int flags, int n_parts, int part, ldw_links* sr_out, ldw_links* lr_out, ldw_links* borderline_out,
                double* thr_out, double* prob_out, ldw_scan_stats* stats_out);

/* ldw_write_lr_tsv writes the long-range rows exactly as perform_MI_computation_ACGTN appends them with
 *   write.table(MI_df_lr, lr_save_path, append = T, quote = F, row.names = F, col.names = F, sep = '\t')
 * (R/computePairwiseMI.R:362): tab-separated pos1 pos2 clust1 clust2 len MI, all of them doubles in the reference's
 * data.frame (pos = as.numeric(POS), :176-177) and written the way write.table encodes a single cell (15 significant
 * digits, scientific notation only when strictly narrower, so a position or a len of 100000 is "1e+05").  Host only, no device needed.  ldw_format_r_real exposes the cell encoder (tests).
 */
LDW_API int ldw_write_lr_tsv(const char* path, const ldw_links* lr, int append);
LDW_API int ldw_format_r_real(double x, char* out, int cap);

/* ------------------------------------------------------------------------------------------------
 * After the scan (SURVEY.md section 8f rows 1-3): the rest of perform_MI_computation, host only -- these take the
 * link columns where R would see them (host memory) and need no device.
 *
 * ldw_sr_postprocess replaces mergeNsort_sr_links(cds_var, sr_links, sr_dist, plt_path, srp_cutoff)
 *   (R/computePairwiseMI.R:400-495): per cluster c = 1..nclust, the short-range links with clust1 == c or
 *   clust2 == c (:372-376) and 0 < len < sr_dist (:417-419); 95th percentile (quantile type 7) of MI per distinct
 *   len (:422); log-log least-squares decay fit (RcppArmadillo::fastLm, :428-429); residuals above the fit, the fitted
 *   values being subscripted BY THE VALUE of len as the reference does (:448); beta maximum-likelihood fit of the
 *   positive residuals (fitdistrplus::fitdist(., "beta") = moment start + optim Nelder-Mead, :452);
 *   srp_max = -pbeta(., lower.tail = F, log.p = T) (:453); links between two clusters kept once, from the cluster
 *   that gives the larger srp_max (:474-483); sr_links_red = srp_max > srp_cutoff (:494);
 *   sr_links_ARACNE_check = MI >= min(sr_links_red$MI) (:495).
 *   The plots and the .rds files the reference also writes (:430-442) are not produced; the fitted curves are returned.
 *   `sr` is the short-range table of ldw_mi_scan (borrowed).  Everything in ldw_sr_post is library-owned and released
 *   by ldw_sr_post_free.  Errors (message in ldw_last_error) mirror the R failures: a cluster without links,
 *   residuals outside [0, 1] ("values must be in [0-1] to fit a beta distribution"), a likelihood that cannot be
 *   evaluated at the start values.
 */
typedef struct ldw_sr_post {
  int64_t n_df;             /* rows of sr_links_df, in the reference's order */
  const int32_t* clust_c;   /* cluster whose fit scored the link */
  const int64_t* row;       /* 0-based row of the link in `sr` */
  const double* srp_max;
  int64_t n_red;            /* sr_links_red: 0-based indices into the df rows, ascending */
  const int64_t* red;
  int64_t n_chk;            /* sr_links_ARACNE_check: 0-based indices into the df rows, ascending */
  const int64_t* chk;
  int32_t nclust;
  const int64_t* fit_off;   /* nclust + 1 offsets into fit_len / fit_q95 / fit_val (maxvls of each cluster) */
  const int32_t* fit_len;   /* distinct lengths, ascending */
  const double* fit_q95;    /* maxvls$max */
  const double* fit_val;    /* maxvls$fit = exp(fitted) */
  const double* coef;       /* nclust x {slope, intercept} of log(max) ~ log(len) */
  const double* shape;      /* nclust x {shape1, shape2} */
  const double* start;      /* nclust x {shape1, shape2} start values */
  const int64_t* n_pos;     /* links above the fit, per cluster */
  const int32_t* nm_evals;  /* Nelder-Mead function evaluations (optim's counts[1]) */
  const int32_t* nm_fail;   /* optim's convergence code (0, 1 = maxit reached, 10 = degenerate simplex) */
  void* priv;
} ldw_sr_post;
LDW_API int ldw_sr_postprocess(const ldw_links* sr, int32_t nclust, double sr_dist, double srp_cutoff, ldw_sr_post* out);
LDW_API void ldw_sr_post_free(ldw_sr_post* p);

/* ldw_sr_postprocess_dev: the same mergeNsort_sr_links, computed from the short-range table the last ldw_mi_scan on `ctx`
 *   left in DEVICE memory (whole job on this device: n_parts = 1; any flags but LDW_SCAN_NO_LINKS / LDW_SCAN_LR_ONLY; with
 *   LDW_SCAN_SR_ON_DEVICE the table never crosses PCIe).  Every pass over the links is a device kernel (group histogram,
 *   per-group order statistics, residual flags and sufficient statistics, srp_max); the decay fits, the beta fit and the
 *   cross-cluster de-duplication are the host code ldw_sr_postprocess uses.  Percentiles, fits and row sets are identical to
 *   ldw_sr_postprocess on the same table; the beta start values / shapes and srp_max agree to ~1e-12 relative (the sums are
 *   formed in another order).  Of sr_links_df (every link above its cluster's fitted decay: 4.5e6 rows at 616 x 100k) only
 *   the rows that are in sr_links_red or sr_links_ARACNE_check come back -- out->n_df counts those, in sr_links_df order,
 *   and out->red / out->chk index them; out->n_pos still holds each cluster's full count.  `out->row` indexes the device
 *   table (= the rows ldw_mi_scan would have returned); *df_rows_out receives the link columns of the out->n_df rows
 *   (owned by `out`, released by ldw_sr_post_free): all that sr_links_red / its ARACNE check / sr_links.tsv need. */
LDW_API int ldw_sr_postprocess_dev(ldw_ctx* ctx, int32_t nclust, double sr_dist, double srp_cutoff, ldw_sr_post* out, ldw_links* df_rows_out);

/* Building blocks of ldw_sr_postprocess, exposed for parity tests: stats::optim's Nelder-Mead (restated from R's nmmin)
 * run on Rosenbrock's function, the example of R's ?optim -- from c(-1.2, 1) R prints par 1.000260 1.000506, value
 * 8.825241e-08, 195 function evaluations --, and out[i] = -pbeta(x[i], shape1, shape2, lower.tail = F, log.p = T). */
LDW_API int ldw_nm_rosenbrock(const double* start, double* par_out, double* value_out, int* count_out);
LDW_API int ldw_neg_log_pbeta_upper(const double* x, int64_t n, double shape1, double shape2, double* out);

/* ldw_run_aracne replaces runARACNE(links_to_check, links_full) (R/io_functions.R:101-164, with .compareToRow,
 *   .vecPosMatch, .compareTriplet of src/computeMI.cpp:25-79 and .fast_intersect of src/fintersect.cpp:6-33):
 *   aracne_out[i] = 0 when some third position Y is linked to both ends of link i in `full` with
 *   MI_i < MI(X,Y) and MI_i < MI(Z,Y) (the first row of `full` holding each pair counts), else 1.
 *   Positions are doubles as in the R matrices.  Used for the short-range links (R/computePairwiseMI.R:124-126) and
 *   for the long-range ones (R/lr_analyser.R:101-108).
 */
LDW_API int ldw_run_aracne(int64_t n_chk, const double* chk_pos1, const double* chk_pos2, const double* chk_MI, int64_t n_full,
                   const double* full_pos1, const double* full_pos2, const double* full_MI, uint8_t* aracne_out);

/* ldw_write_sr_tsv writes sr_links.tsv as perform_MI_computation does (R/computePairwiseMI.R:140,
 *   write.table(sr_links_red, sr_save_path, append = T, quote = F, row.names = F, col.names = F, sep = '\t');
 *   reader R/io_functions.R:62-63): clust_c pos1 pos2 clust1 clust2 len MI srp_max ARACNE.  `rows` (n of them) index
 *   the short-range table `sr`; clust_c / srp_max / aracne are parallel to `rows`.
 */
LDW_API int ldw_write_sr_tsv(const char* path, const ldw_links* sr, int64_t n, const int64_t* rows, const int32_t* clust_c,
                     const double* srp_max, const double* aracne, int append);

/* ldw_read_numeric_tsv reads a link file the way read_LongRangeLinks / read_ShortRangeLinks do
 *   (read.table(path, sep = "\t", header = F, quote = "", comment.char = ""), R/io_functions.R:34,62; also
 *   genomewide_LDMap, R/LDSummaryPlot.R:51-52): `ncols` numeric tab-separated fields per line, no header, "NA" -> NaN.
 *   *cols_out is a library-owned column-major table (ncols x *nrows_out doubles: column k starts at k * nrows),
 *   released by ldw_table_free.  A line with another number of fields is an error (message names the line).
 */
LDW_API int ldw_read_numeric_tsv(const char* path, int ncols, int64_t* nrows_out, double** cols_out);
LDW_API void ldw_table_free(double* cols);

/* Cell of each link in the MI matrix of the block it came from (`links->block`): from_local[i] / to_local[i] are the
 * 0-based local indices of the link's row ("from", pos2) and column ("to", pos1) SNPs (R/computePairwiseMI.R:319-323),
 * i.e. what ldw_mi_pairs_exact takes.  Host only.  Not meaningful for LDW_SCAN_SR_ONLY scans (quirk Q12). */
LDW_API int ldw_links_to_cells(const int32_t* pos, int64_t n_snp, int64_t blk, const ldw_links* links, int32_t* from_local,
                       int32_t* to_local);

/* Copies a link table (library-owned, e.g. what ldw_mi_scan returned) into caller-allocated columns of src->n elements on
 * host threads; a NULL destination skips that column. */
LDW_API int ldw_links_copy(const ldw_links* src, int32_t* pos1, int32_t* pos2, int32_t* clust1, int32_t* clust2, int32_t* len,
                   double* MI, int32_t* block);

/* Dense MI matrix of one block (debug / parity aid; nf x nt doubles, column-major, fp32-accurate values).
 * from/to are 0-based ascending global SNP ids, as `from`/`to` of perform_MI_computation_ACGTN. */
LDW_API int ldw_mi_block_dense(ldw_mi_plan* plan, int64_t block_index, double* mi_out, int64_t* nf_out, int64_t* nt_out);

/* Exact (fp64) MI of explicit pairs of one block: pair k = (from_local[k], to_local[k]). */
LDW_API int ldw_mi_pairs_exact(ldw_mi_plan* plan, int64_t block_index, const int32_t* from_local, const int32_t* to_local,
                       int64_t n_pairs, double* mi_out);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU: device groups (one box, NCCL over NVLink / NVSwitch).
 *
 * Replaces nothing the reference has -- its block loop is serial (R/computePairwiseMI.R:103-116) -- but the blocks are
 * independent given codes, hdw, POS and paint, and the long-range threshold is per block (quirk Q3), so dealing whole
 * blocks to devices reproduces the single-device tables bit for bit.
 *
 * A group holds this process's members of the job: ALL of them (ldw_group_create: the form an R session or a Python
 * process uses; one host thread per device while an operation runs) or ONE rank of a multi-process job
 * (ldw_group_create_rank: rank 0 makes an id with ldw_group_unique_id and the launcher hands it to every rank).
 * Every call below is collective: all processes of the job make it with the same arguments.
 *
 * ldw_group_load_codes: the class matrix (nsnp x nseq, as ldw_mi_plan_create takes it) goes host -> device ONCE, on the
 *   member with rank 0 (other processes may pass NULL), and reaches the other devices by ncclBroadcast; it stays
 *   resident for the calls that follow.
 * ldw_group_hdw: estimate_Hamming_distance_weights on the resident matrix.  The distance GEMM's upper-triangle tiles are
 *   dealt to the ranks, the partial neighbour counts are summed with ncclAllReduce and every rank forms the weights
 *   (so no separate weight broadcast is needed); problems too small to share are computed whole on every rank
 *   (*sharded_out tells which; LDW_HDW_FORCE_SHARD always deals).  Results are bit-identical to ldw_hdw.
 * ldw_group_mi_scan: ldw_mi_plan_create + ldw_mi_scan over the group.  Every member packs its operands from the resident
 *   matrix and scans its share of the make_blocks blocks (dealt by cost exactly as ldw_mi_scan's n_parts / part).
 *   Short-range rows are copied by each device directly to their final rows of ONE pinned host table; long-range and
 *   borderline rows are merged into make_blocks order.  The tables (group-owned, valid until the next scan on the group)
 *   are identical to a single-device ldw_mi_scan when the group holds the whole job; a one-rank group of a
 *   multi-process job returns the rows of its own blocks.  stats_out: one entry per LOCAL member; t_plan_ms_out: wall
 *   time of the operand packing.
 */
typedef struct ldw_group ldw_group;
#define LDW_GROUP_ID_BYTES 128
enum { LDW_HDW_FORCE_SHARD = 1 };
LDW_API int ldw_group_create(const int* devices, int n_devices, ldw_group** out);
LDW_API int ldw_group_unique_id(char* id_out /* LDW_GROUP_ID_BYTES */);
LDW_API int ldw_group_create_rank(int device, int rank, int world, const char* id /* LDW_GROUP_ID_BYTES */, ldw_group** out);
LDW_API void ldw_group_destroy(ldw_group* g);
LDW_API int ldw_group_info(const ldw_group* g, int* world_out, int* n_local_out, int* first_rank_out);
LDW_API ldw_ctx* ldw_group_ctx(ldw_group* g, int local_index);
LDW_API int ldw_group_load_codes(ldw_group* g, const uint8_t* codes, int64_t n_snp, int64_t nseq);
LDW_API int ldw_group_hdw(ldw_group* g, double threshold, int flags, int32_t* cnt_out, double* hdw_out, int* sharded_out);
LDW_API int ldw_group_mi_scan(ldw_group* g, const double* hdw, const int32_t* pos, const int32_t* paint, int64_t blk, double g_len,
                      double sr_dist, double lr_retain_links, double lr_links_approx, int flags, ldw_links* sr_out,
                      ldw_links* lr_out, ldw_links* borderline_out, double* thr_out, double* prob_out,
                      ldw_scan_stats* stats_out, double* t_plan_ms_out);

#ifdef __cplusplus
}
#endif
#endif /* LDW_H */
