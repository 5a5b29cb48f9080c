/* sbq.h - C ABI of the B200-native quantification engine (libsbq.so).
 *
 * Drop-in boundary for the per-locus Latent-Class-Model EM of ruolin/strawberry v1.1.2. The
 * reference has no plugin/FFI API: its boundary is a C++ link seam between alignments.o and
 * estimate.o. Every entry point below names the reference interface it replaces (file:line under
 * the reference checkout); INTEGRATION.md shows the replacement estimate.cpp translation unit a
 * maintainer links instead of the reference's own.
 *
 * Conventions: plain pointers and sizes only; host arrays are BORROWED for the duration of the
 * call (sbq_submit* copy into pinned staging, so they may be freed as soon as it returns); device
 * memory, streams and events are owned by the context. Every function returns SBQ_SUCCESS (0) or a
 * negative sbq_error; nothing exits, aborts or throws across the boundary (the reference exits or
 * asserts instead, SURVEY section 5). There is no CPU fallback: without a CUDA device every entry
 * point that computes returns SBQ_ERR_NO_DEVICE.
 */
#ifndef SBQ_H_
#define SBQ_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SBQ_ABI_VERSION 2

typedef enum {
   SBQ_SUCCESS = 0,
   SBQ_ERR_INVALID = -1,     /* bad argument / malformed CSR                                       */
   SBQ_ERR_NO_DEVICE = -2,   /* no usable CUDA device (product has no CPU path)                    */
   SBQ_ERR_CUDA = -3,        /* a CUDA runtime call failed; see sbq_last_error()                   */
   SBQ_ERR_NOMEM = -4,
   SBQ_ERR_STATE = -5,       /* call sequence violated (e.g. sbq_results before sbq_run)           */
   SBQ_ERR_UNSUPPORTED = -6  /* shape outside the documented limits (n_iso > SBQ_MAX_ISO)          */
} sbq_error;

/* Per-locus outcome. Mirrors what EmSolver::init/run can do (src/estimate.cpp:366-488):
 *   OK          converged: ||theta' - theta||_2 < theta_tol; theta is the PREVIOUS iterate (:479-480)
 *   ITER_CAP    max_iter E-steps executed without meeting the tolerance (:444)
 *   ZERO_DENOM  some kept row had sum_j F_ij theta_j == 0: run() returns false and _theta keeps its
 *               uniform initial value total/T; the caller ignores the return value (:451-453, :308)
 *   NO_ROWS     init() returned false (no row with an entry > row_eps, :377-391): the locus reports
 *               no isoforms at all (src/alignments.cpp:1526-1529); keep[] is 0 for all of them    */
typedef enum { SBQ_LOCUS_OK = 0, SBQ_LOCUS_ITER_CAP = 1, SBQ_LOCUS_ZERO_DENOM = 2, SBQ_LOCUS_NO_ROWS = 3 } sbq_locus_status;

/* Isoforms per locus every multi-row tier accepts: theta, the column sums and at least one private accumulator row live
 * in shared memory (cluster tier 7 T + 64 doubles, grid tier 7 T + 16 doubles of <= 200 KB). Wider loci are refused at
 * submit time with SBQ_ERR_UNSUPPORTED; a locus within the limit never fails an upload - it falls to the other tier. */
#define SBQ_MAX_ISO 3600

/* Replaces the reference's mutable globals read on the hot path (SURVEY section 5 "Config"). */
typedef struct {
   int32_t device;             /* CUDA device ordinal of this context; -1 = current device          */
   int32_t max_iter;           /* EmSolver::_max_iter_num            include/estimate.hpp:236  1000 */
   double  theta_tol;          /* EmSolver::_theta_change_limit      include/estimate.hpp:240  1e-2 */
   double  row_eps;            /* row filter in EmSolver::init       src/estimate.cpp:381      1e-5 */
   double  min_iso_frac;       /* kMinIsoformFrac (-m / 0 with -r)   src/estimate.cpp:346-355       */
   int32_t effective_len_norm; /* effective_len_norm                 src/estimate.cpp:317-324   0   */
   double  insert_mean;        /* InsertSize::_mean, only read when effective_len_norm != 0         */
   int32_t bias_mode;          /* 0 = reference behaviour. 1 = bias-corrected EM, OUR definition    */
                               /*     (DESIGN.md "Bias mode"); the reference has none (bias.cpp     */
                               /*     is commented out) - parity unpinned                           */
   /* bias mode only; defaults are the constants the reference declares but never reads              */
   int32_t max_out_it;         /* EmSolver::_max_out_it_num          include/estimate.hpp:239   100 */
   int32_t max_theta_it;       /* EmSolver::_max_theta_it_num        include/estimate.hpp:238  5000 */
   int32_t max_bias_it;        /* EmSolver::_max_bias_it_num         include/estimate.hpp:237    10 */
   double  bias_tol;           /* EmSolver::_bias_change_limit       include/estimate.hpp:241  1e-2 */
   /* Multi-GPU (SURVEY section 8b/8e). 0 or 1: one device (`device`). N > 1: the context drives the N devices
    * device .. device + N - 1 (device = -1 counts from 0) from this one process: sbq_upload partitions the queued
    * loci over them by non-zeros (greedy LPT, sbq_partition_lpt), every device solves its share with the same
    * kernels, and the TPM denominator - the path's only exchange, src/alignments.cpp:1821-1824 - is ONE
    * ncclAllReduce(ncclDouble, count 1) over the devices (NCCL is loaded on first use; single-device contexts
    * never touch it). Results come back in submit order, independent of the partition. */
   int32_t n_gpus;
} sbq_config;

/* One locus as the host class-table builder emits it: what LocusContext::estimate_abundances
 * densifies into alpha[nrow][niso] and n[nrow] (src/estimate.cpp:281-296). Rows are fragment
 * classes (ExonBin), columns isoforms; CSR with explicit entries only. */
typedef struct {
   int32_t n_iso;              /* _transcripts.size()                                               */
   int32_t n_row;              /* exon_bins.size()                                                  */
   const int64_t* row_ptr;     /* n_row + 1 offsets into col/alpha, row_ptr[0] may be non-zero       */
   const int32_t* col;         /* isoform id of each entry, ascending within a row                  */
   const double*  alpha;       /* ExonBin::_bin_weight_map value     src/estimate.cpp:201-234       */
   const int32_t* count;       /* n_i = (int)ExonBin::read_count()   src/estimate.cpp:288           */
   const int32_t* iso_len;     /* Isoform::_length                   include/estimate.hpp:98        */
} sbq_locus;

typedef struct sbq_ctx sbq_ctx;

/* Timing / accounting of the last sbq_upload / sbq_solve / sbq_download (all on the context's stream,
 * CUDA events; the numbers bench.py reports). */
typedef struct {
   int64_t n_loci, n_row, n_iso, nnz;
   int64_t loci_warp, loci_cta, loci_grid;   /* tier populations chosen by the planner              */
   int64_t kernel_launches;                  /* launches of OUR kernels in the last sbq_solve        */
   int64_t h2d_bytes, d2h_bytes;             /* bytes moved by the last sbq_upload / sbq_download    */
   double  upload_ms, solve_ms, download_ms; /* device time, CUDA events                            */
   double  em_ms;                            /* EM kernels only (subset of solve_ms)                */
   double  grid_em_ms;                       /* multi-CTA giant-locus kernel only                   */
   int64_t em_iters_total;                   /* sum over loci of E-steps executed                   */
   int64_t frag_iters;                       /* sum over loci of (sum_i n_i) * iters                */
   int64_t alg_bytes;                        /* sum over loci of (12 nnz + 12 R + 16 T) * iters      */
   int64_t grid_alg_bytes;                   /* same, loci solved by the giant-locus kernel only    */
   double  weights_ms;                       /* GPU class-weight kernel + its descriptor H2D (deferred-weight batches) */
} sbq_stats;

int  sbq_abi_version(void);
const char* sbq_error_string(int err);
const char* sbq_last_error(const sbq_ctx*);

/* Fill cfg with the reference defaults listed in the struct comments (device = -1). */
void sbq_config_default(sbq_config* cfg);

/* Created once by the driver (where the reference's driver() builds its Sample, src/Strawberry.cpp:237). */
int  sbq_create(const sbq_config* cfg, sbq_ctx** out);
void sbq_destroy(sbq_ctx*);

/* Queue loci for the next run. Thread-safe: may be called concurrently from the reference's
 * per-locus worker threads (src/alignments.cpp:1782-1799). Loci keep submit order in the results.
 * Replaces the per-locus call LocusContext::estimate_abundances (src/estimate.cpp:279-309). */
int  sbq_submit(sbq_ctx*, const sbq_locus* loci, int64_t n_loci);

/* Same, from one flat batch: loc_row_off / loc_iso_off are n_loci + 1 prefix offsets, row_ptr is ONE
 * CSR over all rows of the batch (n_rows + 1 entries), col is local to the locus. */
int  sbq_submit_flat(sbq_ctx*, int64_t n_loci, const int64_t* loc_row_off, const int64_t* loc_iso_off,
                     const int64_t* row_ptr, const int32_t* col, const double* alpha,
                     const int32_t* count, const int32_t* iso_len);

/* Drop everything queued / resident. */
int  sbq_clear(sbq_ctx*);

/* Full structural check of the queued batch (column range, strictly ascending columns, monotone
 * row_ptr) - the conditions the reference guarantees by construction (std::map / std::set iteration
 * in src/estimate.cpp:283-296). O(nnz) on the host; sbq_submit* only do the O(loci) checks. */
int  sbq_validate(sbq_ctx*);

/* Page-locked host memory. A first sbq_submit_flat whose arrays all come from sbq_host_alloc (or are
 * otherwise page-locked) and start at offset 0 is used IN PLACE: no staging copy, H2D straight from
 * the caller's arrays, which must stay valid until sbq_upload / sbq_run returns. */
void* sbq_host_alloc(size_t bytes);
void  sbq_host_free(void* p);

/* The three stages of sbq_run, separately callable so that the device-resident solve can be timed
 * on its own (bench.py "value") next to the host-buffer path (bench.py "e2e"):
 *   sbq_upload    plan tiers (warp / CTA-cluster / grid), H2D of the staged batch
 *   sbq_solve     EM kernels + FPKM/frac/filter epilogue on the resident batch; re-runnable
 *   sbq_download  D2H of theta, fpkm, frac, keep, iters, status and the local FPKM sum        */
int  sbq_upload(sbq_ctx*);
/* Asynchronous sbq_upload: returns as soon as the copies are ENQUEUED - offsets and columns first, then the weights of the
 * largest loci launch by launch, then the rest - and a following sbq_solve lets every kernel launch wait only for the copies
 * it needs, so the longest-running loci iterate while the tail of the batch is still crossing PCIe. Borrowed (page-locked,
 * in-place) arrays must stay valid until that sbq_solve returns. sbq_run uses it. Multi-GPU, deferred-weight and bias
 * batches fall back to the synchronous sbq_upload. */
int  sbq_upload_begin(sbq_ctx*);
int  sbq_solve(sbq_ctx*, int64_t total_mapped_reads);
int  sbq_download(sbq_ctx*);

/* upload + solve + download + TPM with the LOCAL FPKM sum. total_mapped_reads is
 * Sample::total_mapped_reads() (src/estimate.cpp:328). Replaces the quantification loop of
 * Sample::procSample (src/alignments.cpp:1756-1829) for everything numeric. */
int  sbq_run(sbq_ctx*, int64_t total_mapped_reads);

/* Multi-GPU: loci are partitioned over ranks by the caller (strawberry_b200.partition); the only
 * exchange is the TPM denominator, sum of FPKM over surviving isoforms (src/alignments.cpp:1821-1824).
 * sbq_fpkm_sum returns this rank's share; after the all-reduce the caller hands the global sum back. */
int  sbq_fpkm_sum(sbq_ctx*, double* local_sum);
int  sbq_fpkm_sum_to_device(sbq_ctx*, void* dev_double);          /* D2D copy for an NCCL all-reduce */
int  sbq_finalize_tpm(sbq_ctx*, double global_fpkm_sum);

/* Copy results out (any pointer may be NULL). Per isoform, submit order: theta, fpkm, frac, tpm, and
 * keep (0 = erased by the low-fraction filter or NO_ROWS locus; -1 = "NA" effective-length case,
 * src/estimate.cpp:320-323). Per locus: iters (E-steps executed) and status (sbq_locus_status). */
int  sbq_results(sbq_ctx*, double* theta, double* fpkm, double* frac, double* tpm, int32_t* keep,
                 int32_t* iters, int32_t* status);

int  sbq_get_stats(const sbq_ctx*, sbq_stats* out);

/* One record per EM kernel launch of the last sbq_solve, timed with CUDA events on the stream the
 * kernel was launched on (launches of different tiers overlap on separate streams). Byte / iteration
 * accounting is filled in by sbq_download. Returns the number of records (may exceed cap). */
typedef struct {
   int32_t kind;            /* 1 = warp tier, 2 = cluster tier, 3 = grid (giant-locus) tier               */
   int32_t cluster_size;    /* CTAs per locus (cluster tier)                                              */
   int32_t lanes_per_row;   /* threads per CTA of the launch (cluster tier)                               */
   int32_t variant;         /* grid tier: 1 = register-staged loads, 2 = TMA ring, 3 = bank-aligned two-slot layout */
   int64_t n_loci, nnz;
   double  ms;              /* kernel duration                                                            */
   int64_t alg_bytes;       /* sum over its loci of (12 nnz + 12 R + 16 T) * iters                         */
   int64_t frag_iters;
   int64_t max_iters;       /* longest EM run among its loci (the launch's critical path)                 */
   double  start_ms;        /* when the launch's start event fired, relative to the start of sbq_solve    */
} sbq_launch_stat;
int  sbq_get_launch_stats(const sbq_ctx*, sbq_launch_stat* out, int cap);

/* Giant-locus stress input generated ON THE DEVICE from a seed (SURVEY section 8d row 4, BASELINE configs[3]: 200 loci x
 * 1 M single-fragment rows x ~48 compatible isoforms are ~115 GB of CSR that never cross PCIe). The data of a locus is a
 * pure function of (seed, GLOBAL locus id), so any split of the ids over devices or waves yields the same loci; the
 * generator is restated on the CPU in strawberry_b200/synth.py::giant_device (bit-exact, tests/test_gpu_synth.py).
 * Replaces sbq_submit* + sbq_upload: the batch exists in HBM only, sbq_solve / sbq_download / sbq_results follow. */
typedef struct {
   uint64_t seed;
   int32_t  n_loci;            /* loci generated by this call                                                      */
   const int32_t* locus_ids;   /* their n_loci global ids, or NULL for 0 .. n_loci - 1                              */
   int64_t  rows_per_locus;    /* every row is one fragment (n_i = 1)                                               */
   int32_t  iso_lo, iso_hi;    /* T ~ U{iso_lo .. iso_hi}                                                           */
   double   mean_extra;        /* row degree k ~ 1 + Poisson(mean_extra), capped at min(T, 255)                     */
} sbq_synth_giant_spec;
int  sbq_synth_giant(sbq_ctx*, const sbq_synth_giant_spec* spec);

/* Device -> host copy of the resident batch in the sbq_submit_flat layout (any pointer may be NULL); the arrays must hold
 * n_loci + 1, n_loci + 1, n_row + 1, nnz, nnz, n_row and n_iso elements (sbq_get_stats has the sizes). For tests of
 * device-generated batches. After a solve, the weights of giant-locus rows come back in the kernel's bank-sorted order. */
int  sbq_fetch_batch(sbq_ctx*, int64_t* loc_row_off, int64_t* loc_iso_off, int64_t* row_ptr, int32_t* col, double* alpha,
                     int32_t* count, int32_t* iso_len);

/* Greedy longest-processing-time partition of n loci with the given costs over n_parts devices: loci by descending
 * cost (ties: lower index first) onto the currently lightest part (ties: lower part first). owner[l] receives the part
 * of locus l. Host-only and deterministic - it is what sbq_upload runs for n_gpus > 1 with cost = nnz + rows + isoforms
 * (loci are never split across devices). */
int  sbq_partition_lpt(const int64_t* cost, int64_t n, int32_t n_parts, int32_t* owner);

/* Multi-GPU contexts: device ordinal that solved each queued locus (valid after sbq_upload); single-device: all equal. */
int  sbq_locus_devices(sbq_ctx*, int32_t* device_of_locus);

/* Single-locus convenience backing a drop-in EmSolver (EmSolver::init + run, src/estimate.cpp:366-488):
 * theta receives n_iso doubles; returns the sbq_locus_status (>= 0) or a negative sbq_error. */
int  sbq_em_solve(sbq_ctx*, const sbq_locus* locus, double* theta, int32_t* iters);

/* Bias mode (bias_mode = 1, OUR definition - DESIGN.md section 7; no reference behaviour exists). Loci of up to 2165 isoforms
 * (sbq_solve returns SBQ_ERR_UNSUPPORTED beyond: 13 T doubles of shared memory per CTA). Per-row
 * covariates x[n_row][n_cov] (row-major, rows in submit order, n_cov <= 6) must be set after the last sbq_submit*
 * and before sbq_upload / sbq_run; sbq_bias_results returns beta[n_loci][n_cov] and the outer rounds per locus. */
int  sbq_set_covariates(sbq_ctx*, const double* x, int64_t n_row, int32_t n_cov);
int  sbq_bias_results(sbq_ctx*, double* beta, int32_t* outer_iters);

/* Bootstrap replicates (OUR definition, DESIGN.md "Bootstrap replicates"; the reference has none). Replicate b redraws each locus'
 * N = sum n_i fragments from its own classes (multinomial, conditional on N, by a counter-based hash of (seed, b, submit position
 * of the locus)) and runs the same EM + epilogue on those counts; total_mapped_reads and the point estimate stay as they are.
 * Needs a resident batch solved by sbq_solve; SBQ_ERR_UNSUPPORTED in bias mode. Device memory per replicate: 16 n_iso + 8 n_loci
 * bytes (SBQ_ERR_NOMEM leaves the context usable). */
/* Bootstrap replicates first .. first + n - 1 of the resident, solved batch (our definition, DESIGN.md). */
int  sbq_bootstrap(sbq_ctx*, uint64_t seed, int64_t first, int32_t n);
/* Replicates of the last sbq_bootstrap, submit order: theta / tpm [n][n_iso], iters / status [n][n_loci]; any pointer may be NULL. */
int  sbq_bootstrap_results(sbq_ctx*, double* theta, double* tpm, int32_t* iters, int32_t* status);
/* Test aid: the resampled counts of one replicate, n_row values in submit row order (needs a resident batch only). */
int  sbq_bootstrap_counts(sbq_ctx*, uint64_t seed, int64_t replicate, int32_t* count);
/* Device time of the last sbq_bootstrap (CUDA events; multi-GPU: the slowest device). */
typedef struct { int64_t first, n; double resample_ms, em_ms, total_ms; } sbq_bootstrap_stat;
int  sbq_bootstrap_stats(const sbq_ctx*, sbq_bootstrap_stat* out);

/* Gibbs posterior samples (OUR definition, DESIGN.md "Gibbs posterior samples"; the reference has none). A data-augmentation
 * Gibbs chain per locus, started from the resident point estimate: every round assigns each kept fragment to an isoform of its
 * class and redraws the locus' proportions from Dirichlet(counts + prior). Sample s is the state after round
 * burn_in + (s + 1) * thin; its theta is N_kept * pi, its FPKM / TPM come from the usual epilogue. Loci whose point status is
 * NO_ROWS or ZERO_DENOM are not sampled (every sample repeats their epilogue). Needs a resident batch solved by sbq_solve;
 * SBQ_ERR_UNSUPPORTED in bias mode. Device memory: 16 nnz + 16 n_iso per sample + O(n_row + n_iso) bytes (SBQ_ERR_NOMEM leaves
 * the context usable); the point estimate and later solves / bootstraps are unchanged. */
int  sbq_gibbs(sbq_ctx*, uint64_t seed, int32_t n, int32_t thin, int32_t burn_in, double prior);
/* Samples of the last sbq_gibbs, submit order: theta / tpm [n][n_iso], status [n][n_loci] (the point estimate's); any pointer may be NULL. */
int  sbq_gibbs_results(sbq_ctx*, double* theta, double* tpm, int32_t* status);
/* Device time of the last sbq_gibbs (CUDA events; multi-GPU: the slowest device). colsum_ms: the one-off setup (weights back in
 * submitted order, column sums, heavy-row offsets, phi^0); assign_ms / theta_ms: summed over all rounds. */
typedef struct { int64_t n, rounds; double colsum_ms, assign_ms, theta_ms, total_ms; } sbq_gibbs_stat;
int  sbq_gibbs_stats(const sbq_ctx*, sbq_gibbs_stat* out);

/* Planner knobs, mainly for tests: force a tier (0 = auto, 1 = warp, 2 = CTA/cluster, 3 = grid) and
 * the cluster size of the CTA tier (0 = auto, else 1, 2, 4, 8, 16). */
int  sbq_set_plan(sbq_ctx*, int force_tier, int force_cluster);

#ifdef __cplusplus
}
#endif
#endif /* SBQ_H_ */
