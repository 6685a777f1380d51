/*
 * chicdiff_b200.h -- C ABI of libchicdiff_b200.so: the B200-native implementation of Chicdiff's
 * region-test hot path (aggregation -> normalisation offsets -> NB GLM -> dispersion -> Wald).
 *
 * The reference (RegulatoryGenomicsGroup/chicdiff, Chicdiff/R/chicdiff.R) is pure R and exposes no
 * FFI; the drop-in boundary is the numeric core of two exported R functions, which an R front
 * end reaches through .Call -> R/r_glue.c -> the entry points below (INTEGRATION.md shows the
 * binding):
 *
 *   DESeq2Wrap(chicdiff.settings, RU, FullRegionData, suffix, theta)       chicdiff.R:1494-1777
 *     :1540-1547  by=(baitID, regionID, sample) sums of N and FullMean      -> cd_aggregate
 *     :1561-1562  estimateSizeFactors                                       -> cd_region_test (sizeFactors)
 *     :1583-1589, FullMean scaling factors, NA rows, theta mix, rescale     -> cd_region_test (norm, theta)
 *      1614-1615, 1635-1638, 1666-1669
 *     :1619-1662  theta grid: 5 intercept-only fits, argmin sum(deviance)   -> cd_region_test (theta = NaN)
 *     :1573-1574, estimateDispersions + nbinomWaldTest                      -> cd_region_test
 *      1602-1603, 1643-1644, 1673-1674
 *     :1721,1730,1739  results(): Cook's cutoff, independent filtering, BH  -> cd_results_adjust,
 *                                                                              cd_results_resident, cd_results_device
 *   getFullRegionData(chicdiff.settings, RU, RUcontrol, suffix)            chicdiff.R:1460-1478
 *     supplies the per-row N / FullMean columns                            -> cd_set_sample_rows
 *
 * Conventions
 *   - Plain C: pointers and sizes only.  Every function returns 0 on success or a negative
 *     CD_E* code; cd_last_error() returns a message.  Nothing aborts or throws across the ABI,
 *     and there is no CPU fallback: without a CUDA device every compute call fails with CD_ECUDA.
 *   - Host buffers are owned by the caller; the library owns its device memory inside cd_ctx.
 *     Calls are synchronous unless the name says otherwise.
 *   - Matrices are "sample-major" = R's column-major n x S layout: element (region i, sample s)
 *     at [s*n + i].  An R numeric/integer matrix can be passed without transposition.
 *   - NA: integer NA is INT32_MIN (R's NA_integer_); floating NA is any NaN (R's NA_real_ is a
 *     NaN; is.na() is true for both).  All-zero regions get NaN in every output column, as in
 *     DESeq2.
 *   - One context drives one GPU.  For several GPUs either use cd_multi_* (one process, one host thread per
 *     GPU inside the library) or run one process per GPU, shard the regions by bait (cd_plan_shards) and join
 *     the contexts with cd_comm_init.  Either way the few global steps exchange sums and counters only: the
 *     dispersion-trend sums and the median histograms inside their kernels through NVLink peer memory, the
 *     moments-offset sums and the theta-grid deviances with NCCL.
 */
#ifndef CHICDIFF_B200_H
#define CHICDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cd_ctx cd_ctx;

#define CD_OK 0
#define CD_EINVAL (-1)      /* bad argument / call order */
#define CD_ECUDA (-2)       /* CUDA runtime error (message has the CUDA error string) */
#define CD_ENOMEM (-3)
#define CD_ECOMM (-4)       /* NCCL error / NCCL not loadable */
#define CD_ENUMERIC (-5)    /* numerical failure the reference also stops on, or a reference fallback
                               that is not implemented (local dispersion fit, Monte-Carlo prior) */

/* per-region status bits returned in cd_results.flags */
#define CD_FLAG_ALLZERO 1
#define CD_FLAG_GENE_GRID 2
#define CD_FLAG_MAP_GRID 4
#define CD_FLAG_BETA_NOCONV 8
#define CD_FLAG_OUTLIER 16
#define CD_FLAG_GENE_NOINCREASE 32
#define CD_FLAG_COOKS_KEEP 64

#define CD_NORM_STANDARD 0
#define CD_NORM_FULLMEAN 1
#define CD_NORM_COMBINED 2

const char* cd_version(void);

/* ---- lifecycle ------------------------------------------------------------------------- */
int cd_create(cd_ctx** out, int device);
void cd_destroy(cd_ctx* ctx);
const char* cd_last_error(const cd_ctx* ctx);      /* ctx may be NULL: last error of cd_create */

/* ---- multi-GPU: one process per GPU, NCCL communicator over NVLink --------------------- */
/* rank 0 calls cd_comm_unique_id and ships the 128 bytes to the other ranks by any means
 * (the Python host uses torch.distributed); every rank then calls cd_comm_init. */
int cd_comm_unique_id(cd_ctx* ctx, char id[128]);
int cd_comm_init(cd_ctx* ctx, int nranks, int rank, const char id[128]);
/* peer_memory_allreduce: bit 0 set when the sharded trend fit all-reduces its sums through NVLink peer memory inside
 * its kernel (cudaIpc mailboxes), bit 1 set when the median kernels exchange their counters the same way; a clear
 * bit means NCCL all-reduces enqueued by the host between the kernels */
int cd_comm_info(const cd_ctx* ctx, int* nranks, int* rank, int* peer_memory_allreduce);
/* contiguous bait-balanced partition of regions (region_bait must be non-decreasing):
 * shard k owns regions [bounds[k], bounds[k+1]); cuts fall only between baits and balance rows. */
int cd_plan_shards(int64_t n, const int32_t* region_bait, const int64_t* row_off, int nshards,
                   int64_t* bounds /* nshards + 1 */);

/* ---- problem setup ---------------------------------------------------------------------- */
/* design: model.matrix of the reference's `~ condition` (chicdiff.R:1559) or `~ batch + condition`;
 * X is S x p row-major, column 0 the intercept, the LAST column the tested coefficient. */
int cd_set_design(cd_ctx* ctx, int S, int p, const double* X);
/* regions as CSR segments over region-contiguous rows (sorted by regionID, then otherEndID) */
int cd_set_regions(cd_ctx* ctx, int64_t n, const int64_t* row_off /* n + 1 */);
/* per-replicate columns of the long table: N (chicdiff.R:853) and FullMean = Bmean + Tmean
 * (chicdiff.R:896), R = row_off[n] rows, host pointers.  The copy is asynchronous on a copy stream of the context: the
 * buffers must stay valid until the next cd_aggregate has returned (pageable memory is staged by the driver before the
 * call returns; pinned memory is read by the DMA engine later).  Uploads go to a second device buffer while the rows
 * of the previous cd_aggregate are still in use, so a caller that processes several batches (test set, control set,
 * bench steps) can call cd_set_sample_rows for the NEXT batch between cd_aggregate and cd_region_test of the current
 * one, and the upload crosses the bus under the region test. */
int cd_set_sample_rows(cd_ctx* ctx, int s, int64_t R, const int32_t* N, const double* fullmean);
/* same, but the pointers are device pointers holding ALL samples sample-major (S x R); the
 * context borrows them (no copy) until the next cd_set_regions / cd_destroy */
int cd_set_rows_device(cd_ctx* ctx, int64_t R, const int32_t* N_dev, const double* fullmean_dev);
/* skip stage 1: provide already aggregated matrices (host, sample-major S x n) */
int cd_set_aggregated(cd_ctx* ctx, int64_t n, const int32_t* K, const double* fullmean);

/* ---- stage 1 ----------------------------------------------------------------------------- */
/* K_out / fullmean_out: host S x n sample-major, either may be NULL (results stay on the device) */
int cd_aggregate(cd_ctx* ctx, int32_t* K_out, double* fullmean_out);

/* ---- per-replicate assembly fused with stage 1 ---------------------------------------------------- */
/* Instead of handing over the long table, hand over what getFullRegionData1() builds it from
 * (chicdiff.R:609-702, 820-910) and let the device do the joins, Chicago's Bmean = s_j s_i f(d),
 * FullMean = Bmean + Tmean, the count merge with zero fill AND the region sums in one pass.
 * Call order: cd_set_design, cd_set_rmap, cd_set_regions, cd_set_region_rows, cd_set_sample_tables for every
 * replicate, cd_assemble; then cd_region_test as usual. */
typedef struct {
    /* per-fragment tables of one replicate, index = fragID - frag_id0, length F (host pointers) */
    const double* s_j;        /* first s_j per baitID (chicdiff.R:659); NaN = NA or bait absent -> Bmean NA (:702) */
    const int32_t* tblb;      /* bait's tblb bin as an index into tmean rows; -1 = NA */
    const double* s_i;        /* first s_i per otherEndID (:668); NaN = NA -> 1 (:672) */
    const int32_t* tlb;       /* other end's tlb bin (tmean column); -1 = NA -> lowest Tmean of the tblb (:689-692) */
    int n_tblb, n_tlb;
    const double* tmean;      /* n_tblb x n_tlb row-major, first Tmean per (tblb, tlb) (:680); NaN = combination absent */
    double distfun[10];       /* .chicEstimateDistFun (:538-573): cubicFit[4], obs.min, obs.max, head.coef[2], tail.coef[2] */
    /* counts (.chinput, :820-860): CSR by bait fragment over (otherEndID, N) rows sorted by otherEndID */
    const int64_t* cnt_off;   /* F + 1 */
    const int32_t* cnt_oe;
    const int32_t* cnt_N;
} cd_sample_tables;

/* restriction map: F fragments with contiguous IDs frag_id0 .. frag_id0 + F - 1 (chr as integer codes) */
int cd_set_rmap(cd_ctx* ctx, int64_t F, int32_t frag_id0, const int32_t* chr, const int32_t* start, const int32_t* end);
/* getRegionUniverse() on the device (chicdiff.R:369-426): every filtered peak (baitID, oeID) -> the window
 * .expandAvoidBait(bait, oe, RUexpand) (:353-367), trimmed to the genome (:402) and to the bait's chromosome
 * (:404-419); regionID = 1-based index of the peak.  Needs cd_set_design and cd_set_rmap; replaces
 * cd_set_regions + cd_set_region_rows.  R_out receives the number of rows. */
int cd_region_universe(cd_ctx* ctx, int64_t m, const int32_t* peak_bait, const int32_t* peak_oe, int ru_expand, int64_t* R_out);
/* host copies of the universe built by cd_region_universe: row_off[m+1], row_bait[R], row_oe[R] (any may be NULL) */
int cd_get_region_universe(cd_ctx* ctx, int64_t* row_off_out, int32_t* row_bait_out, int32_t* row_oe_out);
/* the region universe's rows (RU: baitID, otherEndID), region-contiguous, R = row_off[n] */
int cd_set_region_rows(cd_ctx* ctx, int64_t R, const int32_t* row_bait, const int32_t* row_oe);
/* Asynchronous like cd_set_sample_rows: the tables are copied on the context's copy stream and belong to the NEXT
 * cd_assemble (the matrices of the last one stay valid, so a region test of the current batch can run while the next
 * batch's tables cross the bus); the host arrays must stay valid until that cd_assemble has returned. */
int cd_set_sample_tables(cd_ctx* ctx, int s, const cd_sample_tables* tables);
/* The same tables built ON THE DEVICE from one replicate's raw CHiCAGO columns, replacing the keyed joins / setkey sorts /
 * first-per-group passes of getFullRegionData1 (chicdiff.R:632-634 setkey(x, baitID, otherEndID); :659 first (s_j, tblb)
 * per bait; :668 first (s_i, tlb) per other end; :678-680 first Tmean per (tblb, tlb); :828-853 the per-pair counts).
 * Rows may come in any order: "first" means first in (baitID, otherEndID, input position) order, as after the
 * reference's setkey.  tblb / tlb are the bin labels as integer codes (index into the Tmean table, -1 = NA); the
 * label -> code map and .chicEstimateDistFun's 10 numbers (:538-573, ~75 points) are the caller's.  Counts: the rows of
 * cnt_* when cnt_rows > 0 (the .chinput file, or the inner join of the replicates' N columns for countData = NULL,
 * :778), otherwise the table's own N column.  Replaces cd_set_sample_tables for replicate s. */
typedef struct {
    int64_t rows;
    const int32_t* baitID; const int32_t* otherEndID;
    const double* s_j; const double* s_i;            /* NaN = NA */
    const int32_t* tblb; const int32_t* tlb;         /* bin codes, -1 = NA */
    const double* Tmean;
    const int32_t* N;                                /* may be NULL when cnt_rows > 0 */
    int n_tblb, n_tlb;
    double distfun[10];
    int64_t cnt_rows;
    const int32_t* cnt_baitID; const int32_t* cnt_otherEndID; const int32_t* cnt_N;
} cd_chicago_table;
int cd_build_sample_tables(cd_ctx* ctx, int s, const cd_chicago_table* table);
/* host copies of replicate s's tables as they stand on the device (any pointer may be NULL): s_j, tblb, s_i, tlb of length
 * F; tmean n_tblb x n_tlb; cnt_off F + 1; cnt_oe / cnt_N of cnt_off[F] entries (ask for cnt_off first to size them) */
int cd_get_sample_tables(cd_ctx* ctx, int s, double* s_j, int32_t* tblb, double* s_i, int32_t* tlb, double* tmean,
                         int64_t* cnt_off, int32_t* cnt_oe, int32_t* cnt_N);
/* assembly + aggregation.  keep_rows != 0 also materialises the per-row N / FullMean columns on the device
 * (cd_get_sample_rows).  Outputs are host pointers and may be NULL: K, FullMean (S x n sample-major) and
 * avDist[n] = mean over the region's rows of the signed distance of chicdiff.R:878-881 (what
 * IHWcorrection() needs from FullRegionData, :1965). */
int cd_assemble(cd_ctx* ctx, int keep_rows, int32_t* K_out, double* fullmean_out, double* avDist_out);
int cd_get_sample_rows(cd_ctx* ctx, int s, int32_t* N_out, double* fullmean_out);
/* per-row Bmean of replicate s (chicdiff.R:701-702); only after cd_assemble(keep_rows != 0) */
int cd_get_sample_bmean(cd_ctx* ctx, int s, double* bmean_out);

/* ---- .chinput codec -------------------------------------------------------------------------------- */
/* Parses the text of a .chinput file (what the reference reads with fread, chicdiff.R:828, 1272): an optional
 * '#' comment line, a header line, then rows `baitID otherEndID N otherEndLen distSign` (tab / space separated,
 * distSign may be NA).  text: host pointer to the file's bytes (nbytes < 2^31).  n_rows_out: parsed rows. */
int cd_parse_chinput(cd_ctx* ctx, const char* text, int64_t nbytes, int64_t* n_rows_out);
/* columns of the last cd_parse_chinput in file order (any pointer may be NULL); otherEndLen NA = INT32_MIN,
 * distSign NA = NaN */
int cd_get_chinput(cd_ctx* ctx, int32_t* baitID, int32_t* otherEndID, int32_t* N, int32_t* otherEndLen, double* distSign);

/* ---- countput ------------------------------------------------------------------------------------- */
/* The per-condition (baitID, otherEndID) table getFullRegionData() saves as <outprefix>_countput.Rds
 * (chicdiff.R:708-735, 755-770): Nav = mean(N), Bav = mean(Bmean), score = max(score), oeID_mid = (start+end)/2
 * over the replicates of ONE condition in which the pair occurs; rows in order of first appearance.
 * Each replicate: the CHiCAGO rows that have a distance (chicdiff.R:715), host pointers.  Needs cd_set_rmap. */
typedef struct {
    int64_t rows;
    const int32_t* baitID; const int32_t* otherEndID; const int32_t* N;
    const double* Bmean; const double* score;
} cd_chicago_rows;
int cd_countput(cd_ctx* ctx, int n_reps, const cd_chicago_rows* reps, int64_t* n_pairs_out);
/* fetch the table built by the last cd_countput (n_pairs rows; any pointer may be NULL) */
int cd_get_countput(cd_ctx* ctx, int32_t* baitID, int32_t* otherEndID, double* Nav, double* Bav, double* score, double* oeID_mid);

/* ---- stages 2-5 -------------------------------------------------------------------------- */
typedef struct {
    int norm;                    /* CD_NORM_*; reference default "combined" */
    double theta;                /* NaN = choose on theta_grid by minimum total deviance */
    const double* theta_grid;    /* NULL = {0, .25, .5, .75, 1} */
    int n_theta_grid;
    double disp_prior_var;       /* NaN = estimate (closed form needs S - p > 3) */
    double disp_prior_var_grid;  /* same for the intercept-only theta-grid fits (needs S - 1 > 3) */
    int disp_grid_len;           /* fitDispGrid length; 0 = 20 */
    /* Designs with S - p <= 3 (2-vs-2; the intercept-only theta-grid fits when S <= 4): DESeq2's
     * estimateDispersionsPriorVar matches a seeded Monte-Carlo histogram with R's own RNG and loess.  When the
     * corresponding disp_prior_var* is NaN and prior_var_fn is set, the library hands the dispersion residuals
     * log(dispGeneEst) - log(dispFit) of the regions with dispGeneEst >= 1e-6 (host array, n_resid values, valid
     * during the call) to the caller on the calling thread, once per dispersion fit, and uses the returned value as
     * dispPriorVar; an R front end evaluates DESeq2's own rule there (INTEGRATION.md).  NaN return = failure. */
    double (*prior_var_fn)(void* user, int df, int64_t n_resid, const double* resid);
    void* prior_var_user;
    /* Global scalars of the FINAL fit taken from the caller instead of being estimated (NaN or 0 = estimate, so a
     * zero-initialised struct behaves as before): the parametric trend dispFit = trend_a0 + trend_a1 / baseMean
     * (DESeq2 dispersionFunction coefficients asymptDisp, extraPois) and varLogDispEsts (the squared MAD of the log
     * residuals).  Like disp_prior_var they exist so that a fit can be repeated with known scalars -- a control set
     * fitted with the test set's trend, or a parity check that hands both implementations the same values so that
     * per-region agreement is not blurred by the coupling through the global fits. */
    double trend_a0, trend_a1;
    double var_log_disp;
} cd_options;

typedef struct {
    /* per region, length n, host, any pointer may be NULL */
    double* baseMean; double* baseVar;
    double* dispGeneEst; double* dispFit; double* dispMAP; double* dispersion;
    double* log2FoldChange; double* lfcSE;      /* tested (last) coefficient */
    double* beta; double* betaSE;               /* all coefficients, p x n, log2 scale */
    double* stat; double* pvalue; double* deviance; double* maxCooks;
    double* normFactors;                        /* S x n, the offsets used by the final fit */
    double* mu;                                 /* S x n, fitted means of the gene-wise step */
    int32_t* dispGeneIter; int32_t* dispIter; int32_t* betaIter;
    uint8_t* flags;
    /* scalars, filled by the call */
    double sizeFactors[32];
    double theta;                               /* NaN when norm != combined */
    double deviances[16];                       /* theta-grid total deviances */
    int n_deviances;
    double trend_a0, trend_a1;                  /* asymptDisp, extraPois */
    double varLogDispEsts, dispPriorVar;
    int64_t n_nonzero, n_gene_grid, n_map_grid, n_beta_noconv;
} cd_results;

/* DESeq2Wrap numerics on the aggregated matrices of this context (this rank's shard).  CD_EINVAL when a count is NA
 * (INT32_MIN) or negative, on every rank of a sharded run (DESeqDataSetFromMatrix, chicdiff.R:1556-1559). */
int cd_region_test(cd_ctx* ctx, const cd_options* opt, cd_results* out);

/* ---- several GPUs from ONE process ------------------------------------------------------ */
/* chicdiffPipeline runs in a single R session (chicdiff.R:301-347); a cd_multi lets that one process use n_gpus devices:
 * it owns one context per device, cuts the regions into contiguous bait-aligned shards (cd_plan_shards), drives the
 * contexts with one host thread per device for the duration of each call, and returns per-region results in region
 * order.  The contexts are joined like the ranks of a multi-process run; sharing an address space, their peer-memory
 * mailboxes are mapped with cudaDeviceEnablePeerAccess.  device_ids == NULL: devices 0 .. n_gpus-1.
 * Semantics of every call = the single-context call of the same name on the whole problem (matrices S x n sample-major,
 * vectors of n regions; cd_results scalars from the global steps, counters summed).  region_bait: baitID per region,
 * non-decreasing (cuts fall between baits).  cd_options.prior_var_fn is not available (it needs all residuals on the
 * host): pass disp_prior_var for designs with S - p <= 3. */
typedef struct cd_multi cd_multi;
int cd_multi_create(cd_multi** out, int n_gpus, const int* device_ids);
void cd_multi_destroy(cd_multi* m);
const char* cd_multi_last_error(const cd_multi* m);       /* m may be NULL: last error of cd_multi_create */
int cd_multi_gpus(const cd_multi* m);
int cd_multi_set_design(cd_multi* m, int S, int p, const double* X);
int cd_multi_set_regions(cd_multi* m, int64_t n, const int64_t* row_off /* n + 1 */, const int32_t* region_bait /* n */);
int cd_multi_get_shards(const cd_multi* m, int64_t* bounds /* n_gpus + 1 */);
int cd_multi_set_sample_rows(cd_multi* m, int s, int64_t R, const int32_t* N, const double* fullmean);
int cd_multi_aggregate(cd_multi* m, int32_t* K_out, double* fullmean_out);
int cd_multi_region_test(cd_multi* m, const cd_options* opt, cd_results* out);
int cd_multi_last_timings(const cd_multi* m, double out_ms[8]);      /* per stage, the slowest device */

/* results(): Cook's cutoff (+ two-level-factor heuristic via CD_FLAG_COOKS_KEEP), independent
 * filtering on baseMean (alpha = 0.1), BH.  Global over all regions: in a sharded run gather
 * first.  pvalue is updated in place (outliers -> NaN); padj is written.  scalars_out (may be
 * NULL) receives {cooksCutoff, filterThreshold, filterTheta, filterIndex(1-based)}. */
int cd_results_adjust(int64_t n, int S, int p, const double* baseMean, const double* maxCooks,
                      const uint8_t* flags, double* pvalue, double* padj, double* scalars_out);

/* The same results() step (chicdiff.R:1721,1730,1739) on the arrays the last successful cd_region_test of this
 * context left in device memory: two radix sorts and prefix counts on the GPU, only the 50-point lowess of the
 * filtering rule on the host.  pvalue_out / padj_out (n doubles each, host; either may be NULL) and scalars_out
 * as in cd_results_adjust.  Not for sharded contexts (the step is global): gather and use cd_results_device or
 * cd_results_adjust. */
int cd_results_resident(cd_ctx* ctx, double* pvalue_out, double* padj_out, double* scalars_out);

/* The same device routine on columns given by the caller: n host doubles each of baseMean, maxCooks (NULL = no Cook's
 * filtering) and pvalue, n flag bytes (NULL = none carries CD_FLAG_COOKS_KEEP), and the design's S and p.  The columns are
 * copied to the context's GPU; nothing of the context's last cd_region_test is read or changed.  For the gathered columns
 * of a sharded run, or any columns results() should see.  Outputs as cd_results_resident; pvalue is not modified. */
int cd_results_device(cd_ctx* ctx, int64_t n, int S, int p, const double* baseMean, const double* maxCooks,
                      const uint8_t* flags, const double* pvalue, double* pvalue_out, double* padj_out, double* scalars_out);

/* IHWcorrection(), "apply to test data" block (chicdiff.R:2038-2049), after R's ihw() has been trained on the control
 * set and the distance lookup learned (:1994-2033): minLogDist / maxLogDist / avWeights are the ngroups rows of
 * distLookup as they stand at :2033 (first minimum set to 0, last maximum to Inf).  Per region, in input order:
 * group = cut(log|avDist|, breaks) (1-based, INT32_MIN = NA), weight = avWeights[group] / mean(avWeights over the
 * rows), weighted_pvalue = pvalue / weight, weighted_padj = BH.  The reference's merge() leaves the table sorted by
 * group; callers that need that order sort by (group, input order).  Host routine; any output may be NULL. */
int cd_ihw_apply(int64_t n, const double* avDist, const double* pvalue, int ngroups, const double* minLogDist,
                 const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                 double* weighted_pvalue_out, double* weighted_padj_out);

/* The same block on the device (csrc/ihw.cu): group look-up, weights, weighted p-values and the BH adjustment (one radix
 * sort + a minimum scan) run on the context's GPU; only the mean weight is taken on the host from the per-group counts
 * (R's long-double mean).  avDist: n host doubles, or NULL to use the avDist column cd_assemble left on the device
 * (n must then equal the context's region count).  pvalue: n host doubles.  Outputs as cd_ihw_apply (host, any may be
 * NULL).  Agrees with cd_ihw_apply bit for bit unless log|avDist| falls within an ulp of a break. */
int cd_ihw_apply_device(cd_ctx* ctx, int64_t n, const double* avDist, const double* pvalue, int ngroups, const double* minLogDist,
                        const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                        double* weighted_pvalue_out, double* weighted_padj_out);

/* ---- dispersion prior variance for 1 <= S - p <= 3 (csrc/priorvar.cpp) ---------------------------------------------- */
/* DESeq2's estimateDispersionsPriorVar for designs with at most 3 residual degrees of freedom (every 2-vs-2 run; reached
 * from chicdiff.R:1573, 1603, 1643, 1673): the seeded Monte-Carlo match of the histogram of the dispersion residuals
 * log(dispGeneEst) - log(dispFit) (set.seed(2), rchisq, rnorm, hist, Kullback-Leibler, loess, floor 0.25).  A host
 * restatement of R's generators, hist() and loess() -- see the header of priorvar.cpp for what is pinned and what is not.
 * cd_region_test uses it by itself when S - p <= 3 and neither disp_prior_var* nor prior_var_fn is given; the same
 * function can be handed to cd_options.prior_var_fn.  resid: the residuals of the regions with dispGeneEst >= 1e-6.
 * The rule needs only the 40 bin counts of hist(resid, breaks = -20:20/2): cd_prior_var_hist makes them (they add up over
 * shards), cd_prior_var_from_hist finishes; NaN for df outside 1..3 or an empty histogram. */
double cd_prior_var_small_df(int df, int64_t n_resid, const double* resid);
int cd_prior_var_hist(int64_t n_resid, const double* resid, double counts[40]);
double cd_prior_var_from_hist(int df, const double counts[40]);
/* test hooks: the first n values after set.seed(seed) of unif_rand (what = 0), norm_rand (1), exp_rand (2),
 * rgamma(shape, 1) (3); the 200 Kullback-Leibler divergences of a histogram and their loess fit on the 1000-point grid */
int cd_prior_var_debug_stream(unsigned int seed, int what, double shape, int n, double* out);
int cd_prior_var_debug_curve(int df, const double counts[40], double kl_out[200], double fitted_out[1000]);

/* ---- introspection ------------------------------------------------------------------------ */
/* sizes of the problem currently set on the context: regions n, samples S, design columns p, region rows R (any pointer
 * may be NULL).  Bindings size their output buffers from these, not from what their caller believes. */
int cd_get_dims(const cd_ctx* ctx, int64_t* n, int* S, int* p, int64_t* R);
/* number of kernel launches issued by this context since creation */
int64_t cd_launch_count(const cd_ctx* ctx);
/* device pointers of the aggregated matrices (S x n): for device-resident pipelines */
int cd_device_buffers(cd_ctx* ctx, const int32_t** K_dev, const double** fullmean_dev);
/* device time of the last cd_aggregate / cd_region_test in ms, measured with CUDA events on the context's
 * stream: [0] aggregation kernel, [1] region_test total, [2] fitDisp line-search kernels (all fits),
 * [3] NB GLM / Wald kernels, [4] grid refits, [5] trend fit + MAD, [6] size factors */
int cd_last_timings(const cd_ctx* ctx, double out_ms[8]);
/* The dispersion line searches of the last cd_region_test, one entry per search launch in launch order (theta-grid batch:
 * gene-wise, MAP; final fit: gene-wise, MAP): fused posterior + derivative evaluations summed over the regions (one to
 * start a search plus one per trip), the design columns p of that fit and the (virtual) regions searched.  This is the
 * unit count of the FP64 roofline in bench.py: evaluations x S replicates x flop per replicate-evaluation. */
int cd_last_search_counts(const cd_ctx* ctx, int* n_calls, int64_t evaluations[16], int design_columns[16], int64_t regions[16]);
/* Cross-rank rendezvous of the trend fits of the last cd_region_test on a sharded context: the number of trend passes (each
 * pass ends with every rank storing its sums into every peer's mailbox over NVLink and waiting for everybody's), and
 * the SM cycles CTA 0 spent waiting for the peers' sequence words, summed over passes and peers (wait_cycles_self: the
 * same for its own slot, i.e. the cost of the store + fence alone).  wait / (passes x (ranks - 1)) / SM clock = the mean
 * wait per rendezvous and peer: arrival skew of the ranks plus the NVLink store-to-visibility latency.
 * wait_cycles_first_pass: the part of wait_cycles_peers spent in the first pass of each trend kernel (two launches per
 * cd_region_test with a theta grid), i.e. waiting for the slowest rank to arrive from its line searches. */
int cd_last_rendezvous(const cd_ctx* ctx, double* trend_passes, double* wait_cycles_peers, double* wait_cycles_self,
                       double* wait_cycles_first_pass);
/* CUDA-event stopwatch on the context's stream (what bench.py brackets its timed region with) */
int cd_timer_start(cd_ctx* ctx);
int cd_timer_stop(cd_ctx* ctx, double* ms_out);      /* synchronises */
/* DFMA micro-benchmark: the FP64 roofline denominator measured on this GPU, in TFLOP/s (FMA = 2 flop) */
int cd_measure_fp64_peak(cd_ctx* ctx, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif
