// kernels.h -- host-callable launchers of the hand-written sm_100a kernels.
// Every launcher enqueues on `st` and returns the cudaGetLastError() of its launches.
// All pointers are device pointers; matrices are sample-major (see common.cuh).
#pragma once
#include "common.cuh"

namespace cd {

// Batches: G fits of the same counts (the theta grid) run as one problem of G * n virtual regions, sample-major over
// v = g * n + i (dispersion.cu).  Per-fit scalars travel by value.
constexpr int kMaxBatch = 16;
struct BatchScalars { double v[kMaxBatch]; };

// ---- stage 1: aggregation (chicdiff.R:1540-1547) --------------------------------------
cudaError_t launch_aggregate(int64_t n, int S, const int64_t* row_off, int64_t R,
                             const int32_t* N_rows, const double* FM_rows,
                             int32_t* K, double* FM, cudaStream_t st);

// ---- region universe (getRegionUniverse, chicdiff.R:353-426) ----
cudaError_t ru_launch_count(int64_t m, const int32_t* peak_bait, const int32_t* peak_oe, int s, int64_t F, int32_t id0,
                            const int32_t* chr, int64_t* counts /*m + 1*/, int32_t* status, cudaStream_t st);
cudaError_t ru_launch_scan(int64_t m, const int64_t* counts, int64_t* row_off, void* tmp, size_t& tmp_bytes, cudaStream_t st);
cudaError_t ru_launch_fill(int64_t m, const int32_t* peak_bait, const int32_t* peak_oe, int s, int64_t F, int32_t id0,
                           const int32_t* chr, const int64_t* row_off, int32_t* row_bait, int32_t* row_oe, cudaStream_t st);

// ---- .chinput text codec (fread of chicdiff.R:828) ----
cudaError_t ch_launch_line_flags(int64_t nbytes, const char* text, uint8_t* flag, cudaStream_t st);
cudaError_t ch_line_starts(void* tmp, size_t& bytes, const uint8_t* flag, int64_t* starts, int64_t* n_out, int64_t nbytes,
                           cudaStream_t st);
cudaError_t ch_launch_parse(int64_t nlines, int64_t nbytes, const char* text, const int64_t* line_start, int32_t* bait,
                            int32_t* oe, int32_t* N, int32_t* oelen, double* dist, uint8_t* valid, cudaStream_t st);
cudaError_t ch_compact_i32(void* tmp, size_t& bytes, const int32_t* in, const uint8_t* flags, int32_t* out, int64_t* n_out,
                           int64_t n, cudaStream_t st);
cudaError_t ch_compact_f64(void* tmp, size_t& bytes, const double* in, const uint8_t* flags, double* out, int64_t* n_out,
                           int64_t n, cudaStream_t st);

// ---- countput (chicdiff.R:708-735, 755-770) ----
cudaError_t cp_launch_keys(int64_t rows, int64_t base, const int32_t* bait, const int32_t* oe, unsigned long long* keys,
                           unsigned int* idx, cudaStream_t st);
cudaError_t cp_sort_pairs_u64(void* tmp, size_t& bytes, const unsigned long long* kin, unsigned long long* kout,
                              const unsigned int* vin, unsigned int* vout, int64_t n, cudaStream_t st);
cudaError_t cp_sort_pairs_u32(void* tmp, size_t& bytes, const unsigned int* kin, unsigned int* kout,
                              const unsigned int* vin, unsigned int* vout, int64_t n, cudaStream_t st);
cudaError_t cp_scan_i64(void* tmp, size_t& bytes, const int64_t* in, int64_t* out, int64_t n, cudaStream_t st);
cudaError_t cp_launch_heads(int64_t T, const unsigned long long* keys, int64_t* head, cudaStream_t st);
cudaError_t cp_launch_reduce(int64_t T, const unsigned long long* keys, const unsigned int* idx, const int64_t* head,
                             const int64_t* slot, const int32_t* N, const double* Bmean, const double* score,
                             unsigned long long* g_key, double* g_nav, double* g_bav, double* g_score,
                             unsigned int* g_first, cudaStream_t st);
cudaError_t cp_launch_iota(int64_t G, unsigned int* v, cudaStream_t st);
cudaError_t cp_launch_gather(int64_t G, const unsigned int* order, const unsigned long long* g_key, const double* g_nav,
                             const double* g_bav, const double* g_score, int64_t F, int32_t id0, const int32_t* frag_start,
                             const int32_t* frag_end, int32_t* o_bait, int32_t* o_oe, double* o_nav, double* o_bav,
                             double* o_score, double* o_mid, cudaStream_t st);

// ---- per-replicate assembly fused with stage 1 (chicdiff.R:609-702, 820-910, 1540-1547) ----
struct AssembleTables {          // device pointers of one replicate, tables indexed by fragID - frag_id0
    const double* s_j; const int32_t* tblb; const double* s_i; const int32_t* tlb;
    const double* tmean; const double* tmin; const double* distfun;
    const int64_t* cnt_off; const int32_t* cnt_oe; const int32_t* cnt_N;
    int n_tblb, n_tlb;
};
cudaError_t launch_tmin(int n_tblb, int n_tlb, const double* tmean, double* tmin, cudaStream_t st);
cudaError_t launch_assemble(int64_t n, int S, const int64_t* row_off, int64_t R, const int32_t* row_bait,
                            const int32_t* row_oe, int64_t F, int32_t frag_id0, const int32_t* frag_chr,
                            const int32_t* frag_start, const int32_t* frag_end, const AssembleTables* tabs_dev,
                            int32_t* K, double* FM, double* avDist, int32_t* N_rows /*S x R or null*/,
                            double* FM_rows /*S x R or null*/, double* BM_rows /*S x R or null*/, int32_t* status,
                            cudaStream_t st);

// ---- per-replicate tables from the raw CHiCAGO columns (tables.cu; chicdiff.R:632-634, 659-692, 828-853) ----
// best: 2 F + 2 n_tblb n_tlb words of scratch (first-by-key winners); status bit 0: a fragment outside the rmap, bit 1: a bin
// code outside the table
cudaError_t tb_launch_first(int64_t m, const int32_t* bait, const int32_t* oe, const int32_t* tblb, const int32_t* tlb, int64_t F,
                            int32_t id0, int n_tblb, int n_tlb, unsigned long long* best, int32_t* status, cudaStream_t st);
cudaError_t tb_launch_fill(int64_t F, int n_tblb, int n_tlb, const unsigned long long* best, const double* s_j_rows,
                           const int32_t* tblb_rows, const double* s_i_rows, const int32_t* tlb_rows, const double* tmean_rows,
                           double* s_j, int32_t* tblb, double* s_i, int32_t* tlb, double* tmean, cudaStream_t st);
cudaError_t tb_launch_count_keys(int64_t m, const int32_t* bait, const int32_t* oe, int64_t F, int32_t id0, unsigned long long* keys,
                                 unsigned int* idx, cudaStream_t st);
cudaError_t tb_launch_count_offsets(int64_t F, int64_t m, const unsigned long long* sorted_keys, int64_t* cnt_off, cudaStream_t st);
cudaError_t tb_launch_count_gather(int64_t m_valid, const unsigned long long* sorted_keys, const unsigned int* sorted_idx,
                                   const int32_t* N_rows, int32_t* cnt_oe, int32_t* cnt_N, cudaStream_t st);

// ---- size factors + stage 2: offsets (chicdiff.R:1561-1562, 1583-1589, 1635-1638) ------
// bad (one double, zeroed by the caller) is set to 1.0 when any count is negative (NA_integer_ included)
cudaError_t launch_log_ratios(int64_t n, int S, const int32_t* K, double* LR /*S x n, +inf = excluded*/, double* bad,
                              cudaStream_t st);
// nf (S x G*n) for the G fits of a batch (mode 2: fit g at theta.v[g]); Kb != null also replicates K (S x n) into the
// batch layout (S x G*n)
cudaError_t launch_norm_factors(int64_t n, int S, int G, const double* FMagg, const double* sf /*S, device*/,
                                int mode, const BatchScalars& theta, double* nf, const int32_t* K, int32_t* Kb, cudaStream_t st);

// ---- deterministic reductions -----------------------------------------------------------
// per fit g: column sums of the sample-major S x G*n matrix over the rows of fit g where mask[row]==0 (mask may be
// null): out[g * (S + 1) + s], and the number of such rows in out[g * (S + 1) + S]
cudaError_t launch_masked_colsums(int64_t n, int G, int S, const double* M, const uint8_t* mask,
                                  double* partial /*>= kReduceBlocks*G*(S+1)*/, double* out, cudaStream_t st);
// out[g] = sum over the rows of fit g (NaN propagates)
cudaError_t launch_segment_sums(int64_t n, int G, const double* v, double* partial, double* out, cudaStream_t st);
// xim[g] from the masked column sums of the normalisation factors (momentsDispEstimate)
cudaError_t launch_xim(int G, int S, const double* sums, double* xim, cudaStream_t st);
constexpr int kReduceBlocks = 592;      // 148 SMs x 4

// ---- exact medians by radix selection (select.cu); B columns at base + c*stride, length n each ----
// One cooperative kernel per batch of B <= 32 medians.  state: B x 8 words, hist: B x 2048 words, aux: 3 B words,
// bar: one word (all device scratch).  out[c] = scale * median of the finite entries of column c (of |x - center[c]|
// when center != null), exp'ed when do_exp.  In a sharded run (pp.nranks > 1) the kernel all-reduces its counters
// through peer memory itself: 8 exchanges, sequence numbers pp.seq .. pp.seq + 7.
constexpr int kSelBinsHost = 2048;
constexpr int kSelStateHost = 8;
constexpr int kSelP2PMaxCols = 32;
constexpr int kSelExchanges = 8;
struct SelP2P {
    int nranks, rank;                       // nranks == 1: no exchange
    unsigned long long* const* peers;       // device array of nranks mailbox pointers (own one included)
    unsigned long long* mymail;             // 2 x nranks x kSelP2PMaxCols slots of 2048 words, then as many flag words
    unsigned long long seq;                 // first sequence number of this launch (nonzero), identical on all ranks
    unsigned long long* err;                // device word, never null: raised when a peer never answered; ends every spin loop
};
inline size_t sel_p2p_mail_words(int nranks) { return (size_t)2 * nranks * kSelP2PMaxCols * (kSelBinsHost + 1); }
cudaError_t sel_launch_fused(int64_t n, int B, const double* base, int64_t stride, const double* center, double* out,
                             int do_exp, double scale, unsigned long long* state, unsigned long long* hist,
                             unsigned long long* aux, unsigned int* bar, const SelP2P& pp, cudaStream_t st);

// ---- IHW weight application on the device (ihw.cu; chicdiff.R:2038-2049) ----
cudaError_t ihw_apply_device(int64_t n, const double* avDist_dev, const double* pvalue_dev, int ngroups, const double* minLogDist,
                             const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                             double* weighted_pvalue_out, double* weighted_padj_out, bool* bad_breaks, cudaStream_t st);

// ---- results() on resident arrays (results_resident.cu) ----
// counts: [0] rows with a p-value after the Cook's filter, [1] rows with baseMean == 0
cudaError_t res_launch_keys(int64_t n, int p, double cutoff, const double* baseMean, const double* maxCooks, const uint8_t* flags,
                            const double* pvalue, double* pv_out, double* padj, unsigned long long* pkey,
                            unsigned long long* bmkey, unsigned int* idx, unsigned long long* counts, cudaStream_t st);
cudaError_t res_launch_cutoffs(int64_t n, const unsigned long long* bm_sorted_keys, const unsigned long long* counts, double* cut,
                               double* theta, cudaStream_t st);
cudaError_t res_launch_gather(int64_t n, const unsigned int* sorted_idx, const double* baseMean, const double* pv, double* bm_s,
                              double* p_s, cudaStream_t st);
int res_chunks(int64_t n);                       // chunks of sorted rows; cnt needs 50 x chunks words, cmin / smin chunks doubles
cudaError_t res_launch_num_rej(int64_t n, const unsigned long long* counts, const double* bm_s, const double* p_s,
                               const double* cut, unsigned int* cnt, unsigned long long* m_tot, double alpha,
                               unsigned long long* best, cudaStream_t st);
cudaError_t res_launch_bh(int64_t n, const unsigned long long* counts, const double* bm_s, const double* p_s,
                          const unsigned int* sorted_idx, const double* cut, int j, const unsigned int* off,
                          const unsigned long long* m_tot, double* cmin, double* smin, double* padj, cudaStream_t st);

// ---- stage 4a: gene-wise dispersion (n = virtual regions of the batch, n_fit = regions per fit) --------------
cudaError_t launch_base_stats(int64_t n, int S, const CdDesign* des, const int32_t* K, const double* nf,
                              double* baseMean, double* baseVar, double* rough, uint8_t* flags,
                              double* mu /*linear-model means, or null*/, cudaStream_t st);
cudaError_t launch_gene_init(int64_t n, int64_t n_fit, int S, const double* baseMean, const double* baseVar,
                             const double* rough, const uint8_t* flags, const double* xim_dev /*per fit*/,
                             double* alpha_init, double* start_log /*log(alpha_init), NaN = all-zero region*/,
                             cudaStream_t st);
// scalar search state of regions parked by the first line-search pass (see dispersion.cu)
struct FitDispPark {
    int64_t capacity;
    int64_t* row;
    double *a, *lp, *dlp, *kappa, *lp0;
    int32_t *iter, *iter_accept;
    unsigned long long* count;
};
// line search from start_log (log alpha; NaN = all-zero region); prior_log_mean == null => no prior (gene-wise), else the
// prior is N(prior_log_mean, prior_sigmasq.v[g]) on log alpha
cudaError_t launch_fit_disp(int64_t n, int64_t n_fit, int S, int p, const CdDesign* des, const int32_t* K, const double* mu,
                            const double* start_log, const double* prior_log_mean, const BatchScalars& prior_sigmasq,
                            double* log_alpha, int32_t* iter, double* initial_lp, double* last_lp,
                            unsigned long long* work_counter /*device scratch, 2 words*/, const FitDispPark& park,
                            cudaStream_t st);
// post-processing of the gene-wise fit + compaction of rows needing the grid
cudaError_t launch_gene_post(int64_t n, int S, const double* alpha_init, const double* log_alpha,
                             const int32_t* iter, const double* initial_lp, const double* last_lp,
                             uint8_t* flags, double* dispGeneEst, int32_t* refit_list, int32_t* refit_count,
                             cudaStream_t st);
cudaError_t launch_map_post(int64_t n, int64_t n_fit, int S, const double* log_alpha, const int32_t* iter,
                            const double* dispGeneEst, const double* dispFit, const BatchScalars& outlier_thr,
                            uint8_t* flags, double* dispMAP, double* dispersion,
                            int32_t* refit_list, int32_t* refit_count, cudaStream_t st);
// grid refit of listed rows, one warp per row; writes disp_out[row] (clamped) and, for MAP,
// re-applies the outlier rule through dispersion_out
cudaError_t launch_fit_disp_grid(int64_t n, int64_t n_fit, int S, int p, const CdDesign* des, const int32_t* n_list_dev,
                                 const int32_t* list, const int32_t* K, const double* mu, const double* prior_mean_disp,
                                 const BatchScalars& prior_sigmasq, int grid_len, double* disp_out,
                                 double* dispersion_out /*null for gene-wise*/, const uint8_t* flags,
                                 const double* dispGeneEst, cudaStream_t st);

// ---- stage 4b: trend ---------------------------------------------------------------------
// the sums of one pass of the Gamma(identity) IRLS at coefficients b, over rows with !allZero, dispGeneEst > 1e-6 and
// residual ratio (w.r.t. the outer coefficients c) in (1e-4, 15): s00, s01, s11, t0, t1, deviance, #invalid mu, #rows
// peer-memory description for the in-kernel all-reduce of the sharded trend fit (nranks == 1: unused)
struct TrendP2P {
    int nranks, rank;
    double* const* peers;       // device array of nranks pointers: every rank's mailbox (own one included)
    double* mymail;             // this rank's mailbox: 2 x nranks slots of (8 kMaxBatch + 8) doubles
    unsigned long long epoch;   // distinct per launch, identical on all ranks
    unsigned long long* err;    // device word, never null (see SelP2P)
    unsigned long long* wait_cycles;   // may be null: [0] += SM cycles CTA 0 waited for peers' sums, [1] += for its own slot, [2] += the first-pass part of [0]
};
inline size_t trend_p2p_mail_doubles(int nranks) { return (size_t)2 * nranks * (8 * kMaxBatch + 8); }
// the whole parametricDispersionFit of the G fits of a batch in one cooperative kernel; out[g * 8 + 0..1] coefs,
// [2] status, [3] outer iterations, [4] passes; xs = one double of scratch per virtual region,
// partial >= 16 * G * #SMs doubles, bar = one word
cudaError_t launch_trend_fit(int64_t n, int G, const double* baseMean, const double* dispGeneEst, const uint8_t* flags,
                             double* xs, double* partial, unsigned int* bar, double* out, const TrendP2P& pp, cudaStream_t st);
// dispFit = a0 + a1/baseMean ; resid = log(dispGeneEst) - log(dispFit) or +inf when excluded ; coefs_dev[g * 8 + 0..1]
// also the MAP search's start value and prior mean as logarithms
cudaError_t launch_trend_apply(int64_t n, int64_t n_fit, const double* baseMean, const double* dispGeneEst,
                               const uint8_t* flags, const double* coefs_dev, double* dispFit, double* resid,
                               double* map_start_log, double* log_fit, cudaStream_t st);

// ---- stages 3 + 5: NB GLM, Cook's, Wald --------------------------------------------------
constexpr int kLfactN = 4096;
cudaError_t launch_lfact_table(double* tab /* kLfactN doubles */, cudaStream_t st);
struct WaldScratch {
    const double* lfact; // kLfactN: log Gamma(k + 1) - 0.5 log(2 pi), see launch_lfact_table
    double* cmat;        // S x n: mu-independent part of the NB log density
    double* beta0;       // p x n: least-squares start
    double* beta_nat;    // p x n: IRLS coefficients, natural-log scale
    int32_t* iter;       // n
    unsigned long long* work_counter;
};
// prep + persistent IRLS (p >= 2) + finalisation.  Also used for the IRLS-mu variant of the gene-wise
// step (mu_out != null => only mu is written).  maxCooks == null skips Cook's distances.
cudaError_t launch_wald(int64_t n, int S, int p, const CdDesign* des, const int32_t* K, const double* nf,
                        const double* dispersion, uint8_t* flags, const WaldScratch& ws,
                        double* beta /*p x n, log2*/, double* betaSE, double* stat, double* pvalue,
                        double* deviance, double* maxCooks, int32_t* betaIter, double* mu_out,
                        cudaStream_t st);

// total deviance input of the theta-grid fits (design ~ 1): -2 logLik per virtual region at the intercept-only
// shortcut's coefficients; nothing else of nbinomWaldTest is needed there (chicdiff.R:1644-1647)
cudaError_t launch_wald_deviance_p1(int64_t n, int S, const int32_t* K, const double* nf, const double* dispersion,
                                    const uint8_t* flags, const double* lfact, double* deviance, cudaStream_t st);

}  // namespace cd
