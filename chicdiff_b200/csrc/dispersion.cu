// dispersion.cu -- stage 4: gene-wise Cox-Reid dispersion line search, grid refit, MAP.
//
// Restates, for the GPU, what DESeq2's estimateDispersionsGeneEst / estimateDispersionsMAP
// do when Chicdiff calls estimateDispersions() (chicdiff.R:1573,1602,1643,1673): rough and
// moments starting values, mu from the hat-matrix projection, the Armijo line search on
// log(alpha) over the Cox-Reid adjusted profile likelihood (DESeq2.cpp fitDisp), and the
// two-level grid refit (fitDispGrid) for rows whose search did not converge.
//
// Mapping: one lane per region; per-sample columns are read coalesced from the
// sample-major matrices and the region's replicates (y_j, mu_j) are staged per lane in a
// conflict-free shared-memory column.
//
// Batches.  The theta grid of DESeq2Wrap (chicdiff.R:1633-1647) fits the SAME counts G = 5 times with different
// normalisation factors.  Those fits run as ONE problem of G * n "virtual regions": every per-region array of the
// batch is sample-major over the virtual index v = g * n + i (the counts are replicated G times), so every kernel
// here works on a batch unchanged; the few per-fit scalars (theta, moments offset, trend coefficients, prior
// variance, outlier threshold) are looked up with g = v / n.  One launch per stage instead of G, and the uneven
// tails of the line searches overlap across the fits.
//
// The design of the running fit is read through a pointer into the context's own device copy (no __constant__
// globals: two contexts of one process, on one or several devices, do not share state).
#include "kernels.h"
#include <cuda_pipeline.h>
#include "posterior.cuh"

namespace cd {

static inline int blocks_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---------------------------------------------------------------------------------------
// normalisation factors for a batch: fit g mixes the FullMean scaling factors with the size factors at theta_g
// (chicdiff.R:1583-1589, 1614-1615, 1635-1638, 1666-1669); also replicates the counts into the batch layout
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
norm_factors_kernel(int64_t n, int S, int G, const double* __restrict__ FMagg, const double* __restrict__ sf,
                    int mode, BatchScalars theta, double* __restrict__ nf, const int32_t* __restrict__ K,
                    int32_t* __restrict__ Kb)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t nv = (int64_t)G * n;
    if (Kb) {
        for (int s = 0; s < S; s++) {
            const int32_t k = K[(int64_t)s * n + i];
            for (int g = 0; g < G; g++) Kb[(int64_t)s * nv + (int64_t)g * n + i] = k;
        }
    }
    if (mode == 0) {
        for (int s = 0; s < S; s++)
            for (int g = 0; g < G; g++) nf[(int64_t)s * nv + (int64_t)g * n + i] = sf[s];
        return;
    }
    double acc = 0.0;
    for (int s = 0; s < S; s++) acc += log(FMagg[(int64_t)s * n + i]);
    const double gm = exp(acc / S);
    double m3[CD_MAXS];                          // the scaling factors, taken once (every fit of the batch uses them)
    bool anyna = false;
    for (int s = 0; s < S; s++) {
        m3[s] = FMagg[(int64_t)s * n + i] / gm;
        anyna = anyna || isnan(m3[s]);
    }
    if (anyna)
        for (int s = 0; s < S; s++) m3[s] = sf[s];
    if (mode == 1) {
        for (int s = 0; s < S; s++)
            for (int g = 0; g < G; g++) nf[(int64_t)s * nv + (int64_t)g * n + i] = m3[s];
        return;
    }
    for (int g = 0; g < G; g++) {
        const double th = theta.v[g];
        double acc2 = 0.0;
        for (int s = 0; s < S; s++) acc2 += log(m3[s] * (1.0 - th) + sf[s] * th);
        const double g2 = exp(acc2 / S);
        for (int s = 0; s < S; s++)
            nf[(int64_t)s * nv + (int64_t)g * n + i] = (m3[s] * (1.0 - th) + sf[s] * th) / g2;
    }
}

cudaError_t launch_norm_factors(int64_t n, int S, int G, const double* FMagg, const double* sf, int mode,
                                const BatchScalars& theta, double* nf, const int32_t* K, int32_t* Kb, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    norm_factors_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, G, FMagg, sf, mode, theta, nf, K, Kb);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// base statistics, rough dispersion, and the linear-model means mu = max(hat q * nf, minmu) (the hat products serve
// both; mu may be null: the caller fits it by IRLS then)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
base_stats_kernel(int64_t n, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ K,
                  const double* __restrict__ nf, double* __restrict__ baseMean, double* __restrict__ baseVar,
                  double* __restrict__ rough, uint8_t* __restrict__ flags, double* __restrict__ mu)
{
    __shared__ double hat[CD_MAXS * CD_MAXS];
    for (int k = threadIdx.x; k < S * S; k += blockDim.x) hat[k] = des->hat[k];
    __syncthreads();
    const int p = des->p;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double q[CD_MAXS];
    double sum = 0.0;
    int64_t tot = 0;
    for (int j = 0; j < S; j++) {
        const int32_t k = K[(int64_t)j * n + i];
        q[j] = (double)k / nf[(int64_t)j * n + i];
        sum += q[j];
        tot += k;
    }
    const double m = sum / S;
    double v = 0.0;
    for (int j = 0; j < S; j++) v += (q[j] - m) * (q[j] - m);
    baseMean[i] = m;
    baseVar[i] = v / (S - 1);
    flags[i] = (tot == 0) ? CD_FLAG_ALLZERO : 0;
    // roughDispEstimate: linearModelMu on normalised counts, floored at 1
    double est = 0.0;
    for (int a = 0; a < S; a++) {
        double mul = 0.0;
        for (int b = 0; b < S; b++) mul += hat[a * S + b] * q[b];
        const double mm = fmax(1.0, mul);
        est += ((q[a] - mm) * (q[a] - mm) - mm) / (mm * mm);
        if (mu) mu[(int64_t)a * n + i] = (tot == 0) ? NAN : fmax(mul * nf[(int64_t)a * n + i], kMinMu);
    }
    rough[i] = fmax(est / (S - p), 0.0);
}

cudaError_t launch_base_stats(int64_t n, int S, const CdDesign* des, const int32_t* K, const double* nf, double* baseMean,
                              double* baseVar, double* rough, uint8_t* flags, double* mu, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    base_stats_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, des, K, nf, baseMean, baseVar, rough, flags, mu);
    return cudaGetLastError();
}

// alpha_init = clamp(min(rough, moments)) and its logarithm, where the gene-wise line search starts.  xim_dev[g] per fit.
__global__ void __launch_bounds__(256)
gene_init_kernel(int64_t n, int64_t n_fit, int S, const double* __restrict__ baseMean, const double* __restrict__ baseVar,
                 const double* __restrict__ rough, const uint8_t* __restrict__ flags,
                 const double* __restrict__ xim_dev, double* __restrict__ alpha_init, double* __restrict__ start_log)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flags[i] & CD_FLAG_ALLZERO) {
        alpha_init[i] = NAN;
        start_log[i] = NAN;                      // the line search recognises an all-zero region by this
        return;
    }
    const double xim = xim_dev[i / n_fit];
    const double bm = baseMean[i], bv = baseVar[i];
    const double moments = (bv - xim * bm) / (bm * bm);
    const double maxDisp = fmax(10.0, (double)S);
    const double a0 = fmin(fmax(kMinDisp, fmin(rough[i], moments)), maxDisp);
    alpha_init[i] = a0;
    start_log[i] = log_pos(a0);                  // taken here, off the line search's refill path
}

cudaError_t launch_gene_init(int64_t n, int64_t n_fit, int S, const double* baseMean, const double* baseVar,
                             const double* rough, const uint8_t* flags, const double* xim_dev, double* alpha_init,
                             double* start_log, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    gene_init_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, n_fit, S, baseMean, baseVar, rough, flags, xim_dev, alpha_init,
                                                       start_log);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// fitDisp line search.  One lane works on one region at a time and the kernel is persistent:
// iteration counts are very uneven (most regions stop after 5-15 trips, ~2 % run all 100), so
// a lane that finishes its region immediately takes the next one -- from the block of 32 consecutive
// regions its warp has staged in shared memory (one atomic on the global work counter per block) --
// instead of idling until the slowest lane of its warp is done.  Every trip of a lane has the same shape -- one fused posterior + derivative
// evaluation -- whether the lane is initialising a fresh region or is inside the line search,
// so lanes in different states do not serialise each other.
// The region's replicates (y_j, mu_j) live in a conflict-free shared-memory column per lane.
// ---------------------------------------------------------------------------------------
constexpr int kFitDispThreads = 128;
constexpr int kFitDispTripCap = 24;     // first pass: a region still searching after this many trips is parked

// One staged block of a warp: the inputs of 32 consecutive regions, S int32 count rows, S double mean rows, the start
// values and the prior means (doubles)
__host__ __device__ static inline size_t fit_disp_block_doubles(int S) { return (size_t)16 * S + (size_t)32 * S + 64; }

// dynamic shared memory of the line-search kernels, in doubles: two staging columns per lane, two staged blocks per warp
// and the model matrix (the logarithm table is a static array)
static inline size_t fit_disp_smem_doubles(int S, int P, int threads)
{
    return (size_t)2 * S * threads + (size_t)(threads / 32) * 2 * fit_disp_block_doubles(S) + (size_t)S * P;
}

// the constants of DESeq2's fitDisp (DESeq2.cpp)
constexpr double kSearchEpsilon = 1.0e-4, kSearchKappa0 = 1.0, kSearchTol = 1e-6;
constexpr int kSearchMaxit = 100;

// The scalar state of one region's line search: the current point a = log(alpha), the posterior and its derivative
// there, the posterior at the start, the step factor and the trip counts.
struct SearchState {
    double a, lp, lp0, dlp, kappa;
    int iter, iter_accept;
};

// one trip of fitDisp, first half: the next proposal, its step clamped to log(alpha) in [-30, 10]
__device__ __forceinline__ double propose(SearchState& s)
{
    s.iter++;
    const double a_propose = s.a + s.kappa * s.dlp;
    if (a_propose < -30.0) s.kappa = (-30.0 - s.a) / s.dlp;
    if (a_propose > 10.0) s.kappa = (10.0 - s.a) / s.dlp;
    return s.a + s.kappa * s.dlp;
}

// second half: the Armijo test of the proposal x (posterior lpx, derivative dlpx), then accept and maybe stop, or shrink
// the step; true when the search has finished.  min_log_alpha = log(kMinDisp / 10): the caller takes it once per thread
// (the device log is not folded at compile time)
__device__ __forceinline__ bool decide(SearchState& s, double x, double lpx, double dlpx, double min_log_alpha)
{
    bool finished = false;
    const double theta_kappa = -1.0 * lpx;
    const double theta_hat_kappa = -1.0 * s.lp - s.kappa * kSearchEpsilon * (s.dlp * s.dlp);
    if (theta_kappa <= theta_hat_kappa) {
        s.iter_accept++;
        s.a = x;
        const double change = lpx - s.lp;
        if (change < kSearchTol) { s.lp = lpx; finished = true; }
        else if (s.a < min_log_alpha) { finished = true; }
        else {
            s.lp = lpx;
            s.dlp = dlpx;
            s.kappa = fmin(s.kappa * 1.1, kSearchKappa0);
            if (s.iter_accept % 5 == 0) s.kappa = s.kappa / 2.0;
        }
    } else {
        s.kappa = s.kappa / 2.0;
    }
    if (s.iter >= kSearchMaxit) finished = true;
    return finished;
}

__device__ __forceinline__ void park_store(const FitDispPark& park, unsigned long long slot, const SearchState& s)
{
    park.a[slot] = s.a; park.lp[slot] = s.lp; park.dlp[slot] = s.dlp; park.kappa[slot] = s.kappa; park.lp0[slot] = s.lp0;
    park.iter[slot] = s.iter; park.iter_accept[slot] = s.iter_accept;
}

__device__ __forceinline__ SearchState park_load(const FitDispPark& park, int64_t w)
{
    SearchState s;
    s.a = park.a[w]; s.lp = park.lp[w]; s.dlp = park.dlp[w]; s.kappa = park.kappa[w]; s.lp0 = park.lp0[w];
    s.iter = park.iter[w]; s.iter_accept = park.iter_accept[w];
    return s;
}

// Two passes.  ~2-3 % of the regions run the full 100 trips while the average is below 10; in a
// single persistent pass such a region pulled near the end keeps its warp alive long after the
// work queue is empty.  Pass 1 therefore parks every region that is still searching after
// kFitDispTripCap trips (its scalar search state goes to the FitDispPark arrays); pass 2 resumes
// all parked regions at once, one per lane, so the long searches overlap each other.
constexpr int kFitDispMinBlocks = 4;    // <= 128 registers; measured in round 1: 5 blocks (<= 102) and 6 blocks (80) are not faster
template <int P, bool RESUME>
__global__ void __launch_bounds__(kFitDispThreads, kFitDispMinBlocks)
fit_disp_kernel(int64_t n, int64_t n_fit, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ K,
                const double* __restrict__ mu_g, const double* __restrict__ start_log,
                const double* __restrict__ prior_log_mean, BatchScalars prior_inv_sigmasq_g,
                double* __restrict__ log_alpha_out, int32_t* __restrict__ iter_out,
                double* __restrict__ initial_lp_out, double* __restrict__ last_lp_out,
                unsigned long long* __restrict__ work_counter, FitDispPark park)
{
    extern __shared__ __align__(16) double smem[];
    // logarithm table (16-byte aligned: one LDS.128 per logarithm); dynamic part: the lanes' columns, the warps' staged blocks, model matrix
    __shared__ __align__(16) double tab[2 * kLogTabN];
    const int stride = kFitDispThreads;
    double* ys = smem + threadIdx.x;
    double* mus = smem + (size_t)S * stride + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const bool use_prior = (prior_log_mean != nullptr);
    const double min_log_alpha = log(kMinDisp / 10.0);
    const double inv_n_fit = 1.0 / (double)n_fit;
    int64_t n_work = n;
    if (RESUME) {
        const unsigned long long parked = *park.count;
        n_work = (int64_t)(parked < (unsigned long long)park.capacity ? parked : (unsigned long long)park.capacity);
    }

    bool active = false, exhausted = false, fresh = false;
    int64_t i = 0;
    SearchState s{0.0, 0.0, 0.0, 0.0, kSearchKappa0, 0, 0};
    double prior_mean = 0.0, prior_sigmasq = 1.0;      // prior_sigmasq holds 1 / variance

    // First pass: the inputs are staged per WARP.  A warp claims 32 consecutive regions with one atomic and its 32 lanes
    // copy their rows into a shared-memory block with cp.async (one coalesced request per row, all lanes active); two
    // blocks per warp, the next one on its way while the lanes draw regions from the current one.  A lane that becomes
    // idle takes the next unconsumed region of the current block: one shared-memory copy, no address arithmetic and no
    // global access on the refill path, which runs with 2-3 of 32 lanes on almost every trip (per-lane prefetching cost
    // 13 % of the kernel's instructions there: profiles/r02_d_fit_disp_source_lines.txt).
    const size_t blk_doubles = fit_disp_block_doubles(S);
    double* blk0 = smem + (size_t)2 * S * stride + (size_t)(threadIdx.x >> 5) * 2 * blk_doubles;
    double* Xs = smem + (size_t)2 * S * stride + (size_t)(kFitDispThreads / 32) * 2 * blk_doubles;
    for (int k = threadIdx.x; k < S * P; k += blockDim.x) Xs[k] = des->X[k];
    load_log_table(tab);
    const LogTab tabh = log_tab_handle(tab);
    __syncthreads();

    // block b of this warp: counts [S][32] (int32), means [S][32], start values [32], prior means [32]
    auto blk_k = [&](int b) { return reinterpret_cast<int*>(blk0 + (size_t)b * blk_doubles); };
    auto blk_mu = [&](int b) { return blk0 + (size_t)b * blk_doubles + (size_t)16 * S; };
    auto load_block = [&](int b, int64_t base) {
        const int64_t r = base + lane;
        if (r < n) {
            int* kb = blk_k(b) + lane;
            double* mb = blk_mu(b) + lane;
            const int32_t* kp = K + r;
            const double* mp = mu_g + r;
            for (int j = 0; j < S; j++) {
                __pipeline_memcpy_async(kb + j * 32, kp, sizeof(int32_t));
                __pipeline_memcpy_async(mb + j * 32, mp, sizeof(double));
                kp += n; mp += n;
            }
            __pipeline_memcpy_async(mb + S * 32, start_log + r, sizeof(double));
            if (use_prior) __pipeline_memcpy_async(mb + S * 32 + 32, prior_log_mean + r, sizeof(double));
        }
        __pipeline_commit();
    };
    auto claim32 = [&]() {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(work_counter, 32ull);
        return (int64_t)__shfl_sync(0xffffffffu, base, 0);
    };
    auto valid_in = [&](int64_t base) { return (int)(base >= n ? 0 : (n - base < 32 ? n - base : 32)); };
    int cur = 0, cur_cnt = 0, cur_pos = 0, next_cnt = 0;      // warp-uniform
    int64_t cur_base = 0, next_base = 0;
    if (!RESUME) {
        cur_base = claim32(); cur_cnt = valid_in(cur_base);
        load_block(0, cur_base);
        next_base = claim32(); next_cnt = valid_in(next_base);
        load_block(1, next_base);
        __pipeline_wait_prior(1);              // block 0 has landed (this lane's part; __syncwarp for the others')
        __syncwarp();
    }

    while (true) {
        // ---- refill idle lanes ----
        const bool want = !active && !exhausted;
        const unsigned need = __ballot_sync(0xffffffffu, want);
        if (!RESUME) {
            bool want_now = want;
            unsigned need_now = need;
            while (need_now) {                                  // warp-uniform
                const int avail = cur_cnt - cur_pos;
                if (avail <= 0) {
                    // the current block is used up: the next one becomes current, and its buffer is refilled
                    if (next_cnt <= 0) {                        // the queue is empty
                        if (want_now) exhausted = true;
                        break;
                    }
                    __pipeline_wait_prior(0);
                    __syncwarp();                               // every lane's part of the block has landed; all reads of the old one are done
                    cur ^= 1; cur_base = next_base; cur_cnt = next_cnt; cur_pos = 0;
                    next_base = claim32(); next_cnt = valid_in(next_base);
                    load_block(cur ^ 1, next_base);
                    continue;
                }
                const int my_rank = __popc(need_now & ((1u << lane) - 1u));
                if (want_now && my_rank < avail) {
                    const int idx = cur_pos + my_rank;
                    i = cur_base + idx;
                    const int* kb = blk_k(cur) + idx;
                    const double* mb = blk_mu(cur) + idx;
                    const double a_start = mb[S * 32];
                    if (isnan(a_start)) {
                        // all-zero region: every estimate is NA (its start value was written as NaN upstream); the lane
                        // stays idle and draws again
                        log_alpha_out[i] = NAN; iter_out[i] = 0; initial_lp_out[i] = NAN; last_lp_out[i] = NAN;
                    } else {
                        for (int j = 0; j < S; j++) {
                            ys[j * stride] = (double)kb[j * 32];
                            mus[j * stride] = mb[j * 32];
                        }
                        // the logarithms of the start value and of the prior mean were taken by the kernels that produced
                        // them (gene_init / trend_apply)
                        s.a = a_start;
                        if (use_prior) {
                            prior_mean = mb[S * 32 + 32];
                            // the fit of virtual region i (no division of either kind on this path); eval_post multiplies
                            // by the reciprocal of the prior variance, which the launcher took
                            int g = 0;
                            if (n_fit < n) {                 // i / n_fit for i < 2^32 from a double product, corrected at the edges
                                g = __double2int_rz((double)(unsigned)i * inv_n_fit);
                                if ((int64_t)(g + 1) * n_fit <= i) g++;
                                else if ((int64_t)g * n_fit > i) g--;
                            }
                            prior_sigmasq = prior_inv_sigmasq_g.v[g];
                        }
                        active = true; fresh = true;
                        s.iter = 0; s.iter_accept = 0; s.kappa = kSearchKappa0;
                        want_now = false;
                    }
                }
                const int wanted = __popc(need_now);
                cur_pos += wanted < avail ? wanted : avail;
                need_now = __ballot_sync(0xffffffffu, want_now);
            }
        } else if (need) {
            unsigned long long base = 0;
            const int leader = __ffs(need) - 1;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned long long)__popc(need));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (want) {
                const int64_t w = (int64_t)(base + __popc(need & ((1u << lane) - 1u)));
                if (w >= n_work) {
                    exhausted = true;
                } else {
                    i = park.row[w];
                    s = park_load(park, w);
                    if (use_prior) {
                        prior_mean = prior_log_mean[i];
                        prior_sigmasq = prior_inv_sigmasq_g.v[(unsigned)i / (unsigned)n_fit];      // eval_post multiplies by the reciprocal
                    }
                    for (int j = 0; j < S; j++) {
                        ys[j * stride] = (double)K[(int64_t)j * n + i];
                        mus[j * stride] = mu_g[(int64_t)j * n + i];
                    }
                    active = true; fresh = false;
                }
            }
        }
        if (__all_sync(0xffffffffu, !active)) {
            if (__all_sync(0xffffffffu, exhausted)) break;
            continue;
        }
        // ---- one posterior + derivative evaluation per active lane ----
        double x = s.a;
        if (active && !fresh) x = propose(s);
        // (explicit reconvergence: without it the branches above tail-merge into separate passes
        //  over the evaluation, which was measured at 13 of 32 lanes per issued instruction)
        __syncwarp();
        double lpx = 0.0, dlpx = 0.0;
        // fitDisp evaluates the posterior at the proposal twice (Armijo test, then "lpnew") and, when
        // the proposal is accepted, the derivative at the same point; the arguments are the same
        // double, so one fused evaluation serves all three
        if (active) eval_post<P, true, true>(x, ys, mus, stride, S, Xs, tabh, prior_mean, prior_sigmasq, use_prior, lpx, dlpx);
        __syncwarp();
        // ---- decision ----
        bool finished = false;
        if (active) {
            if (fresh) {
                s.lp = s.lp0 = lpx;
                s.dlp = dlpx;
                fresh = false;
            } else {
                finished = decide(s, x, lpx, dlpx, min_log_alpha);
            }
        }
        if (finished) {
            log_alpha_out[i] = s.a;
            iter_out[i] = s.iter;
            initial_lp_out[i] = s.lp0;
            last_lp_out[i] = s.lp;
            active = false;
        } else if (!RESUME && active && s.iter >= kFitDispTripCap) {
            const unsigned long long slot = atomicAdd(park.count, 1ull);
            if (slot < (unsigned long long)park.capacity) {
                park.row[slot] = i;
                park_store(park, slot, s);
                active = false;
            }                                   // park full: this lane simply keeps searching
        }
    }
}

// ---------------------------------------------------------------------------------------
// Second pass over the parked regions, sample-parallel.  The ~2-3 % of regions that are still searching after
// kFitDispTripCap trips run up to 100 trips each: a latency problem (the chain of trips is sequential), not a
// throughput problem.  Here G lanes share one region, lane l evaluating replicate l's likelihood terms, and
// the per-replicate contributions (log-likelihood, derivative sum, X'WX, X'dWX) are joined by an xor-butterfly
// inside the group, so a trip costs one replicate's worth of special functions instead of S.  Every lane of a
// group carries the same search state and takes the same decisions.
// ---------------------------------------------------------------------------------------
template <int P, int G>
__global__ void __launch_bounds__(128)
fit_disp_resume_tile_kernel(int64_t n, int64_t n_fit, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ K,
                            const double* __restrict__ mu_g, const double* __restrict__ prior_log_mean,
                            BatchScalars prior_sigmasq_g, double* __restrict__ log_alpha_out, int32_t* __restrict__ iter_out,
                            double* __restrict__ initial_lp_out, double* __restrict__ last_lp_out, FitDispPark park)
{
    constexpr int NS = P * (P + 1) / 2;
    const int lane_g = threadIdx.x & (G - 1);                     // replicate handled by this lane
    const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / G;
    const bool use_prior = (prior_log_mean != nullptr);
    const unsigned long long parked = *park.count;
    const int64_t n_work = (int64_t)(parked < (unsigned long long)park.capacity ? parked : (unsigned long long)park.capacity);
    const double min_log_alpha = log(kMinDisp / 10.0);
    const bool has_sample = lane_g < S;
    double xrow[P];
#pragma unroll
    for (int u = 0; u < P; u++) xrow[u] = has_sample ? des->X[lane_g * P + u] : 0.0;

    for (int64_t w0 = 0; w0 < n_work; w0 += n_groups) {
        const int64_t w = w0 + group;
        bool active = w < n_work;
        int64_t i = 0;
        SearchState s{0.0, 0.0, 0.0, 1.0, kSearchKappa0, 0, 0};
        double prior_mean = 0.0, prior_sigmasq = 1.0, y = 0.0, mu = 1.0;
        if (active) {
            i = park.row[w];
            s = park_load(park, w);
            if (use_prior) { prior_mean = prior_log_mean[i]; prior_sigmasq = prior_sigmasq_g.v[(unsigned)i / (unsigned)n_fit]; }
            if (has_sample) { y = (double)K[(int64_t)lane_g * n + i]; mu = mu_g[(int64_t)lane_g * n + i]; }
        }
        while (__any_sync(0xffffffffu, active)) {
            double x = s.a;
            if (active) x = propose(s);
            // ---- this lane's replicate ----
            const double alpha = exp(x);
            const double r = rcp_pos(alpha);
            const double log_r = -x;
            double lgr, dgr;
            lgamma_digamma_pos(r, lgr, dgr);
            double red[2 * NS + 2];
            {
                const double ma = mu * alpha;
                const double ropm = rcp_pos(1.0 + ma);
                const double wj = mu * ropm, dwj = -wj * wj;
                const double l1 = log_pos(1.0 + ma);
                double lg, dg;
                lgamma_digamma_pos(y + r, lg, dg);
                const double on = has_sample ? 1.0 : 0.0;
                int k = 0;
#pragma unroll
                for (int u = 0; u < P; u++)
#pragma unroll
                    for (int v = 0; v <= u; v++) {
                        const double xx = xrow[u] * xrow[v];
                        red[k] = wj * xx; red[NS + k] = dwj * xx; k++;
                    }
                red[2 * NS] = on * (((lg - lgr) - y * (log_r + l1)) - r * l1);
                red[2 * NS + 1] = on * (((dgr - dg) + (l1 - ma * ropm)) + y * (alpha * ropm));
            }
#pragma unroll
            for (int off = G / 2; off > 0; off >>= 1)
#pragma unroll
                for (int k = 0; k < 2 * NS + 2; k++) red[k] += __shfl_xor_sync(0xffffffffu, red[k], off);
            Sym<P> B, dB, Bi;
#pragma unroll
            for (int k = 0; k < NS; k++) { B.v[k] = red[k]; dB.v[k] = red[NS + k]; }
            const double cr = -0.5 * chol_logdet<P>(B);
            chol_inverse<P>(B, Bi);
            double tr = 0.0;
#pragma unroll
            for (int u = 0; u < P; u++)
#pragma unroll
                for (int v = 0; v < P; v++) tr += Bi.v[sidx<P>(u, v)] * dB.v[sidx<P>(v, u)];
            double lpx = red[2 * NS] + cr;
            double dlpx = ((r * r) * red[2 * NS + 1] - 0.5 * tr) * alpha;
            if (use_prior) {
                const double d = x - prior_mean;
                lpx += -0.5 * d * d / prior_sigmasq;
                dlpx += -1.0 * d / prior_sigmasq;
            }
            // ---- decision (identical in all lanes of the group) ----
            if (active && decide(s, x, lpx, dlpx, min_log_alpha)) {
                if (lane_g == 0) { log_alpha_out[i] = s.a; iter_out[i] = s.iter; initial_lp_out[i] = s.lp0; last_lp_out[i] = s.lp; }
                active = false;
            }
        }
    }
}

// the two passes of launch_fit_disp for a design of P columns
template <int P>
static cudaError_t launch_fit_disp_p(int64_t n, int64_t n_fit, int S, const CdDesign* des, const int32_t* K, const double* mu,
                                     const double* start_log, const double* prior_log_mean, const BatchScalars& prior_sigmasq,
                                     double* log_alpha, int32_t* iter, double* initial_lp, double* last_lp,
                                     unsigned long long* work_counter, const FitDispPark& park, cudaStream_t st)
{
    const int threads = kFitDispThreads;
    const int64_t want = (n + threads - 1) / threads;
    const size_t smem = fit_disp_smem_doubles(S, P, threads) * sizeof(double);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // Second pass: with few parked regions (small shards) the chain of up to 76 remaining trips is a latency
    // problem -> sample-parallel tile kernel; with many it is a throughput problem -> one region per lane again.
    const int G = S <= 8 ? 8 : (S <= 16 ? 16 : 32);
    const bool tile = (double)n * 0.04 * G <= (double)sms * 1024.0;
    BatchScalars prior_inv;                           // 1 / prior variance per fit (IEEE division, as the kernel's own would be)
    for (int g = 0; g < kMaxBatch; g++) prior_inv.v[g] = 1.0 / prior_sigmasq.v[g];
    // persistent grids: exactly the number of CTAs that are resident at once
    int per_sm = 1;
    cudaError_t e = cudaFuncSetAttribute(fit_disp_kernel<P, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fit_disp_kernel<P, false>, threads, smem);
    if (e != cudaSuccess) return e;
    const int64_t resident = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    const int blocks = (int)(want < resident ? want : resident);
    fit_disp_kernel<P, false><<<blocks, threads, smem, st>>>(n, n_fit, S, des, K, mu, start_log, prior_log_mean, prior_inv,
                                                             log_alpha, iter, initial_lp, last_lp, work_counter, park);
    if (tile) {
        auto* tile_kernel = G == 8 ? fit_disp_resume_tile_kernel<P, 8>
                                   : (G == 16 ? fit_disp_resume_tile_kernel<P, 16> : fit_disp_resume_tile_kernel<P, 32>);
        tile_kernel<<<sms * 8, 128, 0, st>>>(n, n_fit, S, des, K, mu, prior_log_mean, prior_sigmasq, log_alpha, iter,
                                             initial_lp, last_lp, park);
    } else {
        e = cudaFuncSetAttribute(fit_disp_kernel<P, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const int64_t want2 = (park.capacity + threads - 1) / threads;
        const int blocks2 = (int)(want2 < resident ? want2 : resident);
        fit_disp_kernel<P, true><<<blocks2 > 0 ? blocks2 : 1, threads, smem, st>>>(n, n_fit, S, des, K, mu, start_log,
            prior_log_mean, prior_inv, log_alpha, iter, initial_lp, last_lp, work_counter + 1, park);
    }
    return cudaGetLastError();
}

cudaError_t launch_fit_disp(int64_t n, int64_t n_fit, int S, int p, const CdDesign* des, const int32_t* K, const double* mu,
                            const double* start_log, const double* prior_log_mean, const BatchScalars& prior_sigmasq,
                            double* log_alpha, int32_t* iter, double* initial_lp, double* last_lp,
                            unsigned long long* work_counter, const FitDispPark& park, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    // work_counter[0]: pass-1 queue head, work_counter[1]: pass-2 queue head ; park.count: parked regions
    cudaError_t e = cudaMemsetAsync(work_counter, 0, 2 * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(park.count, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    decltype(&launch_fit_disp_p<1>) launch;
    switch (p) {
        case 1: launch = launch_fit_disp_p<1>; break;
        case 2: launch = launch_fit_disp_p<2>; break;
        case 3: launch = launch_fit_disp_p<3>; break;
        case 4: launch = launch_fit_disp_p<4>; break;
        default: return cudaErrorInvalidValue;
    }
    return launch(n, n_fit, S, des, K, mu, start_log, prior_log_mean, prior_sigmasq, log_alpha, iter, initial_lp, last_lp,
                  work_counter, park, st);
}

// ---------------------------------------------------------------------------------------
// post-processing
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gene_post_kernel(int64_t n, int S, const double* __restrict__ alpha_init, const double* __restrict__ log_alpha,
                 const int32_t* __restrict__ iter, const double* __restrict__ initial_lp,
                 const double* __restrict__ last_lp, uint8_t* __restrict__ flags,
                 double* __restrict__ dispGeneEst, int32_t* __restrict__ refit_list,
                 int32_t* __restrict__ refit_count)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t f = flags[i];
    if (f & CD_FLAG_ALLZERO) { dispGeneEst[i] = NAN; return; }
    const double maxDisp = fmax(10.0, (double)S);
    double disp = fmin(exp(log_alpha[i]), maxDisp);
    const double l0 = initial_lp[i];
    if (last_lp[i] < l0 + fabs(l0) / 1e6) { disp = alpha_init[i]; f |= CD_FLAG_GENE_NOINCREASE; }
    const int it = iter[i];
    const bool conv = (it < kSearchMaxit) && (it != 1);
    if (!conv && disp > kMinDisp * 10.0) {
        f |= CD_FLAG_GENE_GRID;
        const int32_t slot = atomicAdd(refit_count, 1);
        refit_list[slot] = (int32_t)i;
    }
    dispGeneEst[i] = fmin(fmax(disp, kMinDisp), maxDisp);
    flags[i] = f;
}

cudaError_t launch_gene_post(int64_t n, int S, const double* alpha_init, const double* log_alpha, const int32_t* iter,
                             const double* initial_lp, const double* last_lp, uint8_t* flags, double* dispGeneEst,
                             int32_t* refit_list, int32_t* refit_count, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(refit_count, 0, sizeof(int32_t), st);
    if (e != cudaSuccess || n == 0) return e;
    gene_post_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, alpha_init, log_alpha, iter, initial_lp, last_lp,
                                                       flags, dispGeneEst, refit_list, refit_count);
    return cudaGetLastError();
}

// outlier_thr[g] = 2 sqrt(varLogDispEsts) of fit g
__global__ void __launch_bounds__(256)
map_post_kernel(int64_t n, int64_t n_fit, int S, const double* __restrict__ log_alpha, const int32_t* __restrict__ iter,
                const double* __restrict__ dispGeneEst, const double* __restrict__ dispFit, BatchScalars outlier_thr,
                uint8_t* __restrict__ flags, double* __restrict__ dispMAP, double* __restrict__ dispersion,
                int32_t* __restrict__ refit_list, int32_t* __restrict__ refit_count)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t f = flags[i];
    if (f & CD_FLAG_ALLZERO) { dispMAP[i] = NAN; dispersion[i] = NAN; return; }
    const double maxDisp = fmax(10.0, (double)S);
    if (!(iter[i] < kSearchMaxit)) {
        f |= CD_FLAG_MAP_GRID;
        const int32_t slot = atomicAdd(refit_count, 1);
        refit_list[slot] = (int32_t)i;
    }
    const double dmap = fmin(fmax(exp(log_alpha[i]), kMinDisp), maxDisp);
    const double ge = dispGeneEst[i], ft = dispFit[i];
    const bool outl = log(ge) > log(ft) + outlier_thr.v[(int)(i / n_fit)];
    if (outl) f |= CD_FLAG_OUTLIER;
    dispMAP[i] = dmap;
    dispersion[i] = outl ? ge : dmap;
    flags[i] = f;
}

cudaError_t launch_map_post(int64_t n, int64_t n_fit, int S, const double* log_alpha, const int32_t* iter,
                            const double* dispGeneEst, const double* dispFit, const BatchScalars& outlier_thr, uint8_t* flags,
                            double* dispMAP, double* dispersion, int32_t* refit_list, int32_t* refit_count, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(refit_count, 0, sizeof(int32_t), st);
    if (e != cudaSuccess || n == 0) return e;
    map_post_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, n_fit, S, log_alpha, iter, dispGeneEst, dispFit, outlier_thr,
                                                      flags, dispMAP, dispersion, refit_list, refit_count);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// fitDispGrid: one warp per listed row, lane = grid point (grid_len <= 32)
// ---------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(128)
fit_disp_grid_kernel(int64_t n, int64_t n_fit, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ n_list_dev,
                     const int32_t* __restrict__ list, const int32_t* __restrict__ K, const double* __restrict__ mu_g,
                     const double* __restrict__ prior_mean_disp, BatchScalars prior_sigmasq_g, int grid_len,
                     double* __restrict__ disp_out, double* __restrict__ dispersion_out,
                     const uint8_t* __restrict__ flags, const double* __restrict__ dispGeneEst)
{
    __shared__ double sh[4][2 * CD_MAXS];
    __shared__ double Xs[CD_MAXS * CD_MAXP];
    for (int k = threadIdx.x; k < S * P; k += blockDim.x) Xs[k] = des->X[k];
    __syncthreads();
    const LogTab tab = 0;                        // the grid evaluations use log_pos (no table)
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const int n_list = *n_list_dev;
    double* ys = sh[wib];
    double* mus = sh[wib] + CD_MAXS;
    for (int w = blockIdx.x * warps_per_block + wib; w < n_list; w += gridDim.x * warps_per_block) {
        const int64_t i = list[w];
        __syncwarp();
        if (lane < S) {
            ys[lane] = (double)K[(int64_t)lane * n + i];
            mus[lane] = mu_g[(int64_t)lane * n + i];
        }
        __syncwarp();
        const bool use_prior = (prior_mean_disp != nullptr);
        const double prior_mean = use_prior ? log(prior_mean_disp[i]) : 0.0;
        const double prior_sigmasq = 1.0 / prior_sigmasq_g.v[(int)(i / n_fit)];      // eval_post multiplies by the reciprocal
        const double maxDisp = fmax(10.0, (double)S);
        const double lo = log(1e-8), hi = log(maxDisp);
        const double step = (hi - lo) / (grid_len - 1);
        double best_a = lo;
        double from = lo, to = hi, by = step;
        for (int level = 0; level < 2; level++) {
            const double a = (lane == grid_len - 1) ? to : from + lane * by;
            double v = -INFINITY, unused;
            if (lane < grid_len) eval_post<P, false, false>(a, ys, mus, 1, S, Xs, tab, prior_mean, prior_sigmasq, use_prior, v, unused);
            int idx = lane;
            // arg max, first maximum wins
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, v, off);
                const int oi = __shfl_xor_sync(0xffffffffu, idx, off);
                if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
            }
            best_a = (idx == grid_len - 1) ? to : from + idx * by;
            if (level == 0) {
                const double delta = (lo + step) - lo;
                from = best_a - delta;
                to = best_a + delta;
                by = (to - from) / (grid_len - 1);
            }
        }
        if (lane == 0) {
            const double d = fmin(fmax(exp(best_a), kMinDisp), maxDisp);
            disp_out[i] = d;
            if (dispersion_out) dispersion_out[i] = (flags[i] & CD_FLAG_OUTLIER) ? dispGeneEst[i] : d;
        }
    }
}

cudaError_t launch_fit_disp_grid(int64_t n, int64_t n_fit, int S, int p, const CdDesign* des, const int32_t* n_list_dev,
                                 const int32_t* list, const int32_t* K, const double* mu, const double* prior_mean_disp,
                                 const BatchScalars& prior_sigmasq, int grid_len, double* disp_out, double* dispersion_out,
                                 const uint8_t* flags, const double* dispGeneEst, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    if (grid_len < 2 || grid_len > 32) return cudaErrorInvalidValue;
    const int threads = 128, blocks = 148 * 4;
#define CD_LAUNCH(P_)                                                                                          \
    fit_disp_grid_kernel<P_><<<blocks, threads, 0, st>>>(n, n_fit, S, des, n_list_dev, list, K, mu, prior_mean_disp, \
                                                         prior_sigmasq, grid_len, disp_out, dispersion_out,    \
                                                         flags, dispGeneEst)
    switch (p) {
        case 1: CD_LAUNCH(1); break;
        case 2: CD_LAUNCH(2); break;
        case 3: CD_LAUNCH(3); break;
        case 4: CD_LAUNCH(4); break;
        default: return cudaErrorInvalidValue;
    }
#undef CD_LAUNCH
    return cudaGetLastError();
}

}  // namespace cd
