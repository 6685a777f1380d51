// wald.cu -- stages 3 and 5: batched FP64 negative-binomial GLM (IRLS), hat diagonals,
// Cook's distances, Wald statistic and p-value.
//
// Restates what nbinomWaldTest() does when Chicdiff calls it (chicdiff.R:1574,1603,1644,1674):
// fitNbinomGLMs -> DESeq2.cpp fitBeta (ridge lambda = 1e-6 / ln(2)^2, mu floored at 0.5,
// convergence on the relative deviance change, |beta| > 30 => failure), the intercept-only
// shortcut for design ~ 1 (the theta grid), calculateCooksDistance / recordMaxCooks, and
// p = 2 * pnorm(-|beta / SE|).
//
// Three kernels, one region per lane:
//   wald_prep_kernel   the part of the NB log density that does not depend on mu
//                      (lgamma(y + 1/alpha) - lgamma(1/alpha) - lgamma(y + 1)) and the least-squares
//                      start of the IRLS; uniform work, plain grid
//   wald_irls_kernel   the IRLS itself, persistent with work pulling like the dispersion line
//                      search (iteration counts range from 2 to 100): one trip = solve the ridge
//                      normal equations by an unrolled Cholesky (p <= 4; DESeq2 solves the same system
//                      by QR of the row-augmented matrix), then one sweep over the replicates for
//                      X'WX, X'Wz and the deviance at the new coefficients
//   wald_final_kernel  covariance sandwich, hat diagonals, log likelihood at the unfloored mu,
//                      Cook's distances, Wald statistic, p-value; uniform work, plain grid
//
// NB log density: log f(y; size, mu) = c(y, size) - size log(1 + mu/size) + y log(mu / (size + mu)),
// one instruction sequence for every count including zero.  R's dnbinom_mu() evaluates the same
// quantity through Loader's saddle-point expansion; the two agree to ~1e-14 relative except when
// size = 1/alpha is huge, where the lgamma difference cancels: rows with 1/alpha > 1e6 take the
// saddle-point path (dnbinom_mu_log in common.cuh).
#include "kernels.h"
#include "posterior.cuh"

namespace cd {

// The design of the running fit is read through a pointer into the context's own device copy and staged in shared
// memory (every lane reads the same entry); no __constant__ globals, so contexts of one process do not share state.

constexpr int kWaldThreads = 128;

// log Gamma(k + 1) - 0.5 log(2 pi) for the counts k < kLfactN, filled once per context with lgamma_c_pos itself, so a
// look-up returns the very double the direct evaluation would: a third of the special-function work of the NB log
// density does not depend on the fit at all
__global__ void lfact_table_kernel(double* __restrict__ tab)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < kLfactN) tab[k] = lgamma_c_pos((double)k + 1.0);
}

cudaError_t launch_lfact_table(double* tab, cudaStream_t st)
{
    lfact_table_kernel<<<(kLfactN + 255) / 256, 256, 0, st>>>(tab);
    return cudaGetLastError();
}

__device__ __forceinline__ double lfact_c(double y, const double* __restrict__ lfact)
{
    return (y < (double)kLfactN) ? __ldg(lfact + (int)y) : lgamma_c_pos(y + 1.0);
}
constexpr double kHalfLn2Pi = 0.918938533204672741780329736406;
constexpr double kHugeSize = 1e6;

static inline int blocks_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// mu-dependent part of the log density; the two logarithms by the table scheme of the line search (common.cuh,
// log_pos_v2: the kernels below copy the table to shared memory like fit_disp_kernel does)
__device__ __forceinline__ double nb_logdens(double y, double size, double alpha, double mu, double c, LogTab tab)
{
    if (size > kHugeSize) return dnbinom_mu_log(y, size, mu);
    const double l1 = log_pos_v2(1.0 + mu * alpha, tab);
    const double l2 = log_pos_v2(mu * rcp_fast(size + mu), tab);
    return (c - size * l1) + y * l2;
}


// ---------------------------------------------------------------------------------------
// prep
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
wald_prep_kernel(int64_t n, int S, int P, const CdDesign* __restrict__ des, const int32_t* __restrict__ K,
                 const double* __restrict__ nf, const double* __restrict__ dispersion, const uint8_t* __restrict__ flags,
                 const double* __restrict__ lfact, double* __restrict__ cmat, double* __restrict__ beta0)
{
    __shared__ double ls[CD_MAXP * CD_MAXS];
    for (int k = threadIdx.x; k < P * S; k += blockDim.x) ls[k] = des->ls[k];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flags[i] & CD_FLAG_ALLZERO) return;
    const double alpha = dispersion[i];
    const double size = rcp_pos(alpha);
    const double lgs = lgamma_c_pos(size);
    double b[CD_MAXP];
    for (int u = 0; u < P; u++) b[u] = 0.0;
    for (int j = 0; j < S; j++) {
        const double y = (double)K[(int64_t)j * n + i];
        cmat[(int64_t)j * n + i] = ((lgamma_c_pos(y + size) - lgs) - lfact_c(y, lfact)) - kHalfLn2Pi;
        if (beta0) {
            const double l = log_pos(y * rcp_pos(nf[(int64_t)j * n + i]) + 0.1);
            for (int u = 0; u < P; u++) b[u] += ls[u * S + j] * l;
        }
    }
    if (beta0) for (int u = 0; u < P; u++) beta0[(int64_t)u * n + i] = b[u];
}

// ---------------------------------------------------------------------------------------
// IRLS
// ---------------------------------------------------------------------------------------
// one sweep over the samples at coefficients beta: X'WX (packed, no ridge), X'Wz and the deviance
template <int P>
__device__ __forceinline__ void irls_pass(const double* beta, double alpha, double size, int S, int stride,
                                          const double* ys, const double* nfs, const double* cs, const double* Xs,
                                          LogTab tab, Sym<P>& A, double* b, double& dev)
{
#pragma unroll
    for (int k = 0; k < P * (P + 1) / 2; k++) A.v[k] = 0.0;
#pragma unroll
    for (int u = 0; u < P; u++) b[u] = 0.0;
    double ll = 0.0;
#pragma unroll 1
    for (int j = 0; j < S; j++) {
        const double yj = ys[j * stride], nfj = nfs[j * stride];
        double eta = 0.0;
#pragma unroll
        for (int u = 0; u < P; u++) eta += Xs[j * P + u] * beta[u];
        double mu = nfj * exp(eta);
        double lmn = eta;
        if (!(mu >= kMinMu)) { mu = kMinMu; lmn = log_pos(kMinMu * rcp_pos(nfj)); }     // fmax(mu, minmu)
        ll += nb_logdens(yj, size, alpha, mu, cs[j * stride], tab);
        const double w = mu * rcp_pos(1.0 + alpha * mu);
        const double z = lmn + (yj - mu) * rcp_pos(mu);
#pragma unroll
        for (int u = 0; u < P; u++) {
            const double xu = Xs[j * P + u];
            b[u] += w * z * xu;
#pragma unroll
            for (int v = 0; v <= u; v++) A.v[u * (u + 1) / 2 + v] += w * xu * Xs[j * P + v];
        }
    }
    dev = -2.0 * ll;
}

template <int P>
__global__ void __launch_bounds__(kWaldThreads)
wald_irls_kernel(int64_t n, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ K, const double* __restrict__ nf,
                 const double* __restrict__ dispersion, const uint8_t* __restrict__ flags,
                 const double* __restrict__ cmat, double* __restrict__ beta0,
                 double* __restrict__ beta_out /*P x n, natural log scale*/, int32_t* __restrict__ iter_out,
                 unsigned long long* __restrict__ work_counter)
{
    extern __shared__ double smem[];
    const int stride = kWaldThreads;
    double* ys = smem + threadIdx.x;
    double* nfs = smem + (size_t)S * stride + threadIdx.x;
    double* cs = smem + (size_t)2 * S * stride + threadIdx.x;
    double* Xs = smem + (size_t)3 * S * stride;
    __shared__ __align__(16) double tab[2 * kLogTabN];
    for (int k = threadIdx.x; k < S * P; k += blockDim.x) Xs[k] = des->X[k];
    load_log_table(tab);
    __syncthreads();
    const LogTab tabh = log_tab_handle(tab);
    const unsigned lane = threadIdx.x & 31u;
    const double lambda = 1e-6 / (kLn2 * kLn2);

    bool active = false, exhausted = false, fresh = false;
    int64_t i = 0;
    double beta[P], beta_mu[P], rhs[P];          // beta_mu: the coefficients of the last sweep (of the fitted means)
    Sym<P> A;
    double alpha = 1.0, size = 1.0, dev_old = 0.0;
    int iter = 0;
#pragma unroll
    for (int u = 0; u < P; u++) { beta[u] = 0.0; beta_mu[u] = 0.0; rhs[u] = 0.0; }
#pragma unroll
    for (int k = 0; k < P * (P + 1) / 2; k++) A.v[k] = 0.0;

    while (true) {
        const bool want = !active && !exhausted;
        const unsigned need = __ballot_sync(0xffffffffu, want);
        if (need) {
            unsigned long long base = 0;
            const int leader = __ffs(need) - 1;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned long long)__popc(need));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (want) {
                i = (int64_t)(base + __popc(need & ((1u << lane) - 1u)));
                if (i >= n) {
                    exhausted = true;
                } else if (flags[i] & CD_FLAG_ALLZERO) {
                    iter_out[i] = 0;
#pragma unroll
                    for (int u = 0; u < P; u++) beta_out[(int64_t)u * n + i] = NAN;
                } else {
                    for (int j = 0; j < S; j++) {
                        ys[j * stride] = (double)K[(int64_t)j * n + i];
                        nfs[j * stride] = nf[(int64_t)j * n + i];
                        cs[j * stride] = cmat[(int64_t)j * n + i];
                    }
#pragma unroll
                    for (int u = 0; u < P; u++) beta[u] = beta0[(int64_t)u * n + i];
                    alpha = dispersion[i];
                    size = rcp_pos(alpha);
                    active = true; fresh = true;
                    iter = 0; dev_old = 0.0;
                }
            }
        }
        if (__all_sync(0xffffffffu, !active)) {
            if (__all_sync(0xffffffffu, exhausted)) break;
            continue;
        }
        // ---- solve the ridge normal equations from the previous sweep ----
        bool finished = false;
        if (active && !fresh) {
            iter++;
            Sym<P> Ar = A;
#pragma unroll
            for (int u = 0; u < P; u++) Ar.v[u * (u + 1) / 2 + u] += lambda;
            chol_logdet<P>(Ar);
            double bn[P];
#pragma unroll
            for (int u = 0; u < P; u++) bn[u] = rhs[u];
            chol_solve<P>(Ar, bn);
            bool big = false;
#pragma unroll
            for (int u = 0; u < P; u++) { beta[u] = bn[u]; big = big || (fabs(bn[u]) > 30.0); }
            if (big) { iter = 100; finished = true; }
        }
        __syncwarp();
        // ---- one sweep over the replicates at the current coefficients ----
        double dev = 0.0;
        if (active && !finished) {
            irls_pass<P>(beta, alpha, size, S, stride, ys, nfs, cs, Xs, tabh, A, rhs, dev);
#pragma unroll
            for (int u = 0; u < P; u++) beta_mu[u] = beta[u];
        }
        __syncwarp();
        if (active && !finished) {
            if (fresh) {
                fresh = false;
            } else {
                const double conv_test = fabs(dev - dev_old) / (fabs(dev) + 0.1);
                if (isnan(conv_test)) { iter = 100; finished = true; }
                else if (iter > 1 && conv_test < 1e-8) finished = true;
                else if (iter >= 100) finished = true;
                dev_old = dev;
            }
        }
        if (finished) {
#pragma unroll
            for (int u = 0; u < P; u++) beta_out[(int64_t)u * n + i] = beta[u];
            // DESeq2's fitBeta stops on |beta| > 30 before it updates the fitted means, and its weights for the standard
            // errors and hat values are those means: the finalisation takes them from here (this row's start values
            // are not read again)
#pragma unroll
            for (int u = 0; u < P; u++) beta0[(int64_t)u * n + i] = beta_mu[u];
            iter_out[i] = iter;
            active = false;
        }
    }
}

// ---------------------------------------------------------------------------------------
// finalisation
// ---------------------------------------------------------------------------------------
// R mean(x, trim): sort, drop floor(n * trim) from each end
__device__ __forceinline__ double trimmed_mean_dev(double* v, int n, double trim)
{
    for (int a = 1; a < n; a++) {
        const double x = v[a];
        int b = a - 1;
        while (b >= 0 && v[b] > x) { v[b + 1] = v[b]; b--; }
        v[b + 1] = x;
    }
    const int lo = (int)floor((double)n * trim);
    double s = 0.0;
    for (int a = lo; a < n - lo; a++) s += v[a];
    return s / (double)(n - 2 * lo);
}

__device__ __forceinline__ int trim_bin(int n) { return n <= 3 ? 0 : (n <= 23 ? 1 : 2); }

template <int P>
__global__ void __launch_bounds__(kWaldThreads)
wald_final_kernel(int64_t n, int S, const CdDesign* __restrict__ des, const int32_t* __restrict__ K, const double* __restrict__ nf,
                  const double* __restrict__ dispersion, uint8_t* __restrict__ flags,
                  const double* __restrict__ cmat, const double* __restrict__ beta_nat,
                  const double* __restrict__ beta_mu_in, const int32_t* __restrict__ iter_in,
                  double* __restrict__ beta_out, double* __restrict__ se_out, double* __restrict__ stat_out,
                  double* __restrict__ pvalue_out, double* __restrict__ deviance_out, double* __restrict__ maxCooks_out,
                  int32_t* __restrict__ betaIter_out, double* __restrict__ mu_out)
{
    __shared__ double Xs[CD_MAXS * CD_MAXP];
    __shared__ int cell[CD_MAXS], cell_size[CD_MAXS];
    __shared__ __align__(16) double tab[2 * kLogTabN];
    for (int k = threadIdx.x; k < S * P; k += blockDim.x) Xs[k] = des->X[k];
    for (int k = threadIdx.x; k < S; k += blockDim.x) { cell[k] = des->cell[k]; cell_size[k] = des->cell_size[k]; }
    load_log_table(tab);
    __syncthreads();
    const LogTab tabh = log_tab_handle(tab);
    const int ncell = des->ncell, any3 = des->any3;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool mu_only = (mu_out != nullptr);
    if (flags[i] & CD_FLAG_ALLZERO) {
        if (mu_only) { for (int j = 0; j < S; j++) mu_out[(int64_t)j * n + i] = NAN; return; }
        for (int u = 0; u < P; u++) { beta_out[(int64_t)u * n + i] = NAN; se_out[(int64_t)u * n + i] = NAN; }
        stat_out[i] = NAN; pvalue_out[i] = NAN; deviance_out[i] = NAN; betaIter_out[i] = 0;
        if (maxCooks_out) maxCooks_out[i] = NAN;
        return;
    }
    const double alpha = dispersion[i];
    const double size = rcp_pos(alpha);
    const double lambda = 1e-6 / (kLn2 * kLn2);
    double beta[P], beta_w[P], se[P];       // beta_w: the coefficients of the fitted means that weigh X'WX and the hat values
    int iter = 1;
    double qsum = 0.0;
    for (int j = 0; j < S; j++) qsum += (double)K[(int64_t)j * n + i] * rcp_pos(nf[(int64_t)j * n + i]);
    if (P == 1) {
        beta[0] = log_pos(qsum / S);          // fitNbinomGLMs intercept-only shortcut (natural log scale)
        beta_w[0] = beta[0];
    } else {
#pragma unroll
        for (int u = 0; u < P; u++) { beta[u] = beta_nat[(int64_t)u * n + i]; beta_w[u] = beta_mu_in[(int64_t)u * n + i]; }
        iter = iter_in[i];
    }
    if (mu_only) {
        for (int j = 0; j < S; j++) {
            double eta = 0.0;
#pragma unroll
            for (int u = 0; u < P; u++) eta += Xs[j * P + u] * beta[u];
            mu_out[(int64_t)j * n + i] = fmax(nf[(int64_t)j * n + i] * exp(eta), kMinMu);
        }
        return;
    }
    // X'WX at the final coefficients (weights at the floored mu; at mu itself for the p = 1 shortcut)
    Sym<P> A;
#pragma unroll
    for (int k = 0; k < P * (P + 1) / 2; k++) A.v[k] = 0.0;
    double loglike = 0.0;
    for (int j = 0; j < S; j++) {
        const double yj = (double)K[(int64_t)j * n + i], nfj = nf[(int64_t)j * n + i];
        double eta = 0.0, eta_w = 0.0;
#pragma unroll
        for (int u = 0; u < P; u++) { eta += Xs[j * P + u] * beta[u]; eta_w += Xs[j * P + u] * beta_w[u]; }
        const double muw = nfj * exp(eta);                   // unfloored, as stored by nbinomWaldTest
        loglike += nb_logdens(yj, size, alpha, muw, cmat[(int64_t)j * n + i], tabh);
        const double muc = (P == 1) ? muw : fmax(nfj * exp(eta_w), kMinMu);
        const double w = muc * rcp_pos(1.0 + alpha * muc);
#pragma unroll
        for (int u = 0; u < P; u++)
#pragma unroll
            for (int v = 0; v <= u; v++) A.v[u * (u + 1) / 2 + v] += w * Xs[j * P + u] * Xs[j * P + v];
    }
    Sym<P> Ar = A, Ari;
    if (P > 1) {
#pragma unroll
        for (int u = 0; u < P; u++) Ar.v[u * (u + 1) / 2 + u] += lambda;
    }
    chol_logdet<P>(Ar);
    chol_inverse<P>(Ar, Ari);
    bool noconv = (P > 1) && !(iter < 100);
#pragma unroll
    for (int u = 0; u < P; u++) {
        double s = 0.0;               // sigma_uu = sum_kl Ari[u][k] A[k][l] Ari[l][u]
#pragma unroll
        for (int k = 0; k < P; k++)
#pragma unroll
            for (int l = 0; l < P; l++) s += Ari.v[sidx<P>(u, k)] * A.v[sidx<P>(k, l)] * Ari.v[sidx<P>(l, u)];
        se[u] = kLog2e * sqrt(fmax(s, 0.0));
        noconv = noconv || !(s > 0.0) || isnan(beta[u]);
    }
    uint8_t f = flags[i];
    if (noconv) f |= CD_FLAG_BETA_NOCONV;
    if (maxCooks_out) {
        // robust method-of-moments dispersion for Cook's distance
        double v, tmp[CD_MAXS];
        if (any3) {
            v = -INFINITY;
            for (int c = 0; c < ncell; c++) {
                const int nc = cell_size[c];
                if (nc < 3) continue;
                const double trimr = (trim_bin(nc) == 0) ? 1.0 / 3.0 : (trim_bin(nc) == 1 ? 1.0 / 4.0 : 1.0 / 8.0);
                const double scalec = (trim_bin(nc) == 0) ? 2.04 : (trim_bin(nc) == 1 ? 1.86 : 1.51);
                int k = 0;
                for (int j = 0; j < S; j++) if (cell[j] == c) tmp[k++] = (double)K[(int64_t)j * n + i] / nf[(int64_t)j * n + i];
                const double cm = trimmed_mean_dev(tmp, nc, trimr);
                k = 0;
                for (int j = 0; j < S; j++) if (cell[j] == c) {
                    const double d = (double)K[(int64_t)j * n + i] / nf[(int64_t)j * n + i] - cm;
                    tmp[k++] = d * d;
                }
                const double ve = scalec * trimmed_mean_dev(tmp, nc, trimr);
                if (ve > v) v = ve;
            }
        } else {
            for (int j = 0; j < S; j++) tmp[j] = (double)K[(int64_t)j * n + i] / nf[(int64_t)j * n + i];
            const double rm = trimmed_mean_dev(tmp, S, 1.0 / 8.0);
            for (int j = 0; j < S; j++) { const double d = (double)K[(int64_t)j * n + i] / nf[(int64_t)j * n + i] - rm; tmp[j] = d * d; }
            v = 1.51 * trimmed_mean_dev(tmp, S, 1.0 / 8.0);
        }
        const double mq = qsum / S;
        const double ar = fmax((v - mq) / (mq * mq), 0.04);
        double mc = -INFINITY, ck_best = -INFINITY, y_best = 0.0;
        for (int j = 0; j < S; j++) {
            const double yj = (double)K[(int64_t)j * n + i], nfj = nf[(int64_t)j * n + i];
            double eta = 0.0, eta_w = 0.0;
#pragma unroll
            for (int u = 0; u < P; u++) { eta += Xs[j * P + u] * beta[u]; eta_w += Xs[j * P + u] * beta_w[u]; }
            const double muw = nfj * exp(eta);
            const double muc = (P == 1) ? muw : fmax(nfj * exp(eta_w), kMinMu);
            const double w = muc / (1.0 + alpha * muc);
            double h = 0.0;
#pragma unroll
            for (int u = 0; u < P; u++)
#pragma unroll
                for (int v2 = 0; v2 < P; v2++)
                    h += Xs[j * P + u] * Ari.v[sidx<P>(u, v2)] * Xs[j * P + v2];
            h *= w;
            const double V = muw + ar * muw * muw;
            const double ck = (yj - muw) * (yj - muw) / V / (double)P * h / ((1.0 - h) * (1.0 - h));
            if (cell_size[cell[j]] >= 3 && ck > mc) mc = ck;
            if (ck > ck_best) { ck_best = ck; y_best = yj; }        // which.max: first maximum
        }
        int greater = 0;
        for (int j = 0; j < S; j++) greater += ((double)K[(int64_t)j * n + i] > y_best);
        if (greater >= 3) f |= CD_FLAG_COOKS_KEEP;
        maxCooks_out[i] = (S > P && any3) ? mc : NAN;
    }
    flags[i] = f;
#pragma unroll
    for (int u = 0; u < P; u++) {
        beta_out[(int64_t)u * n + i] = kLog2e * beta[u];
        se_out[(int64_t)u * n + i] = se[u];
    }
    const double st = (kLog2e * beta[P - 1]) / se[P - 1];
    stat_out[i] = st;
    pvalue_out[i] = erfc(fabs(st) * 0.70710678118654752440);
    deviance_out[i] = -2.0 * loglike;
    betaIter_out[i] = iter;
}

// ---------------------------------------------------------------------------------------
// The theta-grid fits (design ~ 1, chicdiff.R:1641-1647) are only asked for their total deviance: fitNbinomGLMs'
// intercept-only shortcut (beta = log mean(K / nf)) and -2 log-likelihood at mu = nf exp(beta), in one kernel over the
// virtual regions of the batch, with the arithmetic of wald_prep_kernel + wald_final_kernel<1>.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
wald_deviance_p1_kernel(int64_t n, int S, const int32_t* __restrict__ K, const double* __restrict__ nf,
                        const double* __restrict__ dispersion, const uint8_t* __restrict__ flags, const double* __restrict__ lfact,
                        double* __restrict__ deviance_out)
{
    __shared__ __align__(16) double tab[2 * kLogTabN];
    load_log_table(tab);
    __syncthreads();
    const LogTab tabh = log_tab_handle(tab);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flags[i] & CD_FLAG_ALLZERO) { deviance_out[i] = NAN; return; }
    const double alpha = dispersion[i];
    const double size = rcp_pos(alpha);
    double qsum = 0.0;
    for (int j = 0; j < S; j++) qsum += (double)K[(int64_t)j * n + i] * rcp_pos(nf[(int64_t)j * n + i]);
    const double beta = log_pos(qsum / S);
    const double eb = exp(beta);
    double loglike = 0.0;
    if (size > kHugeSize) {
        for (int j = 0; j < S; j++)
            loglike += dnbinom_mu_log((double)K[(int64_t)j * n + i], size, nf[(int64_t)j * n + i] * eb);
    } else {
        // lgamma(y + size) - lgamma(size) as in the line search's posterior (posterior.cuh): Stirling parts per sample,
        // the logarithm of the gamma rationals once for the region
        const GammaParts gr = gamma_parts<true>(size, tabh);
        const double inv_den_r = rcp_fast(gr.den);
        double qprod = 1.0;
        for (int j = 0; j < S; j++) {
            const double yj = (double)K[(int64_t)j * n + i], nfj = nf[(int64_t)j * n + i];
            const GammaParts g = gamma_parts<true>(yj + size, tabh);
            qprod *= g.den * inv_den_r;
            if (__double2hiint(qprod) > 0x5fe00000) { loglike -= log_pos_v2(qprod, tabh); qprod = 1.0; }
            const double c = ((g.st - gr.st) - lfact_c(yj, lfact)) - kHalfLn2Pi;
            const double mu = nfj * eb;
            const double l1 = log_pos_v2(1.0 + mu * alpha, tabh);
            const double l2 = log_pos_v2(mu * rcp_fast(size + mu), tabh);
            loglike += (c - size * l1) + yj * l2;
        }
        loglike -= log_pos_v2(qprod, tabh);
    }
    deviance_out[i] = -2.0 * loglike;
}

cudaError_t launch_wald_deviance_p1(int64_t n, int S, const int32_t* K, const double* nf, const double* dispersion,
                                    const uint8_t* flags, const double* lfact, double* deviance, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    wald_deviance_p1_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, K, nf, dispersion, flags, lfact, deviance);
    return cudaGetLastError();
}

cudaError_t launch_wald(int64_t n, int S, int p, const CdDesign* des, const int32_t* K, const double* nf, const double* dispersion,
                        uint8_t* flags, const WaldScratch& ws, double* beta, double* betaSE, double* stat,
                        double* pvalue, double* deviance, double* maxCooks, int32_t* betaIter, double* mu_out,
                        cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    cudaError_t e;
    wald_prep_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, p, des, K, nf, dispersion, flags, ws.lfact, ws.cmat, p > 1 ? ws.beta0 : nullptr);
    const int threads = kWaldThreads;
    const size_t smem = ((size_t)3 * S * threads + (size_t)S * p) * sizeof(double);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t want = (n + threads - 1) / threads;
#define CD_IRLS(P_)                                                                                              \
    {                                                                                                            \
        e = cudaMemsetAsync(ws.work_counter, 0, sizeof(unsigned long long), st);                                 \
        if (e != cudaSuccess) return e;                                                                          \
        e = cudaFuncSetAttribute(wald_irls_kernel<P_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
        if (e != cudaSuccess) return e;                                                                          \
        int per_sm = 1;                                                                                          \
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wald_irls_kernel<P_>, threads, smem);         \
        if (e != cudaSuccess) return e;                                                                          \
        const int64_t resident = (int64_t)sms * (per_sm > 0 ? per_sm : 1);                                       \
        wald_irls_kernel<P_><<<(int)(want < resident ? want : resident), threads, smem, st>>>(                   \
            n, S, des, K, nf, dispersion, flags, ws.cmat, ws.beta0, ws.beta_nat, ws.iter, ws.work_counter);   \
    }
#define CD_FINAL(P_)                                                                                             \
    wald_final_kernel<P_><<<blocks_for(n, threads), threads, 0, st>>>(n, S, des, K, nf, dispersion, flags, ws.cmat, \
        ws.beta_nat, ws.beta0, ws.iter, beta, betaSE, stat, pvalue, deviance, maxCooks, betaIter, mu_out)
    switch (p) {
        case 1: CD_FINAL(1); break;
        case 2: CD_IRLS(2); CD_FINAL(2); break;
        case 3: CD_IRLS(3); CD_FINAL(3); break;
        case 4: CD_IRLS(4); CD_FINAL(4); break;
        default: return cudaErrorInvalidValue;
    }
#undef CD_IRLS
#undef CD_FINAL
    return cudaGetLastError();
}

}  // namespace cd
