// posterior.cuh -- the Cox-Reid adjusted profile log-posterior of log(alpha) and its derivative, the function every
// trip of the dispersion line search evaluates (dispersion.cu).  Kept in a header of its own so that the accuracy
// tests can compile it for the host (tests/device_math) and compare it with the oracle without a GPU.
#pragma once
#include "common.cuh"

namespace cd {

// ---------------------------------------------------------------------------------------
// Cox-Reid adjusted profile log-posterior of log(alpha) (DESeq2.cpp log_posterior) and its
// derivative (dlog_posterior), evaluated together at one point.  The line search needs the
// posterior at every proposal and the derivative at every accepted one; computed together they
// share exp(a), w_j = 1/(1/mu_j + alpha), log(1 + mu_j alpha), log(y_j + r + 10) and the shifted
// gamma-function rationals, so the pair costs ~1.3x the posterior alone, and the lanes of a warp
// never split into "needs the derivative" and "does not".
// ys / mus point at the region's replicates in shared memory, element j at [j * stride];
// Xd is the S x P model matrix (row-major; shared memory on the device: every lane reads the same entry).
// WANT_D = false (grid refit) skips the derivative.
//
// Formulation (what the per-source-line profile of round 1 led to; profiles/r01_final_fit_disp_source_lines.txt):
//   * log Gamma and digamma of x = y_j + r come from the shift-10 scheme of common.cuh, but the logarithm of the
//     rational's denominator is not taken per replicate: with q_j = den_j / den_r (>= 1, the ratio against the rational
//     of r = 1/alpha alone) the sum over replicates of [log den_j - log den_r] is the logarithm of the PRODUCT of the
//     q_j, taken once per evaluation (earlier only if the running product passes 2^511; one q_j is below 2e89 for any
//     32-bit count and alpha <= 32): 2 + 1/S instead of 3 logarithms per replicate, and a zero count still contributes
//     (almost) exactly zero;
//   * the four highest coefficients of the Stirling and of the digamma series are rounded to 21 bits (they multiply
//     f^3 <= 1e-6 and higher: <= 3e-17 absolute), which makes them instruction immediates instead of constant loads;
//   * p = 1 and p = 2 (every fit of the default pipeline) use the closed-form determinant and inverse of X'WX with
//     one Newton reciprocal and one logarithm; p = 3, 4 keep the packed Cholesky;
//   * TABLOG = true takes every logarithm with log_pos_v2 (table in shared memory, no reciprocal): the line search
//     (fit_disp_kernel); false with log_pos: the grid refit (fit_disp_grid_kernel), which has no table.
// ---------------------------------------------------------------------------------------
struct GammaParts { double st, dgs, num, den; };      // st: Stirling part of lgamma; dgs: series part of digamma

template <bool TABLOG>
__device__ __forceinline__ double post_log(double x, LogTab tab)
{
    return TABLOG ? log_pos_v2(x, tab) : log_pos(x);
}

// the pieces of lgamma_digamma_pos, with the rational's denominator handed back instead of logged
template <bool TABLOG>
__device__ __forceinline__ GammaParts gamma_parts(double x, LogTab tab)
{
    GammaParts g;
    // den = x (x+1) ... (x+9) and num = d den / dx (num / den = sum of 1 / (x+k)) through u = x (x+9):
    // (x+k)(x+9-k) = u + k (9-k), so den = u (u+8) (u+14) (u+18) (u+20), and num = d den / du (2x + 9):
    // 16 FP64 instructions instead of the 27 of the factor-by-factor recurrence, all terms positive
    const double u9 = x * (x + 9.0);
    double den = u9, num = 1.0;
    {
        const double t8 = u9 + 8.0, t14 = u9 + 14.0, t18 = u9 + 18.0, t20 = u9 + 20.0;
        num = t8 + den;           den *= t8;
        num = fma(num, t14, den); den *= t14;
        num = fma(num, t18, den); den *= t18;
        num = fma(num, t20, den); den *= t20;
    }
    num *= fma(x, 2.0, 9.0);
    const double xs = x + 10.0;
    const double xi = rcp_fast(xs);
    const double f = xi * xi;
    const double lxs = post_log<TABLOG>(xs, tab);
    // kLgamC[6..3] and kDigamC[6..3] with the low word zero
    double t = fma(f, 0x1.a41a4p-8, -0x1.f6ab1p-10);
    t = fma(f, t, 0x1.b951ep-11);
    t = fma(f, t, -0x1.38138p-11);
#pragma unroll
    for (int k = 2; k >= 0; k--) t = fma(f, t, kLgamC[k]);
    g.st = ((xs - 0.5) * lxs - xs) + xi * t;
    double u = fma(f, -0x1.55555p-4, 0x1.5995ap-6);
    u = fma(f, u, -0x1.f07c2p-8);
    u = fma(f, u, 0x1.11111p-8);
#pragma unroll
    for (int k = 2; k >= 0; k--) u = fma(f, u, kDigamC[k]);
    g.dgs = (lxs - 0.5 * xi) + f * u;
    g.num = num; g.den = den;
    return g;
}

// prior_inv_sigmasq = 1 / prior variance of log(alpha) (the caller takes the reciprocal once per region)
template <int P, bool WANT_D, bool TABLOG>
__device__ __forceinline__ void eval_post(double a, const double* ys, const double* mus, int stride, int S,
                                          const double* Xd, LogTab tab,
                                          double prior_mean, double prior_inv_sigmasq, bool use_prior,
                                          double& lp_out, double& dlp_out)
{
    const double alpha = exp_mid(a);
    const double r = rcp_fast(alpha);
    const double log_r = -a;                            // log(1/alpha)
    const GammaParts gr = gamma_parts<TABLOG>(r, tab);
    const double inv_den_r = rcp_fast(gr.den);
    const double dgr = gr.dgs - gr.num * inv_den_r;
    Sym<P> B, dB;
#pragma unroll
    for (int k = 0; k < P * (P + 1) / 2; k++) { B.v[k] = 0.0; dB.v[k] = 0.0; }
    double ll = 0.0, ds = 0.0, qprod = 1.0;
    // (measured in round 1: unrolling this loop by 2 doubles the registers and is 24 % slower)
#pragma unroll 1
    for (int j = 0; j < S; j++) {
        const double yj = ys[j * stride], muj = mus[j * stride];
        const double ma = muj * alpha;
        const double ropm = rcp_fast(1.0 + ma);
        const double w = muj * ropm;                    // = 1 / (1/mu + alpha)
        const double dw = -w * w;
        if (P == 1) {
            B.v[0] += w;
            if (WANT_D) dB.v[0] += dw;
        } else {
#pragma unroll
            for (int u = 0; u < P; u++)
#pragma unroll
                for (int v = 0; v <= u; v++) {
                    const double xx = Xd[j * P + u] * Xd[j * P + v];
                    B.v[u * (u + 1) / 2 + v] += w * xx;
                    if (WANT_D) dB.v[u * (u + 1) / 2 + v] += dw * xx;
                }
        }
        const double l1 = post_log<TABLOG>(1.0 + ma, tab);
        const GammaParts g = gamma_parts<TABLOG>(yj + r, tab);
        qprod *= g.den * inv_den_r;                       // den_j / den_r >= 1
        if (__double2hiint(qprod) > 0x5fe00000) { ll -= post_log<TABLOG>(qprod, tab); qprod = 1.0; }      // > 2^511: rare
        // mu + r = r (1 + mu alpha): log(mu + r) = log r + log(1 + mu alpha), 1/(mu + r) = alpha / (1 + mu alpha)
        // for a zero count g.st - gr.st and dgr - dg are exactly zero (same instruction sequence, same input)
        ll += ((g.st - gr.st) - yj * (log_r + l1)) - r * l1;
        if (WANT_D) {
            const double dg = g.dgs - g.num * rcp_fast(g.den);
            ds += ((dgr - dg) + (l1 - ma * ropm)) + yj * (alpha * ropm);
        }
    }
    ll -= post_log<TABLOG>(qprod, tab);                  // one logarithm for the gamma rationals of all replicates
    double cr, dcr = 0.0;
    if (P == 1) {
        const double b = B.v[0];
        cr = -0.5 * ((b > 0.0) ? post_log<TABLOG>(b, tab) : NAN);
        if (WANT_D) dcr = -0.5 * (dB.v[0] * rcp_fast(b));
    } else if (P == 2) {
        const double det = B.v[0] * B.v[2] - B.v[1] * B.v[1];
        const bool ok = (B.v[0] > 0.0) && (det > 0.0);
        cr = -0.5 * (ok ? post_log<TABLOG>(det, tab) : NAN);
        if (WANT_D) {
            // tr(B^-1 dB) = (B11 dB00 - 2 B10 dB10 + B00 dB11) / det
            const double tr = (B.v[2] * dB.v[0] - 2.0 * B.v[1] * dB.v[1] + B.v[0] * dB.v[2]) * rcp_fast(det);
            dcr = -0.5 * tr;
        }
    } else {
        Sym<P> L = B;
        cr = -0.5 * chol_logdet<P>(L);
        if (WANT_D) {
            Sym<P> Bi;
            chol_inverse<P>(L, Bi);
            double tr = 0.0;
#pragma unroll
            for (int u = 0; u < P; u++)
#pragma unroll
                for (int v = 0; v < P; v++) tr += Bi.v[sidx<P>(u, v)] * dB.v[sidx<P>(v, u)];
            dcr = -0.5 * tr;
        }
    }
    double pr = 0.0;
    if (use_prior) {
        const double d = a - prior_mean;
        pr = (-0.5 * d * d) * prior_inv_sigmasq;
    }
    lp_out = ll + pr + cr;
    if (WANT_D) {
        const double dpr = use_prior ? (-1.0 * (a - prior_mean)) * prior_inv_sigmasq : 0.0;
        dlp_out = ((r * r) * ds + dcr) * alpha + dpr;
    }
}

// The first formulation (round 1): one lgamma_digamma_pos per replicate with its own log of the rational's denominator,
// Cholesky for every p.  Kept as the reference the accuracy tests compare eval_post with (tests/test_device_math.py);
// the kernels do not use it.
template <int P, bool WANT_D>
__device__ __forceinline__ void eval_post_ref(double a, const double* ys, const double* mus, int stride, int S,
                                              const double* Xd, double prior_mean, double prior_sigmasq, bool use_prior,
                                              double& lp_out, double& dlp_out)
{
    const double alpha = exp(a);
    const double r = rcp_pos(alpha);
    const double log_r = -a;
    double lgr, dgr;
    lgamma_digamma_pos(r, lgr, dgr);
    Sym<P> B, dB;
#pragma unroll
    for (int k = 0; k < P * (P + 1) / 2; k++) { B.v[k] = 0.0; dB.v[k] = 0.0; }
    double ll = 0.0, ds = 0.0;
#pragma unroll 1
    for (int j = 0; j < S; j++) {
        const double yj = ys[j * stride], muj = mus[j * stride];
        const double ma = muj * alpha;
        const double ropm = rcp_pos(1.0 + ma);
        const double w = muj * ropm;
        const double dw = -w * w;
#pragma unroll
        for (int u = 0; u < P; u++)
#pragma unroll
            for (int v = 0; v <= u; v++) {
                const double xx = Xd[j * P + u] * Xd[j * P + v];
                B.v[u * (u + 1) / 2 + v] += w * xx;
                if (WANT_D) dB.v[u * (u + 1) / 2 + v] += dw * xx;
            }
        const double l1 = log_pos(1.0 + ma);
        double lg, dg;
        lgamma_digamma_pos(yj + r, lg, dg);
        ll += ((lg - lgr) - yj * (log_r + l1)) - r * l1;
        if (WANT_D) ds += ((dgr - dg) + (l1 - ma * ropm)) + yj * (alpha * ropm);
    }
    const double cr = -0.5 * chol_logdet<P>(B);
    double pr = 0.0;
    if (use_prior) {
        const double d = a - prior_mean;
        pr = -0.5 * d * d / prior_sigmasq;
    }
    lp_out = ll + pr + cr;
    if (WANT_D) {
        Sym<P> Bi;
        chol_inverse<P>(B, Bi);
        double tr = 0.0;
#pragma unroll
        for (int u = 0; u < P; u++)
#pragma unroll
            for (int v = 0; v < P; v++) tr += Bi.v[sidx<P>(u, v)] * dB.v[sidx<P>(v, u)];
        const double dcr = -0.5 * tr;
        const double dpr = use_prior ? -1.0 * (a - prior_mean) / prior_sigmasq : 0.0;
        dlp_out = ((r * r) * ds + dcr) * alpha + dpr;
    }
}

}  // namespace cd
