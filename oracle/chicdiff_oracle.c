/*
 * chicdiff_oracle.c -- CPU restatement of Chicdiff's region-test hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load this library.
 * The product path (chicdiff_b200/) never links, imports or calls it.
 *
 * PARITY UNPINNED: the reference (/root/reference/Chicdiff/R/chicdiff.R) is R code
 * whose arithmetic on this path runs inside DESeq2 (Bioconductor, not vendored,
 * version not pinned; the golden table was written under R 3.5.1 => DESeq2
 * ~1.20-1.22), Chicago and base R.  No R interpreter exists in this image, the
 * bundled example inputs are absent from the mount, and the reference has no
 * tests, so this file restates the published algorithms from their call sites:
 *
 *   chicdiff.R:1540-1547   region group-by (sum N, sum FullMean)      -> orc_aggregate
 *   chicdiff.R:1561-1562   estimateSizeFactors (median of ratios)     -> orc_size_factors
 *   chicdiff.R:1583-1589,  FullMean scaling factors, NA rows <- size  -> orc_norm_factors
 *              1614-1615,  factors, theta mix, row geo-mean rescale
 *              1635-1638
 *   chicdiff.R:1573,1602,  estimateDispersions: GeneEst (rough/moment -> orc_deseq
 *              1643,1673   start, linear or IRLS mu, Cox-Reid APL
 *                          line search fitDisp, fitDispGrid), parametric
 *                          trend (Gamma-identity glm), prior variance, MAP
 *   chicdiff.R:1574,1603,  nbinomWaldTest: fitBeta ridge-QR IRLS /    -> orc_deseq
 *              1644,1674   intercept-only shortcut, hat diagonals,
 *                          Cook's distance, Wald stat and p-value
 *   chicdiff.R:1647        sum of deviances for the theta grid        -> caller sums out.deviance
 *
 * What IS pinned (tests/test_golden.py): the Wald p-value formula, BH and the
 * independent-filtering rule against the shipped golden table; lgamma, digamma,
 * trigamma, dnbinom_mu, pnorm, qf against SciPy; fitDisp optima against a
 * bounded scalar maximiser; IRLS against a Newton solve of the same likelihood.
 *
 * Matrix layout everywhere: "sample-major" = R's column-major n x S matrix,
 * element (region i, sample s) at [s*n + i].
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_MAXS 64
#define ORC_MAXP 4

/* ------------------------------------------------------------------ */
/* special functions                                                    */
/* ------------------------------------------------------------------ */

double orc_lgamma(double x) { return lgamma(x); }

/* digamma for x > 0: recurrence up to x >= 10, then the asymptotic series */
double orc_digamma(double x)
{
    double r = 0.0;
    if (!(x > 0.0)) return NAN;
    while (x < 10.0) { r -= 1.0 / x; x += 1.0; }
    double f = 1.0 / (x * x);
    double t = f * (-1.0 / 12.0 + f * (1.0 / 120.0 + f * (-1.0 / 252.0 + f * (1.0 / 240.0 +
               f * (-1.0 / 132.0 + f * (691.0 / 32760.0 + f * (-1.0 / 12.0)))))));
    return r + log(x) - 0.5 / x + t;
}

double orc_trigamma(double x)
{
    double r = 0.0;
    if (!(x > 0.0)) return NAN;
    while (x < 10.0) { r += 1.0 / (x * x); x += 1.0; }
    double f = 1.0 / (x * x);
    double t = 1.0 / x + 0.5 * f +
               (1.0 / x) * f * (1.0 / 6.0 + f * (-1.0 / 30.0 + f * (1.0 / 42.0 + f * (-1.0 / 30.0 +
               f * (5.0 / 66.0 + f * (-691.0 / 2730.0 + f * (7.0 / 6.0)))))));
    return r + t;
}

#define M_LN_SQRT_2PI_ 0.918938533204672741780329736406
#define M_LN_2PI_ 1.837877066409345483560659472811

/* Loader's saddle-point helpers as used by R's dbinom_raw (nmath/stirlerr.c, bd0.c) */
static double orc_stirlerr(double n)
{
    static const double S0 = 1.0 / 12.0, S1 = 1.0 / 360.0, S2 = 1.0 / 1260.0,
                        S3 = 1.0 / 1680.0, S4 = 1.0 / 1188.0;
    static const double sferr_halves[31] = {
        0.0, 0.1534264097200273452913848, 0.0810614667953272582196702,
        0.0548141210519176538961390, 0.0413406959554092940938221,
        0.03316287351993628748511048, 0.02767792568499833914878929,
        0.02374616365629749597132920, 0.02079067210376509311152277,
        0.01848845053267318523077934, 0.01664469118982119216319487,
        0.01513497322191737887351255, 0.01387612882307074799874573,
        0.01281046524292022692424986, 0.01189670994589177009505572,
        0.01110455975820691732662991, 0.010411265261972096497478567,
        0.009799416126158803298389475, 0.009255462182712732917728637,
        0.008768700134139385462952823, 0.008330563433362871256469318,
        0.007934114564314020547248100, 0.007573675487951840794972024,
        0.007244554301320383179543912, 0.006942840107209529865664152,
        0.006665247032707682442354394, 0.006408994188004207068439631,
        0.006171712263039457647532867, 0.005951370112758847735624416,
        0.005746216513010115682023589, 0.005554733551962801371038690};
    double nn;
    if (n <= 15.0) {
        nn = n + n;
        if (nn == (int)nn) return sferr_halves[(int)nn];
        return lgamma(n + 1.0) - (n + 0.5) * log(n) + n - M_LN_SQRT_2PI_;
    }
    nn = n * n;
    if (n > 500) return (S0 - S1 / nn) / n;
    if (n > 80) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

static double orc_bd0(double x, double np)
{
    if (!isfinite(x) || !isfinite(np) || np == 0.0) return NAN;
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        if (fabs(s) < 2.2250738585072014e-308) return s;
        double ej = 2 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; j++) {
            ej *= v;
            double s1 = s + ej / ((j << 1) + 1);
            if (s1 == s) return s1;
            s = s1;
        }
    }
    return x * log(x / np) + np - x;
}

static double orc_dbinom_raw_log(double x, double n, double p, double q)
{
    double lc, lf;
    if (p == 0) return (x == 0) ? 0.0 : -INFINITY;
    if (q == 0) return (x == n) ? 0.0 : -INFINITY;
    if (x == 0) {
        if (n == 0) return 0.0;
        return (p < 0.1) ? -orc_bd0(n, n * q) - n * p : n * log(q);
    }
    if (x == n) return (q < 0.1) ? -orc_bd0(n, n * p) - n * q : n * log(p);
    if (x < 0 || x > n) return -INFINITY;
    lc = orc_stirlerr(n) - orc_stirlerr(x) - orc_stirlerr(n - x) - orc_bd0(x, n * p) -
         orc_bd0(n - x, n * q);
    lf = M_LN_2PI_ + log(x) + log1p(-x / n);
    return lc - 0.5 * lf;
}

/* log dnbinom(x; size, mu) following R 3.x nmath/dnbinom.c:dnbinom_mu */
double orc_dnbinom_mu_log(double x, double size, double mu)
{
    if (x == 0 && size == 0) return 0.0;
    if (!isfinite(size)) {              /* Poisson limit */
        if (mu == 0) return (x == 0) ? 0.0 : -INFINITY;
        if (x == 0) return -mu;
        return -0.5 * log(2 * M_PI * x) - orc_stirlerr(x) - orc_bd0(x, mu);
    }
    if (x == 0)
        return size * (size < mu ? log(size / (size + mu)) : log1p(-mu / (size + mu)));
    if (x < 1e-10 * size) {
        double p = (size < mu ? log(size / (1 + size / mu)) : log(mu / (1 + mu / size)));
        return x * p - mu - lgamma(x + 1) + log1p(x * (x - 1) / (2 * size));
    }
    double p = size / (size + x);
    double ans = orc_dbinom_raw_log(size, x + size, size / (size + mu), mu / (size + mu));
    return log(p) + ans;
}

/* 2 * pnorm(|z|, lower.tail = FALSE) */
double orc_wald_pvalue(double z) { return erfc(fabs(z) * M_SQRT1_2); }

/* regularised incomplete beta by Lentz's continued fraction */
static double betacf(double a, double b, double x)
{
    const double tiny = 1e-300;
    double qab = a + b, qap = a + 1, qam = a - 1;
    double c = 1, d = 1 - qab * x / qap;
    if (fabs(d) < tiny) d = tiny;
    d = 1 / d;
    double h = d;
    for (int m = 1; m <= 500; m++) {
        int m2 = 2 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1 / d; h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1 / d;
        double del = d * c;
        h *= del;
        if (fabs(del - 1) < 1e-16) break;
    }
    return h;
}

static double pbeta_(double x, double a, double b)
{
    if (x <= 0) return 0;
    if (x >= 1) return 1;
    double bt = exp(lgamma(a + b) - lgamma(a) - lgamma(b) + a * log(x) + b * log1p(-x));
    if (x < (a + 1) / (a + b + 2)) return bt * betacf(a, b, x) / a;
    return 1 - bt * betacf(b, a, 1 - x) / b;
}

/* qf(prob, df1, df2) by bisection on the beta scale */
double orc_qf(double prob, double df1, double df2)
{
    double lo = 0, hi = 1;
    for (int it = 0; it < 200; it++) {
        double mid = 0.5 * (lo + hi);
        if (pbeta_(mid, 0.5 * df1, 0.5 * df2) < prob) lo = mid; else hi = mid;
    }
    double x = 0.5 * (lo + hi);
    return (df2 * x) / (df1 * (1 - x));
}

/* ------------------------------------------------------------------ */
/* small dense linear algebra (p <= ORC_MAXP)                           */
/* ------------------------------------------------------------------ */

/* Householder least squares: minimise ||A b - y||, A is m x p row-major (overwritten) */
static void ls_householder(double* A, double* y, int m, int p, double* b)
{
    for (int k = 0; k < p; k++) {
        double nrm = 0;
        for (int i = k; i < m; i++) nrm += A[i * p + k] * A[i * p + k];
        nrm = sqrt(nrm);
        if (nrm == 0) continue;
        double alpha = (A[k * p + k] > 0) ? -nrm : nrm;
        double v0 = A[k * p + k] - alpha;
        double vnorm2 = v0 * v0;
        for (int i = k + 1; i < m; i++) vnorm2 += A[i * p + k] * A[i * p + k];
        if (vnorm2 == 0) continue;
        for (int j = k + 1; j < p; j++) {
            double dot = v0 * A[k * p + j];
            for (int i = k + 1; i < m; i++) dot += A[i * p + k] * A[i * p + j];
            double f = 2 * dot / vnorm2;
            A[k * p + j] -= f * v0;
            for (int i = k + 1; i < m; i++) A[i * p + j] -= f * A[i * p + k];
        }
        double dot = v0 * y[k];
        for (int i = k + 1; i < m; i++) dot += A[i * p + k] * y[i];
        double f = 2 * dot / vnorm2;
        y[k] -= f * v0;
        for (int i = k + 1; i < m; i++) y[i] -= f * A[i * p + k];
        A[k * p + k] = alpha;
    }
    for (int k = p - 1; k >= 0; k--) {
        double s = y[k];
        for (int j = k + 1; j < p; j++) s -= A[k * p + j] * b[j];
        b[k] = s / A[k * p + k];
    }
}

/* determinant and inverse of a p x p matrix by Gaussian elimination with partial pivoting */
static double det_inv(const double* Ain, int p, double* inv)
{
    double a[ORC_MAXP][2 * ORC_MAXP];
    for (int i = 0; i < p; i++)
        for (int j = 0; j < p; j++) { a[i][j] = Ain[i * p + j]; a[i][p + j] = (i == j); }
    double det = 1;
    for (int k = 0; k < p; k++) {
        int piv = k;
        for (int i = k + 1; i < p; i++) if (fabs(a[i][k]) > fabs(a[piv][k])) piv = i;
        if (a[piv][k] == 0) { det = 0; if (inv) for (int i = 0; i < p * p; i++) inv[i] = NAN; return 0; }
        if (piv != k) {
            for (int j = 0; j < 2 * p; j++) { double t = a[k][j]; a[k][j] = a[piv][j]; a[piv][j] = t; }
            det = -det;
        }
        det *= a[k][k];
        double d = a[k][k];
        for (int j = 0; j < 2 * p; j++) a[k][j] /= d;
        for (int i = 0; i < p; i++) if (i != k) {
            double f = a[i][k];
            if (f != 0) for (int j = 0; j < 2 * p; j++) a[i][j] -= f * a[k][j];
        }
    }
    if (inv) for (int i = 0; i < p; i++) for (int j = 0; j < p; j++) inv[i * p + j] = a[i][p + j];
    return det;
}

static void xtwx(const double* X, const double* w, int S, int p, double* B)
{
    for (int a = 0; a < p; a++)
        for (int b = 0; b < p; b++) {
            double s = 0;
            for (int j = 0; j < S; j++) s += X[j * p + a] * w[j] * X[j * p + b];
            B[a * p + b] = s;
        }
}

/* ------------------------------------------------------------------ */
/* stage 1: aggregation  (chicdiff.R:1540-1547)                         */
/* ------------------------------------------------------------------ */

/* rows are region-contiguous (regionID, then otherEndID ascending = the order
 * data.table sums them in after setkey(fragData, otherEndID)).  N_rows / FM_rows are
 * sample-major R_rows-long columns.  Integer sums are exact (overflow -> NA_integer_ as in
 * R's isum); FullMean sums accumulate in long double like R's rsum and propagate NA. */
int orc_aggregate(int64_t n, int S, const int64_t* row_off, int64_t R_rows,
                  const int32_t* N_rows, const double* FM_rows,
                  int32_t* K_out, double* FM_out)
{
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) {
        for (int s = 0; s < S; s++) {
            int64_t acc = 0;
            long double f = 0.0L;
            for (int64_t r = row_off[i]; r < row_off[i + 1]; r++) {
                acc += N_rows[(int64_t)s * R_rows + r];
                f += FM_rows[(int64_t)s * R_rows + r];
            }
            K_out[(int64_t)s * n + i] = (acc > INT32_MAX || acc < -INT32_MAX) ? INT32_MIN : (int32_t)acc;
            FM_out[(int64_t)s * n + i] = (double)f;
        }
    }
    return 0;
}

/* ------------------------------------------------------------------ */
/* size factors (DESeq2 estimateSizeFactorsForMatrix; chicdiff.R:1561)  */
/* ------------------------------------------------------------------ */

static int cmp_double(const void* a, const void* b)
{
    double x = *(const double*)a, y = *(const double*)b;
    return (x > y) - (x < y);
}

static double median_inplace(double* v, int64_t m)
{
    if (m == 0) return NAN;
    qsort(v, (size_t)m, sizeof(double), cmp_double);
    return (m & 1) ? v[m / 2] : 0.5 * (v[m / 2 - 1] + v[m / 2]);
}

/* DESeqDataSetFromMatrix (chicdiff.R:1556-1559) refuses NA (NA_integer_ = INT32_MIN) and negative counts */
static int any_negative(int64_t n, int S, const int32_t* K)
{
    for (int64_t j = 0; j < (int64_t)S * n; j++)
        if (K[j] < 0) return 1;
    return 0;
}

/* returns -1 when every region has a zero count, -2 for NA or negative counts */
int orc_size_factors(int64_t n, int S, const int32_t* K, double* sf)
{
    if (any_negative(n, S, K)) return -2;
    double* lgm = (double*)malloc(sizeof(double) * (size_t)n);
    double* buf = (double*)malloc(sizeof(double) * (size_t)n);
    int64_t nfinite = 0;
    for (int64_t i = 0; i < n; i++) {
        long double acc = 0;
        for (int s = 0; s < S; s++) acc += log((double)K[(int64_t)s * n + i]);   /* log 0 = -Inf */
        lgm[i] = (double)(acc / S);
        if (isfinite(lgm[i])) nfinite++;
    }
    if (nfinite == 0) { free(lgm); free(buf); return -1; }
    for (int s = 0; s < S; s++) {
        int64_t m = 0;
        for (int64_t i = 0; i < n; i++) {
            int32_t k = K[(int64_t)s * n + i];
            if (isfinite(lgm[i]) && k > 0) buf[m++] = log((double)k) - lgm[i];
        }
        sf[s] = exp(median_inplace(buf, m));
    }
    free(lgm); free(buf);
    return 0;
}

/* ------------------------------------------------------------------ */
/* stage 2: normalisation factors (chicdiff.R:1583-1589,1614-1615,      */
/*          1635-1638,1666-1669)                                        */
/* ------------------------------------------------------------------ */

/* mode 0: "standard"  nf[i,s] = sf[s]
 * mode 1: "fullmean"  nf = M3
 * mode 2: "combined"  nf = sc(theta) */
int orc_norm_factors(int64_t n, int S, const double* FMagg, const double* sf, int mode,
                     double theta, double* nf)
{
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) {
        double m3[ORC_MAXS];
        if (mode == 0) {
            for (int s = 0; s < S; s++) nf[(int64_t)s * n + i] = sf[s];
            continue;
        }
        long double acc = 0;
        int anyna = 0;
        for (int s = 0; s < S; s++) {
            double v = FMagg[(int64_t)s * n + i];
            acc += log(v);
        }
        double g = exp((double)(acc / S));
        for (int s = 0; s < S; s++) {
            m3[s] = FMagg[(int64_t)s * n + i] / g;
            if (isnan(m3[s])) anyna = 1;
        }
        if (anyna) for (int s = 0; s < S; s++) m3[s] = sf[s];
        if (mode == 1) {
            for (int s = 0; s < S; s++) nf[(int64_t)s * n + i] = m3[s];
            continue;
        }
        long double acc2 = 0;
        double sc[ORC_MAXS];
        for (int s = 0; s < S; s++) {
            sc[s] = m3[s] * (1 - theta) + sf[s] * theta;
            acc2 += log(sc[s]);
        }
        double g2 = exp((double)(acc2 / S));
        for (int s = 0; s < S; s++) nf[(int64_t)s * n + i] = sc[s] / g2;
    }
    return 0;
}

/* ------------------------------------------------------------------ */
/* DESeq2 core                                                          */
/* ------------------------------------------------------------------ */

typedef struct {
    int S, p;
    double X[ORC_MAXS * ORC_MAXP];      /* S x p row-major */
    double hat[ORC_MAXS * ORC_MAXS];    /* X (X'X)^-1 X' */
    int linear_mu;                      /* #distinct design rows == p */
    int cell[ORC_MAXS];                 /* design cell index of each sample */
    int ncell;
    int cell_size[ORC_MAXS];
} design_t;

static void design_init(design_t* d, int S, int p, const double* X)
{
    d->S = S; d->p = p;
    memcpy(d->X, X, sizeof(double) * S * p);
    double xtx[ORC_MAXP * ORC_MAXP], inv[ORC_MAXP * ORC_MAXP], ones[ORC_MAXS] = {0};
    for (int j = 0; j < S; j++) ones[j] = 1;
    xtwx(X, ones, S, p, xtx);
    det_inv(xtx, p, inv);
    for (int a = 0; a < S; a++)
        for (int b = 0; b < S; b++) {
            double s = 0;
            for (int u = 0; u < p; u++)
                for (int v = 0; v < p; v++) s += X[a * p + u] * inv[u * p + v] * X[b * p + v];
            d->hat[a * S + b] = s;
        }
    d->ncell = 0;
    for (int j = 0; j < S; j++) {
        int found = -1;
        for (int k = 0; k < j && found < 0; k++) {
            int same = 1;
            for (int u = 0; u < p; u++) if (X[j * p + u] != X[k * p + u]) same = 0;
            if (same) found = d->cell[k];
        }
        if (found < 0) { found = d->ncell++; d->cell_size[found] = 0; }
        d->cell[j] = found;
        d->cell_size[found]++;
    }
    d->linear_mu = (d->ncell == p);
}

typedef struct { int64_t lp_evals, dlp_evals, irls_iters, disp_iters; } orc_counters;

/* Arithmetic of the posterior.  The default is plain double, like DESeq2.cpp.  -DORC_LD evaluates the same
 * expressions in long double (x87 80-bit: lgammal, logl, expl) and rounds once at the end: a variant used ONLY by
 * scripts/oracle_flip_evidence.py to show which rows' line-search decisions depend on the rounding of the
 * reference's own double arithmetic. */
#ifdef ORC_LD
typedef long double orc_real;
#define ORC_LGAMMA lgammal
#define ORC_LOG logl
#define ORC_EXP expl
#else
typedef double orc_real;
#define ORC_LGAMMA lgamma
#define ORC_LOG log
#define ORC_EXP exp
#endif

/* DESeq2.cpp log_posterior.  noise_out (may be NULL) receives 2^-53 x the sum of the magnitudes of the terms that
 * are added up: the size of one rounding error of the value in double arithmetic. */
static double log_posterior_n(double log_alpha, const double* y, const double* mu, const design_t* d,
                              double prior_mean, double prior_sigmasq, int use_prior, int use_cr, double* noise_out)
{
    int S = d->S, p = d->p;
    orc_real alpha = ORC_EXP((orc_real)log_alpha);
    double w[ORC_MAXS];
    for (int j = 0; j < S; j++) w[j] = (double)(1.0 / (1.0 / (orc_real)mu[j] + alpha));
    orc_real cr = 0;
    if (use_cr) {
        double B[ORC_MAXP * ORC_MAXP];
        xtwx(d->X, w, S, p, B);
        cr = -0.5 * ORC_LOG((orc_real)det_inv(B, p, NULL));
    }
    orc_real an1 = 1.0 / alpha;
    orc_real lgr = ORC_LGAMMA(an1);
    orc_real ll = 0;
    double mag = 0;
    for (int j = 0; j < S; j++) {
        orc_real t1 = ORC_LGAMMA(y[j] + an1), t3 = y[j] * ORC_LOG(mu[j] + an1), t4 = an1 * ORC_LOG(1.0 + mu[j] * alpha);
        ll += t1 - lgr - t3 - t4;
        mag += fabs((double)t1) + fabs((double)lgr) + fabs((double)t3) + fabs((double)t4);
    }
    orc_real pr = use_prior ? -0.5 * ((orc_real)log_alpha - prior_mean) * ((orc_real)log_alpha - prior_mean) / prior_sigmasq : 0.0;
    if (noise_out) *noise_out = 0x1p-53 * (mag + fabs((double)cr) + fabs((double)pr));
    return (double)(ll + pr + cr);
}

static double log_posterior(double log_alpha, const double* y, const double* mu, const design_t* d,
                            double prior_mean, double prior_sigmasq, int use_prior, int use_cr)
{
    return log_posterior_n(log_alpha, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr, NULL);
}

/* DESeq2.cpp dlog_posterior */
static double dlog_posterior(double log_alpha, const double* y, const double* mu, const design_t* d,
                             double prior_mean, double prior_sigmasq, int use_prior, int use_cr)
{
    int S = d->S, p = d->p;
    double alpha = exp(log_alpha);
    double w[ORC_MAXS], dw[ORC_MAXS];
    for (int j = 0; j < S; j++) {
        double t = 1.0 / mu[j] + alpha;
        w[j] = 1.0 / t;
        dw[j] = -1.0 / (t * t);
    }
    double cr = 0;
    if (use_cr) {
        double B[ORC_MAXP * ORC_MAXP], dB[ORC_MAXP * ORC_MAXP], Bi[ORC_MAXP * ORC_MAXP];
        xtwx(d->X, w, S, p, B);
        xtwx(d->X, dw, S, p, dB);
        double detb = det_inv(B, p, Bi);
        double tr = 0;
        for (int a = 0; a < p; a++) for (int b = 0; b < p; b++) tr += Bi[a * p + b] * dB[b * p + a];
        double ddetb = detb * tr;
        cr = -0.5 * ddetb / detb;
    }
    double an1 = 1.0 / alpha, an2 = 1.0 / (alpha * alpha);
    double dgr = orc_digamma(an1);
    double s = 0;
    for (int j = 0; j < S; j++)
        s += dgr + log(1 + mu[j] * alpha) - mu[j] * alpha / (1.0 + mu[j] * alpha) -
             orc_digamma(y[j] + an1) + y[j] / (mu[j] + an1);
    double ll = an2 * s;
    double pr = use_prior ? -1.0 * (log_alpha - prior_mean) / prior_sigmasq : 0.0;
    return (ll + cr) * alpha + pr;
}

typedef struct { double log_alpha; int iter, iter_accept; double initial_lp, last_lp; double margin, margin_keep; } fitdisp_res;

/* DESeq2.cpp fitDisp, one row.
 * r.margin: the smallest distance of any accept / stop comparison of this search from equality, in units of the
 * rounding error of the compared log-posteriors (log_posterior_n's noise).  A search whose margin is of order 1 takes
 * a branch that double rounding decides: any other correctly rounded evaluation of the same formulas (another libm,
 * fused multiply-adds, long double) may take the other one.  The parity tests use it to separate such rows from real
 * disagreements; it does not influence the search. */
static fitdisp_res fit_disp_row(const double* y, const double* mu, const design_t* d, double log_alpha0,
                                double prior_mean, double prior_sigmasq, double min_log_alpha,
                                double kappa_0, double tol, int maxit, int use_prior, int use_cr,
                                orc_counters* cnt)
{
    const double epsilon = 1.0e-4;
    fitdisp_res r;
    double a = log_alpha0;
    double nz0 = 0, nz = 0;
    double lp = log_posterior_n(a, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr, &nz0);
    double dlp = dlog_posterior(a, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr);
    double kappa = kappa_0;
    double margin = INFINITY;
    r.initial_lp = lp; r.iter = 0; r.iter_accept = 0;
    cnt->lp_evals++; cnt->dlp_evals++;
    for (int t = 0; t < maxit; t++) {
        r.iter++;
        double a_propose = a + kappa * dlp;
        if (a_propose < -30.0) kappa = (-30.0 - a) / dlp;
        if (a_propose > 10.0) kappa = (10.0 - a) / dlp;
        double theta_kappa = -1.0 * log_posterior_n(a + kappa * dlp, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr, &nz);
        double theta_hat_kappa = -1.0 * lp - kappa * epsilon * dlp * dlp;
        cnt->lp_evals++;
        {
            /* a proposal that no longer moves a (kappa halved away) is rejected by exact arithmetic, not by noise */
            double u = fmax(nz, nz0);
            if (a + kappa * dlp != a) margin = fmin(margin, fabs(theta_hat_kappa - theta_kappa) / u);
        }
        if (theta_kappa <= theta_hat_kappa) {
            r.iter_accept++;
            a = a + kappa * dlp;
            double lpnew = log_posterior(a, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr);
            cnt->lp_evals++;
            double change = lpnew - lp;
            margin = fmin(margin, fabs(change - tol) / fmax(nz, nz0));
            if (change < tol) { lp = lpnew; break; }
            if (a < min_log_alpha) break;
            lp = lpnew;
            nz0 = nz;
            dlp = dlog_posterior(a, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr);
            cnt->dlp_evals++;
            kappa = fmin(kappa * 1.1, kappa_0);
            if (r.iter_accept % 5 == 0) kappa = kappa / 2.0;
        } else {
            kappa = kappa / 2.0;
        }
    }
    r.last_lp = lp;
    r.log_alpha = a;
    /* estimateDispersionsGeneEst keeps the start value when last_lp < initial_lp + |initial_lp| / 1e6 */
    r.margin_keep = fabs(r.last_lp - (r.initial_lp + fabs(r.initial_lp) / 1e6)) / fmax(nz, nz0);
    r.margin = margin;
    return r;
}

/* DESeq2.cpp fitDispGrid, one row.  margin_out (may be NULL): the smallest gap between the winning grid value and any
 * other grid value of the same level, in units of the larger of the two values' rounding errors -- an arg max over a
 * plateau flatter than that is decided by rounding (the far end of the grid, alpha = 1e-8, carries the rounding error
 * of lgamma(1e8) ~ 1e-6 even when the winner sits where the posterior is known to 1e-11). */
static double grid_level(const double* y, const double* mu, const design_t* d, int grid_n, double lo, double hi,
                         double prior_mean, double prior_sigmasq, int use_prior, int use_cr, orc_counters* cnt, double* margin)
{
    double v[64], nz[64];
    const double step = (hi - lo) / (grid_n - 1);
    int best = 0;
    for (int t = 0; t < grid_n; t++) {
        double a = (t == grid_n - 1) ? hi : lo + t * step;
        v[t] = log_posterior_n(a, y, mu, d, prior_mean, prior_sigmasq, use_prior, use_cr, &nz[t]);
        cnt->lp_evals++;
        if (v[t] > v[best]) best = t;            /* first maximum wins, as which.max */
    }
    for (int t = 0; t < grid_n; t++) {
        if (t == best) continue;
        double m = (v[best] - v[t]) / fmax(nz[best], nz[t]);
        if (!(m >= *margin)) *margin = m;        /* also takes NaN values to the front */
    }
    return (best == grid_n - 1) ? hi : lo + best * step;
}

static double fit_disp_grid_row(const double* y, const double* mu, const design_t* d, int grid_n,
                                double min_la, double max_la, double prior_mean, double prior_sigmasq,
                                int use_prior, int use_cr, orc_counters* cnt, double* margin_out)
{
    double margin = INFINITY;
    if (grid_n > 64) grid_n = 64;
    double step = (max_la - min_la) / (grid_n - 1);
    double a_hat = grid_level(y, mu, d, grid_n, min_la, max_la, prior_mean, prior_sigmasq, use_prior, use_cr, cnt, &margin);
    double delta = (min_la + step) - min_la;
    double a2 = grid_level(y, mu, d, grid_n, a_hat - delta, a_hat + delta, prior_mean, prior_sigmasq, use_prior, use_cr, cnt, &margin);
    if (margin_out) *margin_out = margin;
    return a2;
}

typedef struct {
    double beta[ORC_MAXP], var[ORC_MAXP], hat[ORC_MAXS], mu_clamped[ORC_MAXS];
    int iter; double dev;
} fitbeta_res;

/* DESeq2.cpp fitBeta (useQR = TRUE), one row.  lambda is on the natural-log scale. */
static fitbeta_res fit_beta_row(const double* y, const double* nf, const design_t* d, double alpha,
                                const double* beta0, const double* lambda, double tol, int maxit,
                                double minmu, orc_counters* cnt)
{
    int S = d->S, p = d->p;
    const double large = 30.0;
    fitbeta_res r;
    double beta[ORC_MAXP], mu[ORC_MAXS], w[ORC_MAXS];
    for (int u = 0; u < p; u++) beta[u] = beta0[u];
    for (int j = 0; j < S; j++) {
        double eta = 0;
        for (int u = 0; u < p; u++) eta += d->X[j * p + u] * beta[u];
        mu[j] = fmax(nf[j] * exp(eta), minmu);
    }
    double dev = 0, dev_old = 0;
    r.iter = 0;
    for (int t = 0; t < maxit; t++) {
        r.iter++;
        cnt->irls_iters++;
        double A[(ORC_MAXS + ORC_MAXP) * ORC_MAXP], rhs[ORC_MAXS + ORC_MAXP];
        for (int j = 0; j < S; j++) {
            w[j] = mu[j] / (1.0 + alpha * mu[j]);
            double sw = sqrt(w[j]);
            for (int u = 0; u < p; u++) A[j * p + u] = d->X[j * p + u] * sw;
            double z = log(mu[j] / nf[j]) + (y[j] - mu[j]) / mu[j];
            rhs[j] = z * sw;
        }
        for (int u = 0; u < p; u++) {
            for (int v = 0; v < p; v++) A[(S + u) * p + v] = (u == v) ? sqrt(lambda[u]) : 0.0;
            rhs[S + u] = 0;
        }
        ls_householder(A, rhs, S + p, p, beta);
        int big = 0;
        for (int u = 0; u < p; u++) if (fabs(beta[u]) > large) big = 1;
        if (big) { r.iter = maxit; break; }
        for (int j = 0; j < S; j++) {
            double eta = 0;
            for (int u = 0; u < p; u++) eta += d->X[j * p + u] * beta[u];
            mu[j] = fmax(nf[j] * exp(eta), minmu);
        }
        dev = 0;
        for (int j = 0; j < S; j++) dev += -2.0 * orc_dnbinom_mu_log(y[j], 1.0 / alpha, mu[j]);
        double conv_test = fabs(dev - dev_old) / (fabs(dev) + 0.1);
        if (isnan(conv_test)) { r.iter = maxit; break; }
        if (t > 0 && conv_test < tol) break;
        dev_old = dev;
    }
    r.dev = dev;
    for (int u = 0; u < p; u++) r.beta[u] = beta[u];
    for (int j = 0; j < S; j++) { w[j] = mu[j] / (1.0 + alpha * mu[j]); r.mu_clamped[j] = mu[j]; }
    double B[ORC_MAXP * ORC_MAXP], Br[ORC_MAXP * ORC_MAXP] = {0}, Bri[ORC_MAXP * ORC_MAXP];
    xtwx(d->X, w, S, p, B);
    for (int u = 0; u < p; u++) for (int v = 0; v < p; v++) Br[u * p + v] = B[u * p + v] + ((u == v) ? lambda[u] : 0.0);
    det_inv(Br, p, Bri);
    for (int j = 0; j < S; j++) {
        double s = 0;
        for (int u = 0; u < p; u++) for (int v = 0; v < p; v++) s += d->X[j * p + u] * Bri[u * p + v] * d->X[j * p + v];
        r.hat[j] = w[j] * s;
    }
    /* sigma = (B+ridge)^-1 B (B+ridge)^-1 */
    double T[ORC_MAXP * ORC_MAXP];
    for (int u = 0; u < p; u++) for (int v = 0; v < p; v++) {
        double s = 0;
        for (int k = 0; k < p; k++) s += Bri[u * p + k] * B[k * p + v];
        T[u * p + v] = s;
    }
    for (int u = 0; u < p; u++) {
        double s = 0;
        for (int k = 0; k < p; k++) s += T[u * p + k] * Bri[k * p + u];
        r.var[u] = s;
    }
    return r;
}

/* R mean(x, trim): drop floor(n*trim) from each end after sorting */
static double trimmed_mean(double* v, int n, double trim)
{
    qsort(v, (size_t)n, sizeof(double), cmp_double);
    int lo = (int)floor(n * trim);
    long double s = 0;
    for (int i = lo; i < n - lo; i++) s += v[i];
    return (double)(s / (n - 2 * lo));
}

static int trim_bin(int n) { return n <= 3 ? 0 : (n <= 23 ? 1 : 2); }

typedef struct {
    /* per region, length n; NaN where allZero */
    double *baseMean, *baseVar, *dispGeneEst, *dispFit, *dispMAP, *dispersion;
    double *beta, *betaSE;              /* p x n, log2 scale */
    double *stat, *pvalue, *deviance, *maxCooks;
    double *mu, *H, *cooks;             /* S x n sample-major; mu = GeneEst mu (clamped) */
    int32_t *dispGeneIter, *dispIter, *betaIter;
    uint8_t *allZero, *dispOutlier, *betaConv, *flags;
    /* scalars: [0]=a0 [1]=a1 [2]=varLogDispEsts [3]=dispPriorVar [4]=trend_status(0 ok)
     *          [5]=trend outer iterations [6]=n refit GeneEst [7]=n refit MAP
     *          [8]=lp evals [9]=dlp evals [10]=irls iters [11]=sum deviance (NaN if any allZero)
     *          [12]=n nonzero rows */
    double* scalars;
} orc_out;

#define ORC_FLAG_ALLZERO 1
#define ORC_FLAG_GENE_GRID 2
#define ORC_FLAG_MAP_GRID 4
#define ORC_FLAG_BETA_NOCONV 8
#define ORC_FLAG_OUTLIER 16
#define ORC_FLAG_GENE_NOINCREASE 32

/* parametricDispersionFit: iterated Gamma(identity) glm of disp ~ 1/mean.  returns 0 ok. */
static int parametric_fit(const double* means, const double* disps, int64_t m, double* coefs_out,
                          int* outer_iters)
{
    double c0 = 0.1, c1 = 1.0;
    int iter = 0;
    uint8_t* good = (uint8_t*)malloc((size_t)m);
    *outer_iters = 0;
    while (1) {
        int64_t ngood = 0;
        for (int64_t i = 0; i < m; i++) {
            double r = disps[i] / (c0 + c1 / means[i]);
            good[i] = (r > 1e-4) && (r < 15);
            ngood += good[i];
        }
        if (ngood < 2) { free(good); return 1; }
        /* glm.fit, family Gamma(link identity), start = coefs */
        double b0 = c0, b1 = c1, ob0 = c0, ob1 = c1;
        int conv = 0;
        long double devold = 0;
        for (int64_t i = 0; i < m; i++) if (good[i]) {
            double mu = b0 + b1 / means[i];
            if (!(mu > 0) || !isfinite(mu)) { free(good); return 2; }   /* invalid start */
            devold += -2.0 * (log(disps[i] / mu) - (disps[i] - mu) / mu);
        }
        for (int it = 0; it < 25; it++) {
            long double s00 = 0, s01 = 0, s11 = 0, t0 = 0, t1 = 0;
            for (int64_t i = 0; i < m; i++) if (good[i]) {
                double x = 1.0 / means[i];
                double mu = b0 + b1 * x;
                double w = 1.0 / (mu * mu);
                s00 += w; s01 += w * x; s11 += w * x * x;
                t0 += w * disps[i]; t1 += w * x * disps[i];
            }
            long double det = s00 * s11 - s01 * s01;
            double nb0 = (double)((s11 * t0 - s01 * t1) / det);
            double nb1 = (double)((s00 * t1 - s01 * t0) / det);
            /* deviance, with glm.fit's step halving when mu leaves the valid region */
            int halv = 0;
            long double dev;
            while (1) {
                dev = 0;
                int valid = 1;
                for (int64_t i = 0; i < m; i++) if (good[i]) {
                    double mu = nb0 + nb1 / means[i];
                    if (!(mu > 0) || !isfinite(mu)) { valid = 0; break; }
                    dev += -2.0 * (log(disps[i] / mu) - (disps[i] - mu) / mu);
                }
                if (valid && isfinite((double)dev)) break;
                if (++halv > 25) { free(good); return 3; }
                nb0 = 0.5 * (nb0 + ob0); nb1 = 0.5 * (nb1 + ob1);
            }
            b0 = nb0; b1 = nb1;
            if (fabsl(dev - devold) / (fabsl(dev) + 0.1) < 1e-8) { conv = 1; break; }
            devold = dev; ob0 = b0; ob1 = b1;
        }
        double oc0 = c0, oc1 = c1;
        c0 = b0; c1 = b1;
        if (!(c0 > 0 && c1 > 0)) { free(good); return 4; }
        double l0 = log(c0 / oc0), l1 = log(c1 / oc1);
        if ((l0 * l0 + l1 * l1 < 1e-6) && conv) break;
        iter++;
        if (iter > 10) { free(good); return 5; }
    }
    *outer_iters = iter + 1;
    coefs_out[0] = c0; coefs_out[1] = c1;
    free(good);
    return 0;
}

/*
 * estimateDispersions + nbinomWaldTest for one normalisation-factor matrix.
 * K, nf: sample-major n x S.  X: S x p row-major.  prior_var_override: NaN => compute
 * (closed form needs S - p > 3; otherwise returns -2 unless overridden).
 * grid_n: fitDispGrid length (20 in current DESeq2).
 */
/* Extras of orc_deseq_ex (all optional).  trend_a0 / trend_a1 / var_log_disp: not NaN = take these instead of fitting
 * the trend / taking the MAD (the parity tests hand both sides the same global scalars so that per-region agreement can
 * be checked without the coupling through the global fits).  gene_margin / map_margin (n doubles each, may be NULL):
 * fit_disp_row's decision margin of the gene-wise and MAP searches, in rounding-error units (see fit_disp_row). */
typedef struct {
    double trend_a0, trend_a1, var_log_disp;
    double *gene_margin, *map_margin;
} orc_ext;

int orc_deseq_ex(int64_t n, int S, int p, const double* X, const int32_t* K, const double* nf,
                 double prior_var_override, int grid_n, int nthreads, const orc_ext* ext, orc_out* o);

int orc_deseq(int64_t n, int S, int p, const double* X, const int32_t* K, const double* nf,
              double prior_var_override, int grid_n, int nthreads, orc_out* o)
{
    return orc_deseq_ex(n, S, p, X, K, nf, prior_var_override, grid_n, nthreads, NULL, o);
}

int orc_deseq_ex(int64_t n, int S, int p, const double* X, const int32_t* K, const double* nf,
                 double prior_var_override, int grid_n, int nthreads, const orc_ext* ext, orc_out* o)
{
    const double minDisp = 1e-8, kappa_0 = 1.0, dispTol = 1e-6, betaTol = 1e-8, minmu = 0.5;
    const int maxit = 100;
    const double maxDisp = fmax(10.0, (double)S);
    if (S > ORC_MAXS || p > ORC_MAXP || S <= p) return -1;
    if (any_negative(n, S, K)) return -4;
    design_t d;
    design_init(&d, S, p, X);
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
    const double NA = NAN;
    int64_t nnz = 0;

    /* getBaseMeansAndVariances */
#pragma omp parallel for schedule(static) reduction(+ : nnz)
    for (int64_t i = 0; i < n; i++) {
        long double s = 0; int64_t tot = 0;
        double q[ORC_MAXS];
        for (int j = 0; j < S; j++) {
            q[j] = (double)K[(int64_t)j * n + i] / nf[(int64_t)j * n + i];
            s += q[j]; tot += K[(int64_t)j * n + i];
        }
        double m = (double)(s / S);
        long double v = 0;
        for (int j = 0; j < S; j++) v += (q[j] - m) * (q[j] - m);
        o->baseMean[i] = m;
        o->baseVar[i] = (double)(v / (S - 1));
        o->allZero[i] = (tot == 0);
        o->flags[i] = (tot == 0) ? ORC_FLAG_ALLZERO : 0;
        nnz += (tot != 0);
    }
    o->scalars[12] = (double)nnz;

    /* momentsDispEstimate: xim = mean_j 1/colMeans(nf over non-allZero rows) */
    double xim = 0;
    for (int j = 0; j < S; j++) {
        long double s = 0;
        for (int64_t i = 0; i < n; i++) if (!o->allZero[i]) s += nf[(int64_t)j * n + i];
        xim += 1.0 / (double)(s / nnz);
    }
    xim /= S;

    double lambda[ORC_MAXP];
    for (int u = 0; u < p; u++) lambda[u] = 1e-6 / (M_LN2 * M_LN2);

    int64_t c_lp = 0, c_dlp = 0, c_irls = 0, n_refit_gene = 0;

    /* estimateDispersionsGeneEst */
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : c_lp, c_dlp, c_irls, n_refit_gene)
    for (int64_t i = 0; i < n; i++) {
        orc_counters cnt = {0, 0, 0, 0};
        if (o->allZero[i]) {
            o->dispGeneEst[i] = NA; o->dispGeneIter[i] = 0;
            for (int j = 0; j < S; j++) o->mu[(int64_t)j * n + i] = NA;
            if (ext && ext->gene_margin) ext->gene_margin[i] = NA;
            continue;
        }
        double y[ORC_MAXS], nfr[ORC_MAXS], q[ORC_MAXS], mul[ORC_MAXS], mu[ORC_MAXS];
        for (int j = 0; j < S; j++) {
            y[j] = (double)K[(int64_t)j * n + i];
            nfr[j] = nf[(int64_t)j * n + i];
            q[j] = y[j] / nfr[j];
        }
        /* linearModelMu on normalised counts */
        for (int a = 0; a < S; a++) {
            double s = 0;
            for (int b = 0; b < S; b++) s += d.hat[a * S + b] * q[b];
            mul[a] = s;
        }
        double est = 0;
        for (int j = 0; j < S; j++) {
            double m = fmax(1.0, mul[j]);
            est += ((q[j] - m) * (q[j] - m) - m) / (m * m);
        }
        double rough = fmax(est / (S - p), 0.0);
        double bm = o->baseMean[i], bv = o->baseVar[i];
        double moments = (bv - xim * bm) / (bm * bm);
        double alpha_init = fmin(fmax(minDisp, fmin(rough, moments)), maxDisp);
        if (d.linear_mu) {
            for (int j = 0; j < S; j++) mu[j] = mul[j] * nfr[j];
        } else {
            double beta0[ORC_MAXP], A[ORC_MAXS * ORC_MAXP], rhs[ORC_MAXS];
            for (int j = 0; j < S; j++) {
                for (int u = 0; u < p; u++) A[j * p + u] = d.X[j * p + u];
                rhs[j] = log(q[j] + 0.1);
            }
            ls_householder(A, rhs, S, p, beta0);
            fitbeta_res fb = fit_beta_row(y, nfr, &d, alpha_init, beta0, lambda, betaTol, maxit, minmu, &cnt);
            for (int j = 0; j < S; j++) {
                double eta = 0;
                for (int u = 0; u < p; u++) eta += d.X[j * p + u] * fb.beta[u];
                mu[j] = nfr[j] * exp(eta);
            }
        }
        for (int j = 0; j < S; j++) {
            if (mu[j] < minmu) mu[j] = minmu;
            o->mu[(int64_t)j * n + i] = mu[j];
        }
        double la0 = log(alpha_init);
        fitdisp_res fr = fit_disp_row(y, mu, &d, la0, la0, 1.0, log(minDisp / 10), kappa_0, dispTol,
                                      maxit, 0, 1, &cnt);
        if (ext && ext->gene_margin) ext->gene_margin[i] = fmin(fr.margin, fr.margin_keep);
        double disp = fmin(exp(fr.log_alpha), maxDisp);
        if (fr.last_lp < fr.initial_lp + fabs(fr.initial_lp) / 1e6) {
            disp = alpha_init;
            o->flags[i] |= ORC_FLAG_GENE_NOINCREASE;
        }
        int conv = (fr.iter < maxit) && !(fr.iter == 1);
        if (!conv && disp > minDisp * 10) {
            double gmargin = INFINITY;
            double la = fit_disp_grid_row(y, mu, &d, grid_n, log(1e-8), log(maxDisp), 0.0, 1.0, 0, 1, &cnt, &gmargin);
            if (ext && ext->gene_margin) ext->gene_margin[i] = fmin(ext->gene_margin[i], gmargin);
            disp = exp(la);
            o->flags[i] |= ORC_FLAG_GENE_GRID;
            n_refit_gene++;
        }
        disp = fmin(fmax(disp, minDisp), maxDisp);
        o->dispGeneEst[i] = disp;
        o->dispGeneIter[i] = fr.iter;
        c_lp += cnt.lp_evals; c_dlp += cnt.dlp_evals; c_irls += cnt.irls_iters;
    }

    /* estimateDispersionsFit (parametric) */
    int64_t m_fit = 0;
    double* means = (double*)malloc(sizeof(double) * (size_t)(nnz > 0 ? nnz : 1));
    double* disps = (double*)malloc(sizeof(double) * (size_t)(nnz > 0 ? nnz : 1));
    for (int64_t i = 0; i < n; i++)
        if (!o->allZero[i] && o->dispGeneEst[i] > 100 * minDisp) {
            means[m_fit] = o->baseMean[i]; disps[m_fit] = o->dispGeneEst[i]; m_fit++;
        }
    double coefs[2] = {NA, NA};
    int outer = 0;
    int tstat;
    if (ext && !isnan(ext->trend_a0) && !isnan(ext->trend_a1)) { coefs[0] = ext->trend_a0; coefs[1] = ext->trend_a1; tstat = 0; }
    else tstat = (m_fit == 0) ? 9 : parametric_fit(means, disps, m_fit, coefs, &outer);
    o->scalars[0] = coefs[0]; o->scalars[1] = coefs[1]; o->scalars[4] = tstat; o->scalars[5] = outer;
    if (tstat != 0) { free(means); free(disps); return -3; }   /* local-regression fallback not restated */
    int64_t m_res = 0;
    for (int64_t i = 0; i < n; i++) {
        if (o->allZero[i]) { o->dispFit[i] = NA; continue; }
        o->dispFit[i] = coefs[0] + coefs[1] / o->baseMean[i];
        if (o->dispGeneEst[i] >= 100 * minDisp) means[m_res++] = log(o->dispGeneEst[i]) - log(o->dispFit[i]);
    }
    /* mad()^2 */
    memcpy(disps, means, sizeof(double) * (size_t)m_res);
    double med = median_inplace(disps, m_res);
    for (int64_t k = 0; k < m_res; k++) disps[k] = fabs(means[k] - med);
    double mad = 1.4826 * median_inplace(disps, m_res);
    double varLogDispEsts = mad * mad;
    if (ext && !isnan(ext->var_log_disp)) varLogDispEsts = ext->var_log_disp;
    free(means); free(disps);
    o->scalars[2] = varLogDispEsts;

    /* estimateDispersionsPriorVar */
    double dispPriorVar;
    int df = S - p;
    if (!isnan(prior_var_override)) dispPriorVar = prior_var_override;
    else if (df > 3) dispPriorVar = fmax(varLogDispEsts - orc_trigamma(df / 2.0), 0.25);
    else return -2;     /* Monte-Carlo matching path (set.seed(2), rchisq, loess) not restated here */
    o->scalars[3] = dispPriorVar;

    /* estimateDispersionsMAP */
    int64_t n_refit_map = 0;
    double outlier_thr = 2.0 * sqrt(varLogDispEsts);
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : c_lp, c_dlp, n_refit_map)
    for (int64_t i = 0; i < n; i++) {
        orc_counters cnt = {0, 0, 0, 0};
        if (o->allZero[i]) {
            o->dispMAP[i] = NA; o->dispersion[i] = NA; o->dispIter[i] = 0; o->dispOutlier[i] = 0;
            if (ext && ext->map_margin) ext->map_margin[i] = NA;
            continue;
        }
        double y[ORC_MAXS], mu[ORC_MAXS];
        for (int j = 0; j < S; j++) { y[j] = (double)K[(int64_t)j * n + i]; mu[j] = o->mu[(int64_t)j * n + i]; }
        double ge = o->dispGeneEst[i], ft = o->dispFit[i];
        double init = (ge > 0.1 * ft) ? ge : ft;
        fitdisp_res fr = fit_disp_row(y, mu, &d, log(init), log(ft), dispPriorVar, log(minDisp / 10),
                                      kappa_0, dispTol, maxit, 1, 1, &cnt);
        if (ext && ext->map_margin) ext->map_margin[i] = fr.margin;
        double dmap = exp(fr.log_alpha);
        if (!(fr.iter < maxit)) {
            double gmargin = INFINITY;
            double la = fit_disp_grid_row(y, mu, &d, grid_n, log(1e-8), log(maxDisp), log(ft), dispPriorVar, 1, 1, &cnt, &gmargin);
            if (ext && ext->map_margin) ext->map_margin[i] = fmin(ext->map_margin[i], gmargin);
            dmap = exp(la);
            o->flags[i] |= ORC_FLAG_MAP_GRID;
            n_refit_map++;
        }
        dmap = fmin(fmax(dmap, minDisp), maxDisp);
        o->dispMAP[i] = dmap;
        o->dispIter[i] = fr.iter;
        int outl = log(ge) > log(ft) + outlier_thr;
        o->dispOutlier[i] = (uint8_t)outl;
        if (outl) o->flags[i] |= ORC_FLAG_OUTLIER;
        o->dispersion[i] = outl ? ge : dmap;
        c_lp += cnt.lp_evals; c_dlp += cnt.dlp_evals;
    }
    o->scalars[6] = (double)n_refit_gene; o->scalars[7] = (double)n_refit_map;

    /* nbinomWaldTest */
    int any3 = 0;
    for (int c = 0; c < d.ncell; c++) if (d.cell_size[c] >= 3) any3 = 1;
    const double log2e = 1.0 / M_LN2;   /* log2(exp(1)) */
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : c_irls)
    for (int64_t i = 0; i < n; i++) {
        orc_counters cnt = {0, 0, 0, 0};
        if (o->allZero[i]) {
            for (int u = 0; u < p; u++) { o->beta[(int64_t)u * n + i] = NA; o->betaSE[(int64_t)u * n + i] = NA; }
            o->stat[i] = NA; o->pvalue[i] = NA; o->deviance[i] = NA; o->maxCooks[i] = NA;
            o->betaIter[i] = 0; o->betaConv[i] = 0;
            for (int j = 0; j < S; j++) { o->H[(int64_t)j * n + i] = NA; o->cooks[(int64_t)j * n + i] = NA; }
            continue;
        }
        double y[ORC_MAXS], nfr[ORC_MAXS], q[ORC_MAXS], muw[ORC_MAXS], H[ORC_MAXS];
        double alpha = o->dispersion[i];
        for (int j = 0; j < S; j++) {
            y[j] = (double)K[(int64_t)j * n + i]; nfr[j] = nf[(int64_t)j * n + i]; q[j] = y[j] / nfr[j];
        }
        double b2[ORC_MAXP], se2[ORC_MAXP], loglike = 0;
        if (p == 1) {
            /* fitNbinomGLMs intercept-only shortcut */
            long double s = 0;
            for (int j = 0; j < S; j++) s += q[j];
            b2[0] = log2((double)(s / S));
            double sw = 0, w[ORC_MAXS];
            for (int j = 0; j < S; j++) {
                muw[j] = nfr[j] * exp2(b2[0]);
                loglike += orc_dnbinom_mu_log(y[j], 1.0 / alpha, muw[j]);
                w[j] = 1.0 / (1.0 / muw[j] + alpha);
                sw += w[j];
            }
            se2[0] = log2e * sqrt(1.0 / sw);
            for (int j = 0; j < S; j++) H[j] = w[j] / sw;
            o->betaIter[i] = 1; o->betaConv[i] = 1;
        } else {
            double beta0[ORC_MAXP], A[ORC_MAXS * ORC_MAXP], rhs[ORC_MAXS];
            for (int j = 0; j < S; j++) {
                for (int u = 0; u < p; u++) A[j * p + u] = d.X[j * p + u];
                rhs[j] = log(q[j] + 0.1);
            }
            ls_householder(A, rhs, S, p, beta0);
            fitbeta_res fb = fit_beta_row(y, nfr, &d, alpha, beta0, lambda, betaTol, maxit, minmu, &cnt);
            int stable = 1, varpos = 1;
            for (int u = 0; u < p; u++) {
                b2[u] = log2e * fb.beta[u];
                se2[u] = log2e * sqrt(fmax(fb.var[u], 0.0));
                if (isnan(fb.beta[u])) stable = 0;
                if (!(fb.var[u] > 0)) varpos = 0;
            }
            for (int j = 0; j < S; j++) {
                double eta = 0;
                for (int u = 0; u < p; u++) eta += d.X[j * p + u] * fb.beta[u];
                muw[j] = nfr[j] * exp(eta);
                loglike += orc_dnbinom_mu_log(y[j], 1.0 / alpha, muw[j]);
                H[j] = fb.hat[j];
            }
            o->betaIter[i] = fb.iter;
            o->betaConv[i] = (fb.iter < maxit);
            if (!(fb.iter < maxit) || !stable || !varpos) o->flags[i] |= ORC_FLAG_BETA_NOCONV;   /* R would call optim() */
        }
        for (int u = 0; u < p; u++) { o->beta[(int64_t)u * n + i] = b2[u]; o->betaSE[(int64_t)u * n + i] = se2[u]; }
        o->deviance[i] = -2.0 * loglike;
        double st = b2[p - 1] / se2[p - 1];
        o->stat[i] = st;
        o->pvalue[i] = orc_wald_pvalue(st);
        /* calculateCooksDistance / robustMethodOfMomentsDisp / recordMaxCooks */
        double v;
        if (any3) {
            v = -INFINITY;
            for (int c = 0; c < d.ncell; c++) {
                int nc = d.cell_size[c];
                if (nc < 3) continue;
                static const double trimr[3] = {1.0 / 3.0, 1.0 / 4.0, 1.0 / 8.0};
                static const double scalec[3] = {2.04, 1.86, 1.51};
                double tmp[ORC_MAXS]; int k = 0;
                for (int j = 0; j < S; j++) if (d.cell[j] == c) tmp[k++] = q[j];
                double cm = trimmed_mean(tmp, nc, trimr[trim_bin(nc)]);
                k = 0;
                for (int j = 0; j < S; j++) if (d.cell[j] == c) tmp[k++] = (q[j] - cm) * (q[j] - cm);
                double ve = scalec[trim_bin(nc)] * trimmed_mean(tmp, nc, trimr[trim_bin(nc)]);
                if (ve > v) v = ve;
            }
        } else {
            double tmp[ORC_MAXS];
            for (int j = 0; j < S; j++) tmp[j] = q[j];
            double rm = trimmed_mean(tmp, S, 1.0 / 8.0);
            for (int j = 0; j < S; j++) tmp[j] = (q[j] - rm) * (q[j] - rm);
            v = 1.51 * trimmed_mean(tmp, S, 1.0 / 8.0);
        }
        long double sq = 0;
        for (int j = 0; j < S; j++) sq += q[j];
        double mq = (double)(sq / S);
        double ar = fmax((v - mq) / (mq * mq), 0.04);
        double mc = -INFINITY;
        for (int j = 0; j < S; j++) {
            double V = muw[j] + ar * muw[j] * muw[j];
            double ck = (y[j] - muw[j]) * (y[j] - muw[j]) / V / p * H[j] / ((1 - H[j]) * (1 - H[j]));
            o->cooks[(int64_t)j * n + i] = ck;
            o->H[(int64_t)j * n + i] = H[j];
            if (d.cell_size[d.cell[j]] >= 3 && ck > mc) mc = ck;
        }
        o->maxCooks[i] = (S > p && any3) ? mc : NA;
        c_irls += cnt.irls_iters;
    }
    long double devsum = 0;
    for (int64_t i = 0; i < n; i++) devsum += o->deviance[i];
    o->scalars[8] = (double)c_lp; o->scalars[9] = (double)c_dlp; o->scalars[10] = (double)c_irls;
    o->scalars[11] = (double)devsum;
    return 0;
}

/* exported single-row probes used by the known-answer tests */
double orc_log_posterior(double log_alpha, int S, int p, const double* X, const double* y, const double* mu,
                         double prior_mean, double prior_sigmasq, int use_prior, int use_cr)
{
    design_t d; design_init(&d, S, p, X);
    return log_posterior(log_alpha, y, mu, &d, prior_mean, prior_sigmasq, use_prior, use_cr);
}

double orc_dlog_posterior(double log_alpha, int S, int p, const double* X, const double* y, const double* mu,
                          double prior_mean, double prior_sigmasq, int use_prior, int use_cr)
{
    design_t d; design_init(&d, S, p, X);
    return dlog_posterior(log_alpha, y, mu, &d, prior_mean, prior_sigmasq, use_prior, use_cr);
}

int orc_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* ------------------------------------------------------------------ */
/* per-replicate assembly (getFullRegionData1, chicdiff.R:609-702,      */
/* 820-910): N and FullMean = Bmean + Tmean for every region-universe   */
/* row from one replicate's CHiCAGO tables                              */
/* ------------------------------------------------------------------ */

/* Chicago:::.distFun with the parameters of .chicEstimateDistFun (chicdiff.R:559-569):
 * p = cubicFit[4], obs.min, obs.max, head.coef[2], tail.coef[2] */
double orc_dist_fun(double d, const double* p)
{
    double l = log(d), out;
    if (l > p[5]) out = p[8] + l * p[9];
    else if (l < p[4]) out = p[6] + l * p[7];
    else out = p[0] + p[1] * l + p[2] * (l * l) + p[3] * (l * l * l);
    return exp(out);
}

/*
 * Tables are indexed by fragID - frag_id0 (length F).  s_j NaN = NA / bait absent from this replicate
 * (chicdiff.R:659-662, Bmean := NA :702); tblb/tlb -1 = NA; s_i NaN -> 1 (:672); tmean[n_tblb][n_tlb]
 * NaN = combination never seen (:680-683); tlb NA with tblb known -> min Tmean of that tblb (:689-692).
 * distSign is recomputed for every row (:640-654): round(((oe.start+oe.end)-(bait.start+bait.end))/2),
 * half to even, NA across chromosomes (then Bmean = 0, Chicago:::.estimateBMean).
 * Counts: CSR by bait over (otherEndID, N) rows sorted by otherEndID; missing -> 0 (:853).
 * Outputs (any may be NULL): N, FullMean, distSign (NaN = NA), Bmean, Tmean -- one value per row.
 */
int orc_assemble_sample(int64_t R, const int32_t* row_bait, const int32_t* row_oe,
                        int64_t F, int32_t frag_id0, const int32_t* frag_chr, const int32_t* frag_start,
                        const int32_t* frag_end, const double* s_j, const int32_t* tblb, const double* s_i,
                        const int32_t* tlb, int n_tblb, int n_tlb, const double* tmean, const double* distfun,
                        const int64_t* cnt_off, const int32_t* cnt_oe, const int32_t* cnt_N,
                        int32_t* N_out, double* FM_out, double* dist_out, double* Bmean_out, double* Tmean_out)
{
    double* tmin = (double*)malloc(sizeof(double) * (size_t)(n_tblb > 0 ? n_tblb : 1));
    for (int a = 0; a < n_tblb; a++) {
        double m = NAN;
        for (int b = 0; b < n_tlb; b++) {
            double v = tmean[a * n_tlb + b];
            if (!isnan(v) && (isnan(m) || v < m)) m = v;
        }
        tmin[a] = m;
    }
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (int64_t r = 0; r < R; r++) {
        int64_t b = (int64_t)row_bait[r] - frag_id0, o = (int64_t)row_oe[r] - frag_id0;
        if (b < 0 || b >= F || o < 0 || o >= F) { bad |= 1; continue; }
        double d = NAN;
        if (frag_chr[b] == frag_chr[o])
            d = rint((((double)frag_start[o] + (double)frag_end[o]) - ((double)frag_start[b] + (double)frag_end[b])) / 2.0);
        double sj = s_j[b];
        double si = isnan(s_i[o]) ? 1.0 : s_i[o];
        int tb = tblb[b], tl = tlb[o];
        double tm = NAN;
        if (tb >= 0) tm = (tl >= 0) ? tmean[tb * n_tlb + tl] : tmin[tb];
        double bm;
        if (isnan(d)) bm = 0.0; else bm = sj * si * orc_dist_fun(fabs(d), distfun);
        if (isnan(sj)) bm = NAN;
        /* count lookup */
        int64_t lo = cnt_off[b], hi = cnt_off[b + 1];
        int32_t key = row_oe[r], cnt = 0;
        while (lo < hi) {
            int64_t mid = (lo + hi) / 2;
            if (cnt_oe[mid] < key) lo = mid + 1; else hi = mid;
        }
        if (lo < cnt_off[b + 1] && cnt_oe[lo] == key) cnt = cnt_N[lo];
        if (N_out) N_out[r] = cnt;
        if (FM_out) FM_out[r] = bm + tm;
        if (dist_out) dist_out[r] = d;
        if (Bmean_out) Bmean_out[r] = bm;
        if (Tmean_out) Tmean_out[r] = tm;
    }
    free(tmin);
    return bad ? -1 : 0;
}
