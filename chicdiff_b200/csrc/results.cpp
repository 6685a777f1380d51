// results.cpp -- cd_results_adjust: the part of DESeq2 results() that Chicdiff's output table needs
// (chicdiff.R:1721,1730,1739): Cook's-distance cutoff qf(.99, p, m - p) with the two-level-factor
// heuristic, independent filtering on baseMean (50 quantile cut-offs, BH at each, lowess(f = 1/5)
// threshold rule, alpha = 0.1) and the Benjamini-Hochberg adjusted p-values.
// Global over all regions and O(n log n): host code, outside the five timed stages.
#include "../../include/chicdiff_b200.h"
#include "results_host.h"
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <numeric>
#include <vector>

namespace {

double betacf(double a, double b, double x)
{
    const double tiny = 1e-300;
    const double qab = a + b, qap = a + 1, qam = a - 1;
    double c = 1, d = 1 - qab * x / qap;
    if (std::fabs(d) < tiny) d = tiny;
    d = 1 / d;
    double h = d;
    for (int m = 1; m <= 500; m++) {
        const int m2 = 2 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1 + aa * d; if (std::fabs(d) < tiny) d = tiny;
        c = 1 + aa / c; if (std::fabs(c) < tiny) c = tiny;
        d = 1 / d; h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1 + aa * d; if (std::fabs(d) < tiny) d = tiny;
        c = 1 + aa / c; if (std::fabs(c) < tiny) c = tiny;
        d = 1 / d;
        const double del = d * c;
        h *= del;
        if (std::fabs(del - 1) < 1e-16) break;
    }
    return h;
}

double pbeta(double x, double a, double b)
{
    if (x <= 0) return 0;
    if (x >= 1) return 1;
    const double bt = std::exp(std::lgamma(a + b) - std::lgamma(a) - std::lgamma(b) + a * std::log(x) + b * std::log1p(-x));
    if (x < (a + 1) / (a + b + 2)) return bt * betacf(a, b, x) / a;
    return 1 - bt * betacf(b, a, 1 - x) / b;
}

double qf(double prob, double df1, double df2)
{
    double lo = 0, hi = 1;
    for (int it = 0; it < 200; it++) {
        const double mid = 0.5 * (lo + hi);
        if (pbeta(mid, 0.5 * df1, 0.5 * df2) < prob) lo = mid; else hi = mid;
    }
    const double x = 0.5 * (lo + hi);
    return (df2 * x) / (df1 * (1 - x));
}

// stats::lowess (Cleveland), x ascending
void lowess(const std::vector<double>& x, const std::vector<double>& y, double f, int nsteps, double delta,
            std::vector<double>& ys)
{
    const int n = (int)x.size();
    ys.assign(n, 0.0);
    if (n < 2) { if (n == 1) ys[0] = y[0]; return; }
    std::vector<double> rw(n, 1.0), res(n, 0.0), w(n, 0.0);
    const int ns = std::max(2, std::min(n, (int)(f * n + 1e-7)));
    auto lowest = [&](double xs, int nleft, int nright, bool userw, double& out) -> bool {
        const double range = x[n - 1] - x[0];
        const double h = std::max(xs - x[nleft], x[nright] - xs);
        const double h9 = .999 * h, h1 = .001 * h;
        double a = 0.0;
        int j = nleft;
        while (j < n) {
            w[j] = 0.0;
            const double r = std::fabs(x[j] - xs);
            if (r <= h9) {
                if (r <= h1) w[j] = 1.0;
                else { const double q = r / h; const double t = 1.0 - q * q * q; w[j] = t * t * t; }
                if (userw) w[j] *= rw[j];
                a += w[j];
            } else if (x[j] > xs) break;
            j++;
        }
        const int nrt = j - 1;
        if (a <= 0.0) return false;
        for (j = nleft; j <= nrt; j++) w[j] /= a;
        if (h > 0.0) {
            a = 0.0;
            for (j = nleft; j <= nrt; j++) a += w[j] * x[j];
            double b = xs - a, c = 0.0;
            for (j = nleft; j <= nrt; j++) c += w[j] * (x[j] - a) * (x[j] - a);
            if (std::sqrt(c) > .001 * range) {
                b /= c;
                for (j = nleft; j <= nrt; j++) w[j] *= (b * (x[j] - a) + 1.0);
            }
        }
        out = 0.0;
        for (j = nleft; j <= nrt; j++) out += w[j] * y[j];
        return true;
    };
    for (int iter = 0; iter <= nsteps; iter++) {
        int nleft = 0, nright = ns - 1, last = -1, i = 0;
        while (true) {
            if (nright < n - 1) {
                const double d1 = x[i] - x[nleft], d2 = x[nright + 1] - x[i];
                if (d1 > d2) { nleft++; nright++; continue; }
            }
            double v;
            if (lowest(x[i], nleft, nright, iter > 0, v)) ys[i] = v; else ys[i] = y[i];
            if (last < i - 1) {
                const double denom = x[i] - x[last];
                for (int j = last + 1; j < i; j++) {
                    const double alpha = (x[j] - x[last]) / denom;
                    ys[j] = alpha * ys[i] + (1.0 - alpha) * ys[last];
                }
            }
            last = i;
            const double cut = x[last] + delta;
            for (i = last + 1; i < n; i++) {
                if (x[i] > cut) break;
                if (x[i] == x[last]) { ys[i] = ys[last]; last = i; }
            }
            i = std::max(last + 1, i - 1);
            if (last >= n - 1) break;
        }
        for (int k = 0; k < n; k++) res[k] = y[k] - ys[k];
        double sc = 0.0;
        for (int k = 0; k < n; k++) sc += std::fabs(res[k]);
        sc /= n;
        if (iter >= nsteps) break;
        for (int k = 0; k < n; k++) rw[k] = std::fabs(res[k]);
        std::vector<double> srt(rw);
        std::sort(srt.begin(), srt.end());
        const int m1 = n / 2;
        double cmad;
        if (n % 2 == 0) { const int m2 = n - m1 - 1; cmad = 3.0 * (srt[m1] + srt[m2]); }
        else cmad = 6.0 * srt[m1];
        if (cmad < 1e-7 * sc) break;
        const double c9 = .999 * cmad, c1 = .001 * cmad;
        for (int k = 0; k < n; k++) {
            const double r = std::fabs(res[k]);
            if (r <= c1) rw[k] = 1.0;
            else if (r <= c9) { const double q = r / cmad; rw[k] = (1.0 - q * q) * (1.0 - q * q); }
            else rw[k] = 0.0;
        }
    }
}

}  // namespace

namespace cd {

double res_qf(double prob, double df1, double df2) { return qf(prob, df1, df2); }

// genefilter's rule inside results(): lowess(theta, numRej, f = 1/5); the first cut-off whose rejection count
// exceeds max(fit) - RMS residual over the cut-offs with rejections; cut-off 0 when no count exceeds 10
int res_pick_cutoff(const double* theta_p, const double* numRej_p, int nt)
{
    const std::vector<double> theta(theta_p, theta_p + nt), numRej(numRej_p, numRej_p + nt);
    std::vector<double> lo_fit;
    lowess(theta, numRej, 1.0 / 5.0, 3, 0.01 * (theta[nt - 1] - theta[0]), lo_fit);
    int j = 0;
    const double maxRej = *std::max_element(numRej.begin(), numRej.end());
    if (maxRej > 10.0) {
        double ss = 0.0; int cnt = 0;
        for (int k = 0; k < nt; k++) if (numRej[k] > 0) { const double r = numRej[k] - lo_fit[k]; ss += r * r; cnt++; }
        const double thresh = *std::max_element(lo_fit.begin(), lo_fit.end()) - std::sqrt(ss / cnt);
        for (int k = 0; k < nt; k++) if (numRej[k] > thresh) { j = k; break; }
    }
    return j;
}

}  // namespace cd

extern "C" int cd_results_adjust(int64_t n, int S, int p, const double* baseMean, const double* maxCooks,
                                 const uint8_t* flags, double* pvalue, double* padj, double* scalars_out)
{
    if (n < 0 || S <= p || p < 1 || (n > 0 && (!baseMean || !pvalue || !padj))) return CD_EINVAL;
    const double alpha = 0.1;
    const double cutoff = qf(0.99, (double)p, (double)(S - p));
    if (maxCooks) {
        for (int64_t i = 0; i < n; i++) {
            if (maxCooks[i] > cutoff) {                               // NaN compares false
                const bool keep = flags && (flags[i] & CD_FLAG_COOKS_KEEP) && p == 2;
                if (!keep) pvalue[i] = NAN;
            }
        }
    }
    // independent filtering
    int64_t nzero = 0;
    for (int64_t i = 0; i < n; i++) nzero += (baseMean[i] == 0.0);
    const double lower = n > 0 ? cd::res_mean_of_count((uint64_t)nzero, (uint64_t)n) : 0.0;
    const double upper = lower < .95 ? .95 : 1.0;
    const int NT = 50;
    std::vector<double> theta(NT), cut(NT);
    for (int k = 0; k < NT; k++) theta[k] = (k == NT - 1) ? upper : lower + k * ((upper - lower) / (NT - 1));
    std::vector<double> fs(baseMean, baseMean + n);
    std::sort(fs.begin(), fs.end());
    for (int k = 0; k < NT; k++) {
        if (n == 0) { cut[k] = NAN; continue; }
        const cd::ResQuantileIndex ix = cd::res_quantile7_index(n, theta[k]);
        double q = fs[ix.lo];
        if (ix.h > 0.0 && fs[ix.hi] != q) q = (1.0 - ix.h) * q + ix.h * fs[ix.hi];
        cut[k] = q;
    }
    // rows with a p-value, ascending by p (stable, so ties keep row order like R's order()); the sorted records
    // carry baseMean so that the 50 counting passes below stream through memory
    struct Rec { double p, bm; int64_t i; };
    std::vector<Rec> ord;
    ord.reserve((size_t)n);
    for (int64_t i = 0; i < n; i++) if (!std::isnan(pvalue[i])) ord.push_back(Rec{pvalue[i], baseMean[i], i});
    std::stable_sort(ord.begin(), ord.end(), [](const Rec& a, const Rec& b) { return a.p < b.p; });
    std::vector<double> numRej(NT, 0.0);
    for (int k = 0; k < NT; k++) {
        const double ck = cut[k];
        int64_t m = 0;
        for (const Rec& r : ord) m += (r.bm >= ck);
        int64_t rank = 0, best = 0;
        for (const Rec& r : ord) {
            if (!(r.bm >= ck)) continue;
            rank++;
            if ((double)m / (double)rank * r.p < alpha) best = rank;
        }
        numRej[k] = (double)best;
    }
    const int j = cd::res_pick_cutoff(theta.data(), numRej.data(), NT);
    // BH at the chosen cut-off
    for (int64_t i = 0; i < n; i++) padj[i] = NAN;
    int64_t m = 0;
    for (const Rec& r : ord) m += (r.bm >= cut[j]);
    double running = INFINITY;
    int64_t rank = m;
    for (auto it = ord.rbegin(); it != ord.rend(); ++it) {
        if (!(it->bm >= cut[j])) continue;
        const double v = (double)m / (double)rank * it->p;
        running = std::min(running, v);
        padj[it->i] = std::min(1.0, running);
        rank--;
    }
    if (scalars_out) {
        scalars_out[0] = cutoff; scalars_out[1] = cut[j]; scalars_out[2] = theta[j]; scalars_out[3] = (double)(j + 1);
    }
    return CD_OK;
}

// IHWcorrection(), "apply to test data" (chicdiff.R:2038-2049): stratum of every region by cut(log|avDist|, breaks)
// with breaks half-way between neighbouring strata of the lookup learned on the control set, weight =
// avWeights[stratum] / mean(avWeights over the rows), weighted p-value, BH.
namespace cd {

bool ihw_breaks(int ngroups, const double* minLogDist, const double* maxLogDist, std::vector<double>& breaks)
{
    breaks.assign((size_t)ngroups + 1, 0.0);
    for (int k = 0; k <= ngroups; k++) {
        const double a = k < ngroups ? minLogDist[k] : INFINITY;
        const double b = k > 0 ? maxLogDist[k - 1] : 0.0;
        breaks[(size_t)k] = (a + b) / 2;
        if (std::isnan(breaks[(size_t)k])) return false;
    }
    std::sort(breaks.begin(), breaks.end());
    for (int k = 1; k <= ngroups; k++) if (breaks[(size_t)k] == breaks[(size_t)k - 1]) return false;   // 'breaks' are not unique
    return true;
}

double ihw_mean_weight(int64_t n, int ngroups, const unsigned long long* per_group, const double* avWeights)
{
    if (n <= 0 || per_group[0] != 0) return NAN;
    long double sum = 0.0L;
    for (int g = 1; g <= ngroups; g++)
        for (unsigned long long c = 0; c < per_group[(size_t)g]; c++) sum += (long double)avWeights[g - 1];
    long double m = sum / (long double)n, t = 0.0L;
    for (int g = 1; g <= ngroups; g++)
        for (unsigned long long c = 0; c < per_group[(size_t)g]; c++) t += ((long double)avWeights[g - 1] - m);
    return (double)(m + t / (long double)n);
}

}  // namespace cd

extern "C" int cd_ihw_apply(int64_t n, const double* avDist, const double* pvalue, int ngroups, const double* minLogDist,
                            const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                            double* weighted_pvalue_out, double* weighted_padj_out)
{
    if (n < 0 || ngroups < 1 || !minLogDist || !maxLogDist || !avWeights || (n > 0 && (!avDist || !pvalue))) return CD_EINVAL;
    std::vector<double> breaks;
    if (!cd::ihw_breaks(ngroups, minLogDist, maxLogDist, breaks)) return CD_EINVAL;
    std::vector<int32_t> group((size_t)n);
    std::vector<unsigned long long> per_group((size_t)ngroups + 1, 0);    // [0] = NA
    for (int64_t i = 0; i < n; i++) {
        const double x = std::log(std::fabs(avDist[i]));
        int32_t g = INT32_MIN;                                            // NA_integer_
        if (!std::isnan(x) && x > breaks[0] && x <= breaks[(size_t)ngroups]) {
            // right-closed intervals (breaks[g-1], breaks[g]]
            const auto it = std::lower_bound(breaks.begin(), breaks.end(), x);
            g = (int32_t)(it - breaks.begin());
        }
        group[(size_t)i] = g;
        per_group[g == INT32_MIN ? 0 : (size_t)g]++;
    }
    const double meanw = cd::ihw_mean_weight(n, ngroups, per_group.data(), avWeights);
    std::vector<double> wp((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        const int32_t g = group[(size_t)i];
        const double w = (g == INT32_MIN) ? NAN : avWeights[g - 1] / meanw;
        wp[(size_t)i] = pvalue[i] / w;
        if (group_out) group_out[i] = g;
        if (weight_out) weight_out[i] = w;
        if (weighted_pvalue_out) weighted_pvalue_out[i] = wp[(size_t)i];
    }
    if (weighted_padj_out) {
        // p.adjust(method = "BH") over the non-NA entries
        std::vector<int64_t> ord;
        ord.reserve((size_t)n);
        for (int64_t i = 0; i < n; i++) { weighted_padj_out[i] = NAN; if (!std::isnan(wp[(size_t)i])) ord.push_back(i); }
        std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return wp[(size_t)a] < wp[(size_t)b]; });
        // p.adjust returns p unchanged when at most one is not NA (`if (n <= 1) return(p0)`): a single weighted p-value
        // above 1 stays above 1
        const int64_t m = (int64_t)ord.size();
        double running = INFINITY;
        for (int64_t r = m; r >= 1; r--) {
            const int64_t i = ord[(size_t)r - 1];
            running = std::min(running, (double)m / (double)r * wp[(size_t)i]);
            weighted_padj_out[i] = m > 1 ? std::min(1.0, running) : running;
        }
    }
    return CD_OK;
}
