// results_host.h -- host pieces of results() shared by cd_results_adjust (results.cpp) and the device-resident
// variant orchestrated in context.cu
#pragma once
#include <cmath>
#include <cstdint>
#include <vector>

#ifdef __CUDACC__
#define CD_HD __host__ __device__
#else
#define CD_HD
#endif

namespace cd {

// lowerQuantile <- mean(filter == 0) in DESeq2's pvalueAdjustment.  R's mean() of a logical sums it in long double and
// returns (double)(s / n) (summary.c): the quotient rounded to a 64-bit significand (x87 extended precision, as in R on
// x86-64), then to double.  That double rounding differs from nzero / n in double for some counts (nzero = 115,
// n = 2051).  Emulated here with integers so that the host and the device give the same bits; 0 <= nzero <= n.
CD_HD inline double res_mean_of_count(uint64_t a, uint64_t b)
{
    if (a == 0 || b == 0) return b == 0 ? NAN : 0.0;
    if (a >= b) return 1.0;
    uint64_t r = a;
    int e = 0;
    while (r < b) { r <<= 1; e--; }                     // a / b = (r / b) * 2^e with 1 <= r / b < 2
    uint64_t q = 0;
    for (int i = 0; i < 64; i++) {                      // 64 significant bits of r / b
        const bool bit = r >= b;
        if (bit) r -= b;
        q = (q << 1) | (bit ? 1u : 0u);
        r <<= 1;
    }
    const bool guard = r >= b;
    if (guard) r -= b;
    if (guard && (r != 0 || (q & 1))) {                 // round to nearest even at 64 bits
        if (++q == 0) { q = 1ull << 63; e++; }
    }
    uint64_t m = q >> 11;                                // then at 53 bits
    const uint64_t low = q & 0x7ffu;
    if (low > 0x400u || (low == 0x400u && (m & 1))) {
        if (++m == (1ull << 53)) { m = 1ull << 52; e++; }
    }
    return ldexp((double)m, e - 52);
}

// The index of quantile(x, theta, type = 7) as quantile.default computes it: index <- 1 + (n - 1) * probs (1-based),
// lo <- floor(index), hi <- ceiling(index), h <- index - lo; the interpolation (1 - h) * x[lo] + h * x[hi] applies where
// index > lo and x[hi] != x[lo].  lo and hi are returned 0-based.  A 0-based index (n - 1) * theta skips the rounding of
// 1 + (n - 1) * theta, which gives another h in the last bits and can move the cut from a tied baseMean to the next
// double above it (scripts/quantile_index_search.py).  n >= 1.
struct ResQuantileIndex { int64_t lo, hi; double h; };
CD_HD inline ResQuantileIndex res_quantile7_index(int64_t n, double theta)
{
#ifdef __CUDA_ARCH__
    const double index = __dadd_rn(1.0, __dmul_rn((double)(n - 1), theta));
#else
    const double index = 1.0 + (double)(n - 1) * theta;
#endif
    const double lo = floor(index), hi = ceil(index);
    return ResQuantileIndex{(int64_t)lo - 1, (int64_t)hi - 1, index - lo};
}

double res_qf(double prob, double df1, double df2);                          // stats::qf by bisection on pbeta
int res_pick_cutoff(const double* theta, const double* numRej, int nt);     // lowess + threshold rule -> index
// IHWcorrection's breaks <- (c(minLogDist, Inf) + c(0, maxLogDist)) / 2 (chicdiff.R:2039), sorted as cut() sorts them;
// false when one is NaN or two coincide ('breaks' are not unique)
bool ihw_breaks(int ngroups, const double* minLogDist, const double* maxLogDist, std::vector<double>& breaks);
// mean(out$avWeights) over the n rows from the per-group row counts (per_group[0] = rows without a group, which poison
// it), as R's two-pass long-double mean over the rows ordered by stratum computes it
double ihw_mean_weight(int64_t n, int ngroups, const unsigned long long* per_group, const double* avWeights);

}  // namespace cd
