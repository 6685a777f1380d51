"""results() and the IHW weight application at their edges, against a restatement of R's rules written here.

The statistics a user reads come out of two steps after the Wald test: DESeq2's results() (Cook's cutoff, independent
filtering, BH; device: cd_results_device / cd_results_resident, host: cd_results_adjust) and the "apply to test data"
block of IHWcorrection() (device: cd_ihw_apply_device, host: cd_ihw_apply).  Each case below runs the host routine
against the reference (no GPU needed) and, marked gpu, the device routine against the host routine bit for bit and
against the reference.

The reference restates, from the R and Bioconductor sources, and shares no code with oracle/ or csrc/:
  * stats::quantile.default, type 7 branch:
        index <- 1 + max(n - 1, 0) * probs; lo <- floor(index); hi <- ceiling(index)
        qs <- x[lo]; i <- which(index > lo & x[hi] != qs); h <- (index - lo)[i]; qs[i] <- (1 - h) * qs[i] + h * x[hi[i]]
    (no fuzz: the 4 * .Machine$double.eps fuzz belongs to types 4 to 9)
  * base::seq.default(from, to, length.out = 50): c(from, from + seq_len(48) * ((to - from) / 49), to)
  * base::mean of a logical (summary.c): long-double sum, (double)(s / n); of doubles: long-double sum, s /= n, and if
    finite a second pass s += sum(x - s) / n
  * stats::p.adjust(p, "BH"): n = length(p) is evaluated after the NAs are dropped, `if (n <= 1) return(p0)`, else
    i <- lp:1; o <- order(p, decreasing = TRUE); pmin(1, cummin(n / i * p[o]))[order(o)]
  * genefilter::filtered_p: cutoffs <- quantile(filter, theta); use <- filter >= cutoffs[i]; p.adjust(test[use], method)
  * DESeq2:::pvalueAdjustment: lowerQuantile <- mean(filter == 0); upperQuantile <- if (lowerQuantile < .95) .95 else 1;
    theta <- seq(lowerQuantile, upperQuantile, length = 50); numRej <- colSums(filtPadj < alpha, na.rm = TRUE);
    lo.fit <- lowess(numRej ~ theta, f = 1/5); if (max(numRej) <= 10) j <- 1 else { residual <- numRej[numRej > 0] -
    lo.fit$y[numRej > 0]; thresh <- max(lo.fit$y) - sqrt(mean(residual^2)); j <- if (any(numRej > thresh))
    which(numRej > thresh)[1] else 1 }  (lowess itself is taken from the oracle: the comparisons here are of counts)
  * DESeq2::results, Cook's filter: cooksOutlier <- maxCooks > qf(.99, p, m - p) (NA is never an outlier); the
    heuristic that keeps a row with three or more counts above the outlier's applies only to a single two-level factor
    (p == 2; the per-row part is CD_FLAG_COOKS_KEEP)
  * IHWcorrection (chicdiff.R:2038-2049): breaks <- (c(minLogDist, Inf) + c(0, maxLogDist)) / 2; cut(log(abs(avDist)),
    breaks) with right-closed intervals and NA outside (.bincode); weight <- avWeights / mean(avWeights) over the rows;
    weighted_pvalue <- pvalue / weight; weighted_padj <- p.adjust(weighted_pvalue, "BH")
"""
import math

import numpy as np
import pytest

from chicdiff_b200 import engine

ALPHA = 0.1
NT = 50


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------

def r_mean_logical(mask):
    return float(np.longdouble(np.count_nonzero(mask)) / np.longdouble(len(mask)))


def r_mean(x):
    x = np.asarray(x, dtype=np.float64)
    if np.isnan(x).any():
        return float("nan")
    s = x.astype(np.longdouble).sum() / np.longdouble(len(x))
    if np.isfinite(np.float64(s)):
        s = s + (x.astype(np.longdouble) - s).sum() / np.longdouble(len(x))
    return float(s)


def r_seq50(lower, upper):
    if lower == upper:
        return np.full(NT, lower)
    by = (upper - lower) / (NT - 1)
    return np.concatenate([[lower], lower + np.arange(1, NT - 1, dtype=np.float64) * by, [upper]])


def r_quantile7(x, probs):
    xs = np.sort(np.asarray(x, dtype=np.float64))
    n = len(xs)
    out = np.empty(len(probs))
    for k, pr in enumerate(probs):
        index = 1.0 + max(n - 1, 0) * float(pr)
        lo, hi = math.floor(index), math.ceil(index)
        qs = xs[lo - 1]
        if index > lo and xs[hi - 1] != qs:
            h = index - lo
            qs = (1.0 - h) * qs + h * xs[hi - 1]
        out[k] = qs
    return out


def _bh_ascending(ps):
    """p.adjust(., "BH") of non-NA p-values given in ascending order; result in the same order"""
    n = len(ps)
    if n <= 1:
        return ps.copy()
    i = np.arange(1, n + 1)
    v = n / i * ps
    return np.minimum(1.0, np.minimum.accumulate(v[::-1])[::-1])


def r_p_adjust_bh(p):
    p = np.asarray(p, dtype=np.float64)
    out = p.copy()
    ok = np.flatnonzero(~np.isnan(p))
    o = ok[np.argsort(p[ok], kind="stable")]
    out[o] = _bh_ascending(p[o])
    return out


def r_results(baseMean, maxCooks, flags, pvalue, p, cutoff):
    """results(): Cook's filter with the given cutoff (the library's qf(.99, p, m - p), checked against scipy on its own),
    then pvalueAdjustment.  Returns pvalue, padj, j (0-based), theta, cut (50 each), numRej."""
    from oracle import oracle as O
    bm = np.asarray(baseMean, dtype=np.float64)
    pv = np.array(pvalue, dtype=np.float64, copy=True)
    n = len(bm)
    if maxCooks is not None:
        with np.errstate(invalid="ignore"):
            outlier = np.asarray(maxCooks) > cutoff
        if p == 2 and flags is not None:
            outlier &= (np.asarray(flags) & engine.FLAG_COOKS_KEEP) == 0
        pv[outlier] = np.nan
    if n == 0:          # R stops here (mean(logical(0)) is NaN in an if()); the library returns nothing per row
        return dict(pvalue=pv, padj=np.zeros(0), j=0, theta=np.full(NT, np.nan), cut=np.full(NT, np.nan),
                    numRej=np.zeros(NT, np.int64))
    lower = r_mean_logical(bm == 0)
    upper = .95 if lower < .95 else 1.0
    theta = r_seq50(lower, upper)
    cut = r_quantile7(bm, theta)
    # filtered_p column by column, over the rows sorted once by p-value (p.adjust's values do not depend on the order
    # of tied p-values)
    ok = np.flatnonzero(~np.isnan(pv))
    o = ok[np.argsort(pv[ok], kind="stable")]
    ps, bs = pv[o], bm[o]
    numRej = np.zeros(NT, np.int64)
    for k in range(NT):
        use = bs >= cut[k]
        if use.any():
            numRej[k] = np.count_nonzero(_bh_ascending(ps[use]) < ALPHA)
    if numRej.max() <= 10:
        j = 0
    else:
        lo_fit = O.lowess(theta, numRej.astype(np.float64), f=1 / 5)
        pos = numRej > 0
        thresh = lo_fit.max() - np.sqrt(np.mean((numRej[pos] - lo_fit[pos]) ** 2))
        w = np.flatnonzero(numRej > thresh)
        j = int(w[0]) if len(w) else 0
    padj = np.full(n, np.nan)
    if n:
        use = bs >= cut[j]
        padj[o[use]] = _bh_ascending(ps[use])
    return dict(pvalue=pv, padj=padj, j=j, theta=theta, cut=cut, numRej=numRej)


def r_log(x):
    """log(abs(x)) with the C library's log, as the host routine takes it"""
    with np.errstate(divide="ignore"):
        return np.array([math.log(abs(v)) if abs(v) > 0 and not math.isnan(v) else
                         (-math.inf if v == 0 else math.nan) for v in np.asarray(x, dtype=np.float64)])


def r_breaks(minLogDist, maxLogDist):
    return np.sort((np.concatenate([minLogDist, [np.inf]]) + np.concatenate([[0.0], maxLogDist])) / 2)


def r_bincode(x, breaks):
    """.bincode(x, breaks, right = TRUE, include.lowest = FALSE); -1 = NA"""
    nb1 = len(breaks) - 1
    out = np.full(len(x), -1, np.int64)
    for i, v in enumerate(x):
        if math.isnan(v) or v < breaks[0] or breaks[nb1] < v or v == breaks[0]:
            continue
        lo, hi = 0, nb1
        while hi - lo >= 2:
            new = (hi + lo) // 2
            if v > breaks[new]:
                lo = new
            else:
                hi = new
        out[i] = lo + 1
    return out


def r_ihw(avDist, pvalue, minLogDist, maxLogDist, avWeights, group=None):
    """IHWcorrection's weight application.  group: the strata to use instead of cut() (to follow a routine whose log
    put a row on the other side of a break)"""
    w = np.asarray(avWeights, dtype=np.float64)
    if group is None:
        group = r_bincode(r_log(avDist), r_breaks(minLogDist, maxLogDist))
    group = np.asarray(group, dtype=np.int64)
    na = group < 0
    avw = np.where(na, np.nan, w[np.clip(group, 1, len(w)) - 1])
    meanw = r_mean(avw[np.argsort(group, kind="stable")]) if len(avw) else float("nan")   # merge() sorts by group
    weight = avw / meanw
    wp = np.asarray(pvalue, dtype=np.float64) / weight
    return dict(group=group, weight=weight, weighted_pvalue=wp, weighted_padj=r_p_adjust_bh(wp))


# ---------------------------------------------------------------------------------------------------------------------
# comparisons
# ---------------------------------------------------------------------------------------------------------------------

def same(a, b):
    """equal values and NaN at the same places (NaN payloads may differ between host and device)"""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def close(got, ref, tol=1e-15):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    if not np.array_equal(np.isnan(got), np.isnan(ref)):
        return False
    ok = ~np.isnan(ref)
    return bool(np.all(np.abs(got[ok] - ref[ok]) <= tol * np.maximum(1.0, np.abs(ref[ok]))))


def check_against_reference(got, ref):
    assert same(got["pvalue"], ref["pvalue"]), "Cook's filter"
    assert got["filterIndex"] == ref["j"] + 1, ("filter index", got["filterIndex"], ref["j"] + 1, ref["numRej"])
    if len(ref["pvalue"]):
        assert got["filterThreshold"] == ref["cut"][ref["j"]], (got["filterThreshold"], ref["cut"][ref["j"]])
        assert got["filterTheta"] == ref["theta"][ref["j"]], (got["filterTheta"], ref["theta"][ref["j"]])
    assert np.array_equal(np.isnan(got["padj"]), np.isnan(ref["padj"])), "NA pattern of padj"
    assert close(got["padj"], ref["padj"]), "padj"


def check_device_against_host(dev, host):
    assert same(dev["pvalue"], host["pvalue"]), "Cook's filter"
    assert same(dev["padj"], host["padj"]), "padj"
    for k in ("cooksCutoff", "filterThreshold", "filterTheta", "filterIndex"):
        assert dev[k] == host[k] or (np.isnan(dev[k]) and np.isnan(host[k])), k


# ---------------------------------------------------------------------------------------------------------------------
# results() cases: name -> (baseMean, maxCooks, flags, pvalue, S, p)
# ---------------------------------------------------------------------------------------------------------------------

def _cutoff(S, p):
    return engine.results_adjust(np.ones(1), None, None, np.ones(1), S, p)["cooksCutoff"]


def _typical(n, seed):
    """tied low baseMeans (rounded), 10 % zeros, 10 % signal, a few NA p-values and Cook's outliers"""
    rng = np.random.default_rng(seed)
    bm = np.round(np.exp(rng.normal(2.0, 1.5, n)), 1)
    bm[rng.random(n) < 0.1] = 0.0
    sig = rng.random(n) < 0.1
    p = np.where(sig, rng.random(n) ** 6 * 1e-3, rng.random(n))
    p[bm == 0] = np.nan
    p[rng.random(n) < 0.01] = np.nan
    mc = rng.random(n) * 12
    mc[rng.random(n) < 0.01] = 40.0
    fl = np.where(rng.random(n) < 0.5, engine.FLAG_COOKS_KEEP, 0).astype(np.uint8)
    return bm, mc, fl, p, 6, 2


def _index_case(n, k, tied=500, signal=200, seed=0):
    """A dataset on which quantile()'s 1-based index keeps rows the 0-based index (n - 1) * theta drops (found by
    scripts/quantile_index_search.py): no zero baseMean, so theta_k = k * (0.95 / 49); in R's index h is exactly 0
    and the cut is the sorted value at lo, 1.0, shared by `tied` rows; (n - 1) * theta_k is one ulp above an integer,
    so the 0-based cut interpolates towards the next value, 2.0, and lands above 1.0.  Signal p-values are rejected
    from cut-off k on and not before, so that results() picks cut-off k."""
    theta = r_seq50(0.0, 0.95)
    x = (n - 1) * theta[k]
    lo0 = math.floor(x)                                                    # 0-based sorted position of the cut
    rng = np.random.default_rng(seed)
    low = np.sort(rng.uniform(0.01, 0.9, lo0 - tied + 1))
    high = np.sort(rng.uniform(2.0, 100.0, n - lo0 - 1))
    high[0] = 2.0
    bm = np.concatenate([low, np.full(tied, 1.0), high])
    p = rng.uniform(0.2, 1.0, n)
    m_k = n - (lo0 - tied + 1)                                             # rows at or above the cut in R
    m_prev = n - math.floor(1.0 + (n - 1) * theta[k - 1]) + 1
    s = ALPHA * signal / ((m_k + m_prev) / 2.0)
    p[n - signal:] = s                                                     # the largest baseMeans: kept at every cut-off
    perm = rng.permutation(n)
    return bm[perm], None, None, p[perm], 6, 2


def _pvalue_case(kind, n=3 * 2048 + 300, seed=11):
    rng = np.random.default_rng(seed)
    bm = np.exp(rng.normal(3, 1, n))
    p = rng.random(n)
    if kind == "all_na":
        p[:] = np.nan
    elif kind == "one_non_na":
        p[:] = np.nan
        p[n // 2] = 1e-8
    elif kind == "all_equal":
        p[:] = 0.003
    elif kind == "zero_and_one":
        p[rng.random(n) < 0.1] = 0.0
        p[rng.random(n) < 0.1] = 1.0
        p[rng.random(n) < 0.05] = 1e-6
    elif kind == "tie_runs":
        # runs of 700 equal p-values: in p order they straddle the 2048-row chunks and the 256-row blocks
        vals = np.array([1e-9, 1e-5, 2e-4, 1e-3, 0.02, 0.3, 0.7, 1.0])
        p = np.sort(vals[np.minimum(np.arange(n) // 700, len(vals) - 1)])
        bm = rng.permutation(np.exp(rng.normal(3, 1, n)))
    elif kind == "tiny_last_rank":
        p = rng.uniform(0.5, 0.5001, n)
        p[n // 3] = 1e-300
    return bm, None, None, p, 6, 2


def _basemean_case(kind, n=4000, seed=12):
    rng = np.random.default_rng(seed)
    p = np.where(rng.random(n) < 0.2, rng.random(n) * 1e-4, rng.random(n))
    if kind == "all_zero":
        bm = np.zeros(n)
    elif kind in ("zero_95", "zero_95_plus", "zero_95_minus"):
        nz = {"zero_95": 3800, "zero_95_plus": 3801, "zero_95_minus": 3799}[kind]
        bm = np.exp(rng.normal(3, 1, n))
        bm[rng.permutation(n)[:nz]] = 0.0
    elif kind == "tied_at_cut":
        bm = rng.choice(np.array([0.5, 1.0, 2.0, 7.25, 30.0]), n)        # every cut-off is one of five values
    elif kind == "huge_range":
        bm = 10.0 ** rng.uniform(-300, 300, n)
    return bm, None, None, p, 6, 2


def _rejection_case(kind, n=3000, seed=13):
    rng = np.random.default_rng(seed)
    bm = np.exp(rng.normal(3, 1, n))
    p = rng.uniform(0.3, 1.0, n)
    top = np.argsort(bm)[::-1]
    if kind in ("max10", "max11"):
        # signal rows spread over baseMean: numRej falls as the filter rises, its maximum is 10 or 11
        r = 10 if kind == "max10" else 11
        p[top[np.linspace(0, n - 1, r).astype(int)]] = 1e-9
    elif kind == "constant":
        p[top[:60]] = 1e-12                                                # kept and rejected at every cut-off
    # "none": no p-value below 0.3
    return bm, None, None, p, 6, 2


def _cooks_case(kind, seed=14):
    n = 600
    rng = np.random.default_rng(seed)
    bm = np.exp(rng.normal(3, 1, n))
    p = np.where(rng.random(n) < 0.2, 1e-6, rng.random(n))
    S, pp = (6, 2) if kind != "keep_p3" else (9, 3)
    c = _cutoff(S, pp)
    mc = rng.random(n) * c * 0.5
    mc[0:50] = c                                                           # not an outlier: the test is '>'
    mc[50:100] = np.nextafter(c, np.inf)                                   # outlier
    mc[100:150] = np.nan                                                   # never an outlier
    mc[150:200] = np.nextafter(c, np.inf)
    fl = np.zeros(n, np.uint8)
    fl[150:200] = engine.FLAG_COOKS_KEEP                                   # kept only when p == 2
    return bm, mc, fl, p, S, pp


def _lower_case():
    """mean(filter == 0) with nzero = 115, n = 2051: R's long-double quotient rounds to another double than 115 / 2051"""
    n, nz = 2051, 115
    rng = np.random.default_rng(15)
    bm = np.exp(rng.normal(3, 1, n))
    bm[:nz] = 0.0
    p = rng.uniform(0.5, 1.0, n)                                           # no rejection: j = 1, filterTheta = lower
    return bm, None, None, p, 6, 2


SMALL_N = [0, 1, 2, 49, 50, 51, 2047, 2048, 2049]
BIG_N = [256 * 2048 - 1, 256 * 2048, 256 * 2048 + 1, 1_100_000]           # chunk count crosses 256; > 512 chunks
INDEX_CASES = [(375586, 36), (2253511, 6)]

CASES = {}
for _n in SMALL_N + BIG_N:
    CASES["n%d" % _n] = (lambda n=_n: _typical(n, n % 97))
for _k in ("all_na", "one_non_na", "all_equal", "zero_and_one", "tie_runs", "tiny_last_rank"):
    CASES["p_" + _k] = (lambda k=_k: _pvalue_case(k))
for _k in ("all_zero", "zero_95", "zero_95_plus", "zero_95_minus", "tied_at_cut", "huge_range"):
    CASES["bm_" + _k] = (lambda k=_k: _basemean_case(k))
for _k in ("max10", "max11", "none", "constant"):
    CASES["rej_" + _k] = (lambda k=_k: _rejection_case(k))
for _k in ("keep_p2", "keep_p3"):
    CASES["cooks_" + _k] = (lambda k=_k: _cooks_case(k))
for _n, _k in INDEX_CASES:
    CASES["index_n%d_k%d" % (_n, _k)] = (lambda n=_n, k=_k: _index_case(n, k))
CASES["lower_long_double"] = _lower_case

_built_cases = {}


def case(name):
    if name not in _built_cases:
        _built_cases.clear()                                               # keep one (possibly large) case in memory
        _built_cases[name] = CASES[name]()
    return _built_cases[name]


def run_host(c):
    bm, mc, fl, p, S, pp = c
    return engine.results_adjust(bm, mc, fl, p, S, pp)


def run_reference(c, cutoff):
    bm, mc, fl, p, S, pp = c
    return r_results(bm, mc, fl, p, pp, cutoff)


# ---------------------------------------------------------------------------------------------------------------------
# results(): host routine against the reference
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(CASES))
def test_results_host_matches_r(built, name):
    c = case(name)
    host = run_host(c)
    ref = run_reference(c, host["cooksCutoff"])
    assert len(host["padj"]) == len(c[0])
    check_against_reference(host, ref)


def test_cooks_cutoff_is_qf():
    from scipy import stats
    for S, p in ((4, 2), (6, 2), (9, 3), (16, 2), (16, 3)):
        got = _cutoff(S, p)
        assert abs(got - stats.f.ppf(0.99, p, S - p)) <= 1e-12 * got, (S, p)


def test_cases_reach_their_edges(built):
    """The cases do what their names say, per the reference"""
    bm, mc, fl, p, S, pp = case("cooks_keep_p2")
    host = run_host(case("cooks_keep_p2"))
    pv = host["pvalue"]
    assert not np.isnan(pv[0:50]).any() and np.isnan(pv[50:100]).all() and not np.isnan(pv[100:150]).any()
    assert not np.isnan(pv[150:200]).any()
    assert np.isnan(run_host(case("cooks_keep_p3"))["pvalue"][150:200]).all()
    for name, upper in (("bm_zero_95", 1.0), ("bm_zero_95_plus", 1.0), ("bm_zero_95_minus", .95), ("bm_all_zero", 1.0)):
        c = case(name)
        r = run_reference(c, 18.0)
        assert r["theta"][-1] == upper, name
    assert np.all(run_reference(case("bm_all_zero"), 18.0)["theta"] == 1.0)
    assert run_reference(case("rej_max10"), 18.0)["numRej"].max() == 10
    assert run_reference(case("rej_max11"), 18.0)["numRej"].max() == 11
    assert run_reference(case("rej_none"), 18.0)["numRej"].max() == 0
    r = run_reference(case("rej_constant"), 18.0)["numRej"]
    assert r.min() == r.max() > 10
    c = case("p_tie_runs")
    assert len(np.unique(c[3])) == 8


def test_order_within_tied_pvalues_does_not_change_padj(built):
    bm, mc, fl, p, S, pp = case("p_tie_runs")
    host = engine.results_adjust(bm, mc, fl, p, S, pp)
    perm = np.random.default_rng(1).permutation(len(p))
    again = engine.results_adjust(bm[perm], None, None, p[perm], S, pp)
    assert same(again["padj"], host["padj"][perm])


# ---------------------------------------------------------------------------------------------------------------------
# the discrepancies these cases found, one test each
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,k", INDEX_CASES)
def test_quantile_index_is_one_based(built, n, k):
    """quantile(type = 7) computes index <- 1 + (n - 1) * probs.  The library used (n - 1) * theta (0-based): on this
    dataset the cut at theta_k came out one ulp above 1.0 and the rows tied at 1.0 were filtered out.

    scripts/quantile_index_search.py finds such n for (n - 1) * theta_k in [2^18 - 1, 2^18) one ulp above an
    integer (k = 36 at n = 375 586, k = 6 at n = 2 253 511, among others below 10^7)."""
    c = case("index_n%d_k%d" % (n, k))
    theta = r_seq50(0.0, 0.95)[k]
    x = (n - 1) * theta
    assert 1.0 + x == math.floor(1.0 + x) and x != math.floor(x)          # R: h == 0; 0-based: h > 0
    ref = run_reference(c, 18.0)
    assert ref["j"] == k and ref["cut"][k] == 1.0
    host = run_host(c)
    check_against_reference(host, ref)
    assert host["filterThreshold"] == 1.0 and not np.isnan(host["padj"][c[0] == 1.0]).any()


def test_lower_quantile_is_rs_long_double_mean(built):
    """mean(filter == 0) is a long-double quotient rounded to double; 115 / 2051 in double is another number"""
    c = case("lower_long_double")
    lower = r_mean_logical(c[0] == 0)
    assert lower != 115 / 2051
    host = run_host(c)
    assert host["filterIndex"] == 1 and host["filterTheta"] == lower


def test_oracle_quantile_and_bh_follow_r():
    """the oracle's quantile7 had the fuzz of types 4-9 and a 0-based index; its BH capped a lone p-value at 1"""
    from oracle import oracle as O
    for n, k in INDEX_CASES[:1]:
        bm = case("index_n%d_k%d" % (n, k))[0]
        th = r_seq50(0.0, 0.95)
        assert same(O.quantile7(bm, th), r_quantile7(bm, th))
    rng = np.random.default_rng(2)
    for n in (1, 2, 3, 7, 1000):
        x = np.round(rng.random(n) * 5, 1)
        th = r_seq50(r_mean_logical(x == 0), .95)
        assert same(O.quantile7(x, th), r_quantile7(x, th)), n
    assert same(O.p_adjust_bh(np.array([np.nan, 1.7, np.nan])), [np.nan, 1.7, np.nan])


# ---------------------------------------------------------------------------------------------------------------------
# IHW weight application
# ---------------------------------------------------------------------------------------------------------------------

def _lookup(G, seed=21, spread=(0.2, 3.0)):
    """minLogDist / maxLogDist whose breaks are B_1 < ... < B_{G-1} in (1, 14), with breaks[0] = 0 and Inf at the end"""
    rng = np.random.default_rng(seed)
    B = np.sort(rng.uniform(1.0, 14.0, G - 1)) if G > 1 else np.zeros(0)
    B = np.unique(B)
    while len(B) < G - 1:                                                  # uniform draws rarely repeat; keep G groups
        B = np.unique(np.concatenate([B, rng.uniform(1.0, 14.0, G - 1 - len(B))]))
    lo = np.concatenate([[0.0], B])
    hi = np.concatenate([B, [np.inf]])
    w = rng.uniform(*spread, G)
    return lo, hi, w


def _ihw_case(kind, n=3000, G=6, seed=22):
    rng = np.random.default_rng(seed)
    lo, hi, w = _lookup(G)
    av = np.exp(rng.uniform(0.5, 14.5, n)) * np.where(rng.random(n) < 0.5, -1, 1)
    p = rng.random(n)
    if kind == "edges":
        br = r_breaks(lo, hi)[1:-1]
        e = np.exp(br)
        special = np.concatenate([[0.0, -0.0, np.inf, -np.inf, np.nan, -5.0, 1.0, np.exp(0.0)], e, np.nextafter(e, np.inf),
                                  np.nextafter(e, -np.inf), -e])
        av[:len(special)] = special
    elif kind == "above_one":
        lo, hi, w = _lookup(G, spread=(0.01, 100.0))
        p = rng.uniform(0.9, 1.0, n)
    elif kind == "ties":
        av = np.full(n, np.exp(0.7))                                       # one group: equal weights
        p = np.sort(np.array([1e-6, 1e-3, 0.05, 0.5])[np.arange(n) * 4 // n])
    elif kind == "zeros":
        p[::3] = 0.0
        p[1::3] = -0.0
    elif kind == "all_na":
        p[:] = np.nan
    elif kind == "lone":
        p[:] = np.nan
        p[n // 2] = 0.999
        lo, hi, w = _lookup(G, spread=(0.01, 100.0))
        av[n // 2] = np.exp(hi[np.argmin(w)] - 1e-3) if np.isfinite(hi[np.argmin(w)]) else np.exp(20.0)
    return av, p, lo, hi, w


IHW_CASES = {}
for _n in (0, 1, 255, 256, 257):
    IHW_CASES["n%d" % _n] = (lambda n=_n: _ihw_case("plain", n=n))
for _G in (1, 1024, 1025, 3000):
    IHW_CASES["G%d" % _G] = (lambda G=_G: _ihw_case("plain", n=20000, G=G))
for _k in ("edges", "above_one", "ties", "zeros", "all_na", "lone"):
    IHW_CASES[_k] = (lambda k=_k: _ihw_case(k))


def check_ihw_against_reference(got, ref):
    assert np.array_equal(np.where(got["group"] == np.iinfo(np.int32).min, -1, got["group"]), ref["group"]), "group"
    for k in ("weight", "weighted_pvalue", "weighted_padj"):
        assert close(got[k], ref[k]), k


@pytest.mark.parametrize("name", list(IHW_CASES))
def test_ihw_host_matches_r(built, name):
    av, p, lo, hi, w = IHW_CASES[name]()
    host = engine.ihw_apply(av, p, lo, hi, w)
    check_ihw_against_reference(host, r_ihw(av, p, lo, hi, w))


def test_ihw_cases_reach_their_edges(built):
    av, p, lo, hi, w = IHW_CASES["above_one"]()
    r = r_ihw(av, p, lo, hi, w)
    assert (r["weighted_pvalue"] > 1).sum() > 100 and np.nanmax(r["weighted_padj"]) == 1.0
    av, p, lo, hi, w = IHW_CASES["edges"]()
    r = r_ihw(av, p, lo, hi, w)
    assert r["group"][0] == -1 and r["group"][2] == len(w) and r["group"][4] == -1   # log 0 = -Inf: NA; Inf: last group
    r = r_ihw(*IHW_CASES["lone"]())
    assert np.count_nonzero(~np.isnan(r["weighted_pvalue"])) == 1 and np.nanmax(r["weighted_pvalue"]) > 1


def test_ihw_lone_weighted_pvalue_is_not_capped(built):
    """p.adjust returns its input when at most one p-value is not NA: a lone weighted p-value above 1 stays above 1.
    The library capped it at 1."""
    av, p, lo, hi, w = IHW_CASES["lone"]()
    host = engine.ihw_apply(av, p, lo, hi, w)
    i = np.flatnonzero(~np.isnan(host["weighted_pvalue"]))
    assert len(i) == 1 and host["weighted_pvalue"][i[0]] > 1
    assert host["weighted_padj"][i[0]] == host["weighted_pvalue"][i[0]]


# ---------------------------------------------------------------------------------------------------------------------
# the device routines
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu_engine(built):
    e = engine.Engine(0)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_results_device_matches_host_and_r(gpu_engine, name):
    c = case(name)
    bm, mc, fl, p, S, pp = c
    dev = gpu_engine.results_device(bm, mc, fl, p, S, pp)
    host = run_host(c)
    check_device_against_host(dev, host)
    check_against_reference(dev, run_reference(c, host["cooksCutoff"]))


@pytest.mark.gpu
def test_results_device_tied_order_and_bad_arguments(gpu_engine):
    bm, mc, fl, p, S, pp = case("p_tie_runs")
    a = gpu_engine.results_device(bm, mc, fl, p, S, pp)
    perm = np.random.default_rng(1).permutation(len(p))
    b = gpu_engine.results_device(bm[perm], None, None, p[perm], S, pp)
    assert same(b["padj"], a["padj"][perm])
    with pytest.raises(engine.ChicdiffError):
        gpu_engine.results_device(bm, None, None, p, 2, 2)                # S <= p


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(IHW_CASES))
def test_ihw_device_matches_host_and_r(gpu_engine, name):
    av, p, lo, hi, w = IHW_CASES[name]()
    host = engine.ihw_apply(av, p, lo, hi, w)
    dev = gpu_engine.ihw_apply_device(p, lo, hi, w, avDist=av)
    if not np.array_equal(dev["group"], host["group"]):
        # only where the device log and the host log fall on opposite sides of a break
        br = r_breaks(lo, hi)
        x = r_log(av)
        for i in np.flatnonzero(dev["group"] != host["group"]):
            near = br[np.argmin(np.abs(br - x[i]))]
            assert np.nextafter(x[i], -np.inf) <= near <= np.nextafter(x[i], np.inf), (i, x[i], near)
        dg = np.where(dev["group"] == np.iinfo(np.int32).min, -1, dev["group"])
        check_ihw_against_reference(dev, r_ihw(av, p, lo, hi, w, group=dg))
        return
    for k in ("group", "weight", "weighted_pvalue", "weighted_padj"):
        assert same(dev[k], host[k]), k
    check_ihw_against_reference(dev, r_ihw(av, p, lo, hi, w))
