"""ctypes front end of the CPU oracle (oracle/chicdiff_oracle.c) plus the NumPy restatement
of DESeq2 ``results()`` (Cook's cutoff, independent filtering, BH).

TEST INFRASTRUCTURE -- see the header of chicdiff_oracle.c.  PARITY UNPINNED at the DESeq2
boundary; pinned pieces are listed there.  Imported only by tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs.
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_VARIANTS = {}

FLAG_ALLZERO, FLAG_GENE_GRID, FLAG_MAP_GRID, FLAG_BETA_NOCONV, FLAG_OUTLIER, FLAG_GENE_NOINCREASE = 1, 2, 4, 8, 16, 32


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle.so"])


def variant(name):
    """The same source built differently (oracle/Makefile: "O0", "fma", "ld"); only orc_deseq_ex is bound.  Used by
    scripts/oracle_flip_evidence.py to show which rows depend on the rounding of the reference's own arithmetic."""
    if name not in _VARIANTS:
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle_%s.so" % name])
        _VARIANTS[name] = C.CDLL(os.path.join(_HERE, "liboracle_%s.so" % name))
    return _VARIANTS[name]


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(os.path.join(_HERE, "chicdiff_oracle.c")):
            build()
        L = C.CDLL(path)
        d = C.c_double
        for name, nargs in [("orc_lgamma", 1), ("orc_digamma", 1), ("orc_trigamma", 1), ("orc_wald_pvalue", 1)]:
            getattr(L, name).restype = d
            getattr(L, name).argtypes = [d] * nargs
        L.orc_dnbinom_mu_log.restype = d
        L.orc_dnbinom_mu_log.argtypes = [d, d, d]
        L.orc_qf.restype = d
        L.orc_qf.argtypes = [d, d, d]
        for name in ("orc_log_posterior", "orc_dlog_posterior"):
            f = getattr(L, name)
            f.restype = d
            f.argtypes = [d, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, d, d, C.c_int, C.c_int]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class _OrcOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in (
        "baseMean", "baseVar", "dispGeneEst", "dispFit", "dispMAP", "dispersion", "beta", "betaSE",
        "stat", "pvalue", "deviance", "maxCooks", "mu", "H", "cooks", "dispGeneIter", "dispIter",
        "betaIter", "allZero", "dispOutlier", "betaConv", "flags", "scalars")]


def aggregate(row_off, N_rows, FM_rows):
    """row_off int64[n+1]; N_rows int32[S, R]; FM_rows float64[S, R] -> K int32[S, n], FM float64[S, n]."""
    row_off = np.ascontiguousarray(row_off, dtype=np.int64)
    N_rows = np.ascontiguousarray(N_rows, dtype=np.int32)
    FM_rows = np.ascontiguousarray(FM_rows, dtype=np.float64)
    S, R = N_rows.shape
    n = len(row_off) - 1
    K = np.empty((S, n), np.int32)
    FM = np.empty((S, n), np.float64)
    rc = lib().orc_aggregate(C.c_int64(n), C.c_int(S), _p(row_off), C.c_int64(R), _p(N_rows), _p(FM_rows), _p(K), _p(FM))
    assert rc == 0
    return K, FM


NEGATIVE_COUNTS = "NA or negative values in the count matrix"


def size_factors(K):
    K = np.ascontiguousarray(K, dtype=np.int32)
    S, n = K.shape
    sf = np.empty(S, np.float64)
    rc = lib().orc_size_factors(C.c_int64(n), C.c_int(S), _p(K), _p(sf))
    if rc == -2:
        raise ValueError(NEGATIVE_COUNTS)
    if rc != 0:
        raise ValueError("every gene contains at least one zero, cannot compute log geometric means")
    return sf


NORM_MODES = {"standard": 0, "fullmean": 1, "combined": 2}


def norm_factors(FMagg, sf, norm, theta=0.0):
    FMagg = np.ascontiguousarray(FMagg, dtype=np.float64)
    sf = np.ascontiguousarray(sf, dtype=np.float64)
    S, n = FMagg.shape
    nf = np.empty((S, n), np.float64)
    lib().orc_norm_factors(C.c_int64(n), C.c_int(S), _p(FMagg), _p(sf), C.c_int(NORM_MODES[norm]),
                           C.c_double(theta), _p(nf))
    return nf


class _OrcExt(C.Structure):
    _fields_ = [("trend_a0", C.c_double), ("trend_a1", C.c_double), ("var_log_disp", C.c_double),
                ("gene_margin", C.c_void_p), ("map_margin", C.c_void_p)]


def deseq(K, nf, X, prior_var=float("nan"), grid_n=20, nthreads=0, trend=None, var_log_disp=None, margins=False, L=None):
    """estimateDispersions + nbinomWaldTest.  K int32[S,n], nf float64[S,n], X float64[S,p].
    trend = (a0, a1) / var_log_disp: take these global scalars instead of fitting them; margins: also return
    geneMargin / mapMargin (decision margins of the two line searches in rounding-error units); L: a variant build."""
    K = np.ascontiguousarray(K, dtype=np.int32)
    nf = np.ascontiguousarray(nf, dtype=np.float64)
    X = np.ascontiguousarray(X, dtype=np.float64)
    S, n = K.shape
    p = X.shape[1]
    f8 = lambda *sh: np.full(sh, np.nan, np.float64)
    res = dict(
        baseMean=f8(n), baseVar=f8(n), dispGeneEst=f8(n), dispFit=f8(n), dispMAP=f8(n), dispersion=f8(n),
        beta=f8(p, n), betaSE=f8(p, n), stat=f8(n), pvalue=f8(n), deviance=f8(n), maxCooks=f8(n),
        mu=f8(S, n), H=f8(S, n), cooks=f8(S, n),
        dispGeneIter=np.zeros(n, np.int32), dispIter=np.zeros(n, np.int32), betaIter=np.zeros(n, np.int32),
        allZero=np.zeros(n, np.uint8), dispOutlier=np.zeros(n, np.uint8), betaConv=np.zeros(n, np.uint8),
        flags=np.zeros(n, np.uint8), scalars=f8(16))
    out = _OrcOut(**{k: _p(v) for k, v in res.items()})
    nan = float("nan")
    ext = _OrcExt(nan, nan, nan, None, None)
    if trend is not None:
        ext.trend_a0, ext.trend_a1 = float(trend[0]), float(trend[1])
    if var_log_disp is not None:
        ext.var_log_disp = float(var_log_disp)
    if margins:
        res["geneMargin"], res["mapMargin"] = f8(n), f8(n)
        ext.gene_margin, ext.map_margin = res["geneMargin"].ctypes.data, res["mapMargin"].ctypes.data
    rc = (L or lib()).orc_deseq_ex(C.c_int64(n), C.c_int(S), C.c_int(p), _p(X), _p(K), _p(nf), C.c_double(prior_var),
                                   C.c_int(grid_n), C.c_int(nthreads), C.byref(ext), C.byref(out))
    res["rc"] = rc
    sc = res["scalars"]
    res.update(trend_a0=sc[0], trend_a1=sc[1], varLogDispEsts=sc[2], dispPriorVar=sc[3], trend_status=int(sc[4]) if sc[4] == sc[4] else -1,
               lp_evals=sc[8], dlp_evals=sc[9], irls_iters=sc[10], sum_deviance=sc[11], n_nonzero=sc[12])
    if rc != 0:
        raise RuntimeError({-1: "bad design (S<=p or too large)", -2: "S-p<=3 needs dispPriorVar (Monte-Carlo path not restated)",
                            -3: "parametric dispersion trend failed (local fit not restated)",
                            -4: NEGATIVE_COUNTS}.get(rc, "rc=%d" % rc))
    return res


def region_test(K, FMagg, X, norm="combined", theta=None, theta_grid=(0, .25, .5, .75, 1), prior_var=float("nan"),
                prior_var_grid=float("nan"), nthreads=0, trend=None, var_log_disp=None, margins=False, L=None, grid_n=20):
    """DESeq2Wrap numerics (chicdiff.R:1551-1674): size factors, offsets, theta grid, final fit.
    trend / var_log_disp / margins / L apply to the final fit only (see deseq); grid_n (fitDispGrid length) to every fit.
    NA (INT32_MIN) or negative counts raise ValueError, as DESeqDataSetFromMatrix stops on them."""
    S, n = K.shape
    sf = size_factors(K)
    out = {"sizeFactors": sf, "deviances": None}
    if norm == "combined" and theta is not None:
        if theta == 1:
            norm = "standard"
        elif theta == 0:
            norm = "fullmean"
    if norm == "combined" and theta is None:
        devs = []
        X1 = np.ones((S, 1))
        for tt in theta_grid:
            nf = norm_factors(FMagg, sf, "combined", tt)
            r = deseq(K, nf, X1, prior_var=prior_var_grid, grid_n=grid_n, nthreads=nthreads)
            devs.append(r["sum_deviance"])
        devs = np.asarray(devs)
        out["deviances"] = devs
        if np.any(np.isnan(devs)):
            raise ValueError("theta grid: NA deviance (all-zero region present; chicdiff.R:1647 has no na.rm)")
        w = np.flatnonzero(devs == devs.min())
        if len(w) != 1:
            raise ValueError("theta grid: tied minimum")
        theta = float(theta_grid[w[0]])
    # chicdiff.R:1759: the theta attribute exists only when the "combined" branch assigned `tt`
    out["theta"] = theta if norm == "combined" else None
    nf = norm_factors(FMagg, sf, norm, 0.0 if theta is None else theta)
    out["nf"] = nf
    out.update(deseq(K, nf, X, prior_var=prior_var, grid_n=grid_n, nthreads=nthreads, trend=trend, var_log_disp=var_log_disp,
                     margins=margins, L=L))
    return out


# ---------------------------------------------------------------------------------------------
# DESeq2 results(): Cook's cutoff, independent filtering (genefilter::filtered_p + lowess), BH.
# Pinned by tests/test_golden.py against the shipped golden table.
# ---------------------------------------------------------------------------------------------

def ihw_apply(avDist, pvalue, minLogDist, maxLogDist, avWeights):
    """IHWcorrection(), "apply to test data" (chicdiff.R:2038-2049).  Lookup columns as they stand at :2033.
    Rows stay in input order (the reference's merge() sorts by group afterwards)."""
    avDist = np.asarray(avDist, dtype=np.float64)
    lo, hi, w = (np.asarray(a, dtype=np.float64) for a in (minLogDist, maxLogDist, avWeights))
    breaks = (np.concatenate([lo, [np.inf]]) + np.concatenate([[0.0], hi])) / 2          # :2039
    breaks = np.sort(breaks)
    if np.any(np.diff(breaks) == 0):
        raise ValueError("'breaks' are not unique")
    with np.errstate(divide="ignore", invalid="ignore"):
        x = np.log(np.abs(avDist))
    # cut(x, breaks): right-closed (b[g-1], b[g]], NA outside
    g = np.searchsorted(breaks, x, side="left")
    na = np.isnan(x) | (g < 1) | (g > len(w))
    group = np.where(na, -1, g)
    avw = np.where(na, np.nan, w[np.clip(group, 1, len(w)) - 1])
    # mean() over the merged table (ordered by group); R accumulates in long double and refines once
    srt = avw[np.argsort(group, kind="stable")].astype(np.longdouble)
    m = srt.sum() / len(srt) if len(srt) else np.longdouble(np.nan)
    m = m + (srt - m).sum() / len(srt) if len(srt) else m
    weight = avw / float(m)
    wp = np.asarray(pvalue, dtype=np.float64) / weight
    return dict(group=group, weight=weight, weighted_pvalue=wp, weighted_padj=p_adjust_bh(wp))


def p_adjust_bh(p):
    p = np.asarray(p, dtype=np.float64)
    out = np.full(p.shape, np.nan)
    ok = ~np.isnan(p)
    pv = p[ok]
    m = len(pv)
    if m == 0:
        return out
    o = np.argsort(-pv, kind="stable")          # decreasing
    ranks = np.arange(m, 0, -1)
    adj = np.minimum(1.0, np.minimum.accumulate(m / ranks * pv[o]))
    res = np.empty(m)
    res[o] = adj
    out[ok] = res
    return out


def quantile7(x, probs):
    xs = np.sort(np.asarray(x, dtype=np.float64))
    n = len(xs)
    h = (n - 1) * np.asarray(probs, dtype=np.float64)
    lo = np.floor(h + 4 * np.finfo(float).eps).astype(np.int64)     # R's fuzz
    lo = np.clip(lo, 0, n - 1)
    hi = np.clip(lo + 1, 0, n - 1)
    frac = h - lo
    frac = np.where(np.abs(frac) < 4 * np.finfo(float).eps, 0.0, frac)
    return xs[lo] + frac * (xs[hi] - xs[lo])


def lowess(x, y, f=2.0 / 3.0, nsteps=3, delta=None):
    """Cleveland's lowess as in R stats::lowess (x must be sorted ascending)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    n = len(x)
    if delta is None:
        delta = 0.01 * (x[-1] - x[0])
    ys = np.zeros(n)
    rw = np.ones(n)
    res = np.zeros(n)
    if n < 2:
        return y.copy()
    ns = max(2, min(n, int(f * n + 1e-7)))

    def lowest(xs, nleft, nright, userw):
        rng = x[n - 1] - x[0]
        h = max(xs - x[nleft], x[nright] - xs)
        h9, h1 = .999 * h, .001 * h
        w = np.zeros(n)
        a = 0.0
        j = nleft
        while j < n:
            r = abs(x[j] - xs)
            if r <= h9:
                w[j] = 1.0 if r <= h1 else (1.0 - (r / h) ** 3) ** 3
                if userw:
                    w[j] *= rw[j]
                a += w[j]
            elif x[j] > xs:
                break
            j += 1
        nrt = j - 1
        if a <= 0:
            return None
        w[nleft:nrt + 1] /= a
        if h > 0:
            a = float(np.sum(w[nleft:nrt + 1] * x[nleft:nrt + 1]))
            b = xs - a
            c = float(np.sum(w[nleft:nrt + 1] * (x[nleft:nrt + 1] - a) ** 2))
            if np.sqrt(c) > .001 * rng:
                b /= c
                w[nleft:nrt + 1] *= (b * (x[nleft:nrt + 1] - a) + 1.0)
        return float(np.sum(w[nleft:nrt + 1] * y[nleft:nrt + 1]))

    for it in range(nsteps + 1):
        nleft, nright, last, i = 0, ns - 1, -1, 0
        while True:
            if nright < n - 1:
                d1 = x[i] - x[nleft]
                d2 = x[nright + 1] - x[i]
                if d1 > d2:
                    nleft += 1
                    nright += 1
                    continue
            v = lowest(x[i], nleft, nright, it > 0)
            ys[i] = y[i] if v is None else v
            if last < i - 1:
                denom = x[i] - x[last]
                for j in range(last + 1, i):
                    alpha = (x[j] - x[last]) / denom
                    ys[j] = alpha * ys[i] + (1.0 - alpha) * ys[last]
            last = i
            cut = x[last] + delta
            i = last + 1
            while i < n:
                if x[i] > cut:
                    break
                if x[i] == x[last]:
                    ys[i] = ys[last]
                    last = i
                i += 1
            i = max(last + 1, i - 1)
            if last >= n - 1:
                break
        res = y - ys
        sc = np.sum(np.abs(res)) / n
        if it >= nsteps:
            break
        rw = np.abs(res)
        srt = np.sort(rw)
        m1 = n // 2
        if n % 2 == 0:
            m2 = n - m1 - 1
            cmad = 3.0 * (srt[m1] + srt[m2])
        else:
            cmad = 6.0 * srt[m1]
        if cmad < 1e-7 * sc:
            break
        c9, c1 = .999 * cmad, .001 * cmad
        r = np.abs(res)
        rw = np.where(r <= c1, 1.0, np.where(r <= c9, (1.0 - (r / cmad) ** 2) ** 2, 0.0))
    return ys


def independent_filtering(base_mean, pvalue, alpha=0.1):
    """DESeq2 pvalueAdjustment (independentFiltering=TRUE, filter=baseMean).  Returns dict."""
    flt = np.asarray(base_mean, dtype=np.float64)
    p = np.asarray(pvalue, dtype=np.float64)
    lower = np.mean(flt == 0)
    upper = .95 if lower < .95 else 1.0
    theta = np.linspace(lower, upper, 50)
    cut = quantile7(flt, theta)
    padj_mat = np.full((len(p), 50), np.nan)
    for k in range(50):
        use = flt >= cut[k]
        if use.any():
            padj_mat[use, k] = p_adjust_bh(p[use])
    with np.errstate(invalid="ignore"):
        num_rej = np.sum(padj_mat < alpha, axis=0)
    lo = lowess(theta, num_rej.astype(np.float64), f=1 / 5)
    if num_rej.max() <= 10:
        j = 0
    else:
        pos = num_rej > 0
        resid = num_rej[pos] - lo[pos]
        thresh = lo.max() - np.sqrt(np.mean(resid ** 2))
        w = np.flatnonzero(num_rej > thresh)
        j = int(w[0]) if len(w) else 0
    return dict(padj=padj_mat[:, j], j=j, theta=theta[j], cutoff=cut[j], num_rej=num_rej, lowess=lo)


def results(res, K, X, alpha=0.1):
    """DESeq2 results() defaults on the output of deseq(): Cook's outlier NA + independent filtering."""
    S, n = K.shape
    p = X.shape[1]
    pvalue = res["pvalue"].copy()
    max_cooks = res["maxCooks"]
    cutoff = lib().orc_qf(0.99, float(p), float(S - p))
    with np.errstate(invalid="ignore"):
        outlier = max_cooks > cutoff
    # two-level single-factor heuristic: keep rows where >= 3 counts exceed the max-Cook's sample's count
    two_level = (p == 2 and set(np.unique(X[:, 0])) == {1.0} and len(np.unique(X[:, 1])) == 2)
    if outlier.any() and two_level:
        idx = np.flatnonzero(outlier)
        worst = np.argmax(res["cooks"][:, idx], axis=0)
        out_count = K[worst, idx]
        keep = (K[:, idx] > out_count[None, :]).sum(axis=0) >= 3
        outlier[idx[keep]] = False
    pvalue[outlier] = np.nan
    f = independent_filtering(res["baseMean"], pvalue, alpha)
    return dict(baseMean=res["baseMean"], log2FoldChange=res["beta"][p - 1], lfcSE=res["betaSE"][p - 1],
                stat=res["stat"], pvalue=pvalue, padj=f["padj"], cooksCutoff=cutoff, cooksOutlier=outlier,
                filterThreshold=f["cutoff"], filterTheta=f["theta"], filterIndex=f["j"])


def assemble_sample(row_bait, row_oe, frag_chr, frag_start, frag_end, tab, frag_id0=1, want_all=False):
    """getFullRegionData1's per-replicate step (chicdiff.R:609-702, 820-910) for one replicate's tables
    (dict with s_j, tblb, s_i, tlb, tmean, distfun, cnt_off, cnt_oe, cnt_N).  Returns N, FullMean per row
    (and distSign, Bmean, Tmean when want_all)."""
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    row_bait, row_oe = i32(row_bait), i32(row_oe)
    R, F = len(row_bait), len(frag_chr)
    tm = f64(tab["tmean"])
    N = np.empty(R, np.int32)
    FM = np.empty(R, np.float64)
    extra = [np.empty(R, np.float64) for _ in range(3)] if want_all else [None, None, None]
    keep = [row_bait, row_oe, i32(frag_chr), i32(frag_start), i32(frag_end), f64(tab["s_j"]), i32(tab["tblb"]), f64(tab["s_i"]),
            i32(tab["tlb"]), tm, f64(tab["distfun"]), np.ascontiguousarray(tab["cnt_off"], dtype=np.int64), i32(tab["cnt_oe"]),
            i32(tab["cnt_N"])]
    rc = lib().orc_assemble_sample(C.c_int64(R), _p(keep[0]), _p(keep[1]), C.c_int64(F), C.c_int32(frag_id0), _p(keep[2]), _p(keep[3]),
                                   _p(keep[4]), _p(keep[5]), _p(keep[6]), _p(keep[7]), _p(keep[8]), C.c_int(tm.shape[0]),
                                   C.c_int(tm.shape[1]), _p(keep[9]), _p(keep[10]), _p(keep[11]), _p(keep[12]), _p(keep[13]),
                                   _p(N), _p(FM), *[None if e is None else _p(e) for e in extra])
    if rc != 0:
        raise ValueError("fragment ID outside the rmap")
    return (N, FM) + tuple(extra) if want_all else (N, FM)


def region_universe(peak_bait, peak_oe, ru_expand, frag_chr, frag_id0=1):
    """getRegionUniverse (chicdiff.R:369-426) restated with NumPy: windows by .expandAvoidBait (:353-367), rows
    with otherEndID beyond the last fragment dropped (:402), rows not on the bait's chromosome dropped (:404-419;
    IDs below the first fragment are NA after the rmap join and drop out with them).
    Returns row_off[m+1], row_bait[R], row_oe[R]; regionID = 1-based peak index."""
    bait = np.asarray(peak_bait, dtype=np.int64)
    oe = np.asarray(peak_oe, dtype=np.int64)
    s = int(ru_expand)
    if np.any(bait == oe):
        raise ValueError("Invalid parameters bait == oe")
    F = len(frag_chr)
    far = np.abs(bait - oe) > s + 1
    lo = np.where(far | (oe < bait), oe - s, bait + 2)
    hi = np.where(far | (oe > bait), oe + s, bait - 2)
    width = hi - lo + 1
    reg = np.repeat(np.arange(len(bait)), width)
    start = np.concatenate([[0], np.cumsum(width)])[:-1]
    f = np.arange(int(width.sum())) - np.repeat(start, width) + np.repeat(lo, width)
    b = np.repeat(bait, width)
    k = f - frag_id0
    ok = (k >= 0) & (k < F)
    chr_ = np.asarray(frag_chr)
    same = np.zeros(len(f), bool)
    same[ok] = chr_[k[ok]] == chr_[(b - frag_id0)[ok]]
    keep = ok & same
    counts = np.bincount(reg[keep], minlength=len(bait))
    row_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return row_off, b[keep].astype(np.int32), f[keep].astype(np.int32)


def countput(reps, frag_start, frag_end, frag_id0=1):
    """chicdiff.R:755-770 for ONE condition: rbind the replicates' CHiCAGO rows, then by (baitID, otherEndID) in
    first-appearance order: Nav = mean(N), Bav = mean(Bmean), score = max(score) (NA if any NA),
    oeID_mid = (start + end) / 2 (unrounded, :711)."""
    bait = np.concatenate([np.asarray(r["baitID"], dtype=np.int64) for r in reps])
    oe = np.concatenate([np.asarray(r["otherEndID"], dtype=np.int64) for r in reps])
    N = np.concatenate([np.asarray(r["N"], dtype=np.float64) for r in reps])
    B = np.concatenate([np.asarray(r["Bmean"], dtype=np.float64) for r in reps])
    sc = np.concatenate([np.asarray(r["score"], dtype=np.float64) for r in reps])
    key = bait * (1 << 32) + oe
    _, first, inv, cnt = np.unique(key, return_index=True, return_inverse=True, return_counts=True)
    order = np.argsort(first, kind="stable")                 # groups in order of first appearance
    rank = np.empty_like(order); rank[order] = np.arange(len(order))
    g = rank[inv]
    G = len(first)
    sumN = np.bincount(g, weights=N, minlength=G)
    sumB = np.zeros(G); np.add.at(sumB, g, B)
    mx = np.full(G, -np.inf); np.maximum.at(mx, g, np.where(np.isnan(sc), -np.inf, sc))
    anyna = np.bincount(g, weights=np.isnan(sc), minlength=G) > 0
    c = cnt[order]
    f0 = first[order]
    return dict(baitID=bait[f0].astype(np.int32), otherEndID=oe[f0].astype(np.int32), Nav=sumN / c, Bav=sumB / c,
                score=np.where(anyna, np.nan, mx),
                oeID_mid=(np.asarray(frag_start, float)[oe[f0] - frag_id0] + np.asarray(frag_end, float)[oe[f0] - frag_id0]) / 2.0)


# ---------------------------------------------------------------------------------------------
# The per-replicate look-up tables of getFullRegionData1 (chicdiff.R:632-634, 659-692, 828-853) the way data.table gets them:
# sort by key, take the first row of every group.  Checker for cd_build_sample_tables (csrc/tables.cu).
# ---------------------------------------------------------------------------------------------

def _first_by(keys, *cols):
    """data.table's x[, list(v = v[1]), by = key] on a table sorted by (baitID, otherEndID): first row per key."""
    u, first = np.unique(keys, return_index=True)
    return (u,) + tuple(np.asarray(c)[first] for c in cols)


def replicate_tables(x, rmap_ids, counts=None, binsize=20000):
    """One replicate's CHiCAGO table (dict of columns: baitID, otherEndID, N, s_j, s_i, tblb, tlb, Tmean, distbin,
    refBinMean) -> the per-fragment look-up tables of cd_sample_tables, exactly the intermediate tables of
    getFullRegionData1: per-bait first (s_j, tblb) (:659), per-other-end first (s_i, tlb) (:668), first Tmean per
    (tblb, tlb) (:680), .chicEstimateDistFun (:696), and the count rows (the .chinput, :828-853, or x's own N)."""
    ids = np.asarray(rmap_ids, dtype=np.int64)
    id0, F = int(ids[0]), len(ids)
    if not np.array_equal(ids, np.arange(id0, id0 + F)):
        raise ValueError("the rmap fragment IDs must be contiguous")
    bait = np.asarray(x["baitID"], dtype=np.int64)
    oe = np.asarray(x["otherEndID"], dtype=np.int64)
    order = np.lexsort((oe, bait))                                   # setkey(x, baitID, otherEndID) (:632)
    bait, oe = bait[order], oe[order]
    col = lambda k: np.asarray(x[k])[order]
    tb_lab, tl_lab = col("tblb"), col("tlb")

    def codes(lab):
        lab = np.asarray(lab, dtype=object)
        na = np.array([v is None or (isinstance(v, float) and np.isnan(v)) for v in lab])
        levels = sorted(set(lab[~na].tolist()))
        lut = {v: k for k, v in enumerate(levels)}
        return np.array([-1 if m else lut[v] for v, m in zip(lab, na)], dtype=np.int32), levels
    tb_code, tb_levels = codes(tb_lab)
    tl_code, tl_levels = codes(tl_lab)
    s_j = np.full(F, np.nan); tblb = np.full(F, -1, np.int32)
    ub, sj1, tb1 = _first_by(bait, col("s_j").astype(np.float64), tb_code)
    s_j[ub - id0] = sj1; tblb[ub - id0] = tb1
    s_i = np.full(F, np.nan); tlb = np.full(F, -1, np.int32)
    o2 = np.lexsort((bait, oe))                                      # first row per otherEndID in (baitID, otherEndID) order
    uo, first = np.unique(oe[o2], return_index=True)
    s_i[uo - id0] = col("s_i").astype(np.float64)[o2][first]
    tlb[uo - id0] = tl_code[o2][first]
    tmean = np.full((max(1, len(tb_levels)), max(1, len(tl_levels))), np.nan)
    tm = col("Tmean").astype(np.float64)
    okc = (tb_code >= 0) & (tl_code >= 0)
    key = tb_code[okc].astype(np.int64) * max(1, len(tl_levels)) + tl_code[okc]
    uk, firstk = np.unique(key, return_index=True)
    tmean.reshape(-1)[uk] = tm[okc][firstk]
    from chicdiff_b200.api import chicEstimateDistFun          # host-side by design (75 points), not part of the check
    distfun = chicEstimateDistFun(col("distbin"), col("refBinMean"), binsize)
    if counts is None:
        cb, co, cn = bait, oe, np.asarray(x["N"])[order]
    else:
        cb = np.asarray(counts["baitID"], dtype=np.int64); co = np.asarray(counts["otherEndID"], dtype=np.int64)
        o3 = np.lexsort((co, cb))
        cb, co, cn = cb[o3], co[o3], np.asarray(counts["N"])[o3]
    inside = (cb >= id0) & (cb < id0 + F)
    cb, co, cn = cb[inside], co[inside], cn[inside]
    cnt_off = np.searchsorted(cb, np.arange(id0, id0 + F + 1)).astype(np.int64)
    return dict(s_j=s_j, tblb=tblb, s_i=s_i, tlb=tlb, tmean=tmean, distfun=distfun, cnt_off=cnt_off,
                cnt_oe=co.astype(np.int32), cnt_N=cn.astype(np.int32), tblb_levels=tb_levels, tlb_levels=tl_levels)


def parse_chinput(data):
    """fread() of a .chinput (chicdiff.R:828): skip the '#' comment line and the header, five columns, NA -> NaN.
    baitID / otherEndID / N are integer columns: a row where one of them is not a whole number (or not a number) is not
    a .chinput row and is dropped, never truncated; numbers may carry a fraction or an exponent ("12.0", "1e5")."""
    def num(tok):
        if tok.upper().startswith("N"):
            return np.nan
        try:
            return float(tok)
        except ValueError:
            return np.nan
    rows = []
    for line in data.decode().splitlines():
        f = line.replace(",", "\t").split()
        if not f or not f[0][0].isdigit():
            continue
        v = [num(t) for t in f[:5]] + [np.nan] * (5 - min(len(f), 5))
        if any(np.isnan(x) or x != np.floor(x) or abs(x) > 2147483647 for x in v[:3]):
            continue
        rows.append(v)
    a = np.array(rows, dtype=np.float64).reshape(-1, 5)
    ln = a[:, 3]
    with np.errstate(invalid="ignore"):
        ln_ok = ~np.isnan(ln) & (ln == np.floor(ln)) & (np.abs(ln) <= 2147483647)
    return dict(baitID=a[:, 0].astype(np.int32), otherEndID=a[:, 1].astype(np.int32), N=a[:, 2].astype(np.int32),
                otherEndLen=np.where(ln_ok, np.nan_to_num(ln), -2147483648).astype(np.int32), distSign=a[:, 4].copy())
