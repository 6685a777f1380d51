"""Per-region parity of the CUDA path (through the C ABI) with the CPU oracle: the comparison the GPU tests assert on
and scripts/parity_strict.py prints.  Test infrastructure (imports the oracle).

The bar (BASELINE.json north_star): aggregated counts bit-exact; dispersions, log2FC and p-values within 1e-6 relative,
per region.  Two properties of the reference ALGORITHM shape how that bar can be checked at scale:

1. The dispersion trend and the MAD are global fits.  One region whose gene-wise estimate differs moves the trend
   coefficients by ~1/n of its weight and with them every region's dispFit, MAP estimate, standard error and
   p-value (amplified by z^2 in the tail).  Per-region agreement is therefore checked on a second run of the CUDA path
   that is handed the oracle's global scalars (theta, trend coefficients, varLogDispEsts, dispPriorVar) through
   cd_options -- every per-region number then depends on that region's data only -- while the free run (each side
   fitting its own trend) is held to what the coupling allows: identical theta, identical significance calls,
   coupling below 1e-4.

2. DESeq2's fitDisp compares log-posteriors that can differ by less than the rounding error of their own
   evaluation (Armijo test, `change < 1e-6` stop test, "did the search raise the posterior" test, the arg max of
   fitDispGrid over a plateau).  Which branch such a search takes is decided by rounding: the oracle itself takes
   the other branch when built with fused multiply-adds or with a long-double posterior
   (scripts/oracle_flip_evidence.py, profiles/r02_oracle_flip_evidence.txt).  The oracle records, per region, the
   smallest margin of all those comparisons in units of the rounding error (fit_disp_row in chicdiff_oracle.c).
   Regions whose margin is at least MARGIN_NOISE rounding errors ("clean") must agree to 1e-6 in EVERY column, all of
   them.  Regions below it must still agree except for a bounded number of branch flips (<= FLIP_BOUND * n + 2), which
   are listed.  Gene-wise estimates below 1e-6 (which DESeq2 excludes from the trend) are rounding noise of
   lgamma(1/alpha) at 1/alpha >= 1e6 in the reference itself: both sides must be below 1e-6, not equal.
"""
import types

import numpy as np

from chicdiff_b200 import engine
from oracle import oracle as O

TOL = 1e-6
MARGIN_NOISE = 64.0
FLIP_BOUND = 1e-4
COUPLING_BOUND = 1e-4


def rel(a, b, scale=None):
    a, b = np.asarray(a, float), np.asarray(b, float)
    ref = np.abs(b) if scale is None else np.maximum(np.abs(b), scale)
    with np.errstate(invalid="ignore", divide="ignore"):
        e = np.abs(a - b) / np.maximum(ref, 1e-300)
    e[(np.isnan(a) & np.isnan(b)) | (a == b)] = 0
    e[np.isnan(e)] = np.inf          # NA on one side only
    return e


def columns(r, ro, p):
    """(name, CUDA values, oracle values, scale) of every compared per-region column.  maxCooks decides the Cook's
    filter of results(); the coefficients other than the tested one (intercept, covariates) are compared like it, each
    on the scale of its own standard error."""
    floor = ro["dispGeneEst"] < 1e-6
    with np.errstate(invalid="ignore"):
        ge = np.where(floor & (r["dispGeneEst"] < 1e-6 * (1 + 1e-9)), ro["dispGeneEst"], r["dispGeneEst"])
    cols = [("dispGeneEst", ge, ro["dispGeneEst"], None),
            ("dispFit", r["dispFit"], ro["dispFit"], None), ("dispMAP", r["dispMAP"], ro["dispMAP"], None),
            ("dispersion", r["dispersion"], ro["dispersion"], None),
            ("log2FoldChange", r["log2FoldChange"], ro["beta"][p - 1], ro["betaSE"][p - 1]),
            ("lfcSE", r["lfcSE"], ro["betaSE"][p - 1], None), ("stat", r["stat"], ro["stat"], 1.0),
            ("pvalue", r["pvalue"], ro["pvalue"], None), ("deviance", r["deviance"], ro["deviance"], None),
            ("maxCooks", r["maxCooks"], ro["maxCooks"], None)]
    for j in range(p - 1):
        cols += [("beta[%d]" % j, r["beta"][j], ro["beta"][j], ro["betaSE"][j]), ("betaSE[%d]" % j, r["betaSE"][j], ro["betaSE"][j], None)]
    return cols


def run_three(d, prior=None, prior_grid=None, oracle=None, **kw):
    """free CUDA run, oracle run (with decision margins), CUDA run with the oracle's global scalars.
    kw: norm / theta / theta_grid / disp_grid_len as for Engine.region_test.  oracle: a result of an earlier oracle run
    on the same inputs and options, to be reused."""
    e = engine.Engine(0)
    e.set_design(d.X)
    e.set_regions(d.row_off)
    for s in range(d.S):
        e.set_sample_rows(s, d.N_rows[s], d.FM_rows[s])
    K, FM = e.aggregate()
    Ko, FMo = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
    return _fits(e, K, FM, Ko, FMo, d.X, prior, prior_grid, oracle, kw)


def run_three_aggregated(K, FM, X, prior=None, prior_grid=None, oracle=None, **kw):
    """run_three on aggregated matrices (K int32 S x n, FM float64 S x n) handed to the device with
    Engine.set_aggregated; the result's "inputs" (X, S, n) stands in for the data set in compare()."""
    K = np.ascontiguousarray(K, dtype=np.int32)
    FM = np.ascontiguousarray(FM, dtype=np.float64)
    e = engine.Engine(0)
    e.set_design(X)
    e.set_aggregated(K, FM)
    t = _fits(e, K, FM, K, FM, X, prior, prior_grid, oracle, kw)
    t["inputs"] = types.SimpleNamespace(X=np.asarray(X, float), S=K.shape[0], n=K.shape[1])
    return t


def oracle_region_test(K, FM, X, prior=None, prior_grid=None, **kw):
    """the oracle's run that run_three compares with (decision margins included); kw as for run_three"""
    nan = float("nan")
    okw = {k: v for k, v in kw.items() if k in ("norm", "theta", "theta_grid")}
    if "disp_grid_len" in kw:
        okw["grid_n"] = kw["disp_grid_len"]
    return O.region_test(K, FM, X, prior_var=nan if prior is None else prior, prior_var_grid=nan if prior_grid is None else prior_grid,
                         margins=True, **okw)


def aggregate_edge_rows():
    """(X, row_off, N, FM rows) of a 2-vs-2 set whose regions are empty, single-row, wider than the aggregation's
    shared-memory chunk, NA-poisoned (FullMean) or overflowing: region 6 sums to more than 2^31-1, so its count is
    NA_integer_ (INT32_MIN) after the aggregation, and the region test must refuse the matrix."""
    X = np.array([[1, 0], [1, 0], [1, 1], [1, 1]], float)
    widths = np.array([0, 1, 3, 9000, 0, 11, 2, 7000, 1], np.int64)
    row_off = np.concatenate([[0], np.cumsum(widths)])
    R = int(row_off[-1])
    rng = np.random.default_rng(0)
    N = rng.integers(0, 50, (4, R)).astype(np.int32)
    FMr = rng.random((4, R)) + 0.01
    FMr[1, 5] = np.nan
    N[2, row_off[6]] = 2147483647
    N[2, row_off[6] + 1] = 5
    return X, row_off, N, FMr


def _fits(e, K, FM, Ko, FMo, X, prior, prior_grid, oracle, kw):
    r = e.region_test(disp_prior_var=prior, disp_prior_var_grid=prior_grid, **kw)
    ro = oracle if oracle is not None else oracle_region_test(Ko, FMo, X, prior, prior_grid, **kw)
    kw2 = dict(kw)
    if ro["deviances"] is not None:
        # the grid's winner is fitted with norm = "combined" at that theta (chicdiff.R:1666-1669); a one-point grid says the
        # same (an explicit theta of 0 or 1 would switch to "fullmean" / "standard", :1511-1521)
        kw2.pop("theta", None)
        kw2["theta_grid"] = [ro["theta"]]
    rs = e.region_test(disp_prior_var=ro["dispPriorVar"], disp_prior_var_grid=prior_grid, trend=(ro["trend_a0"], ro["trend_a1"]),
                       var_log_disp=ro["varLogDispEsts"], **kw2)
    launches = e.launch_count()
    e.close()
    return dict(K=K, FM=FM, Ko=Ko, FMo=FMo, free=r, oracle=ro, shared=rs, launches=launches)


def compare(d, t, out=None):
    """-> summary dict; appends report lines to `out` (a list) when given"""
    say = (lambda s: out.append(s)) if out is not None else (lambda s: None)
    r, ro, rs, K, Ko, FM, FMo = t["free"], t["oracle"], t["shared"], t["K"], t["Ko"], t["FM"], t["FMo"]
    p = d.X.shape[1]
    n = d.n
    S = {}
    S["counts_exact"] = bool(np.array_equal(K, Ko))
    S["fullmean_na_equal"] = bool(np.array_equal(np.isnan(FM), np.isnan(FMo)))
    okm = ~np.isnan(FMo)
    S["fullmean_max_rel"] = float(rel(FM[okm], FMo[okm]).max()) if okm.any() else 0.0           # (a FullMean may be 0)
    S["sf_max_rel"] = float(np.max(np.abs(r["sizeFactors"] - ro["sizeFactors"]) / ro["sizeFactors"]))
    S["theta"] = (r["theta"], ro["theta"])
    S["dev_max_rel"] = 0.0 if ro["deviances"] is None else float(np.max(np.abs(r["deviances"] - ro["deviances"]) / np.abs(ro["deviances"])))
    S["nf_max_rel"] = float(rel(r["normFactors"], ro["nf"]).max())
    S["baseMean_max_rel"] = float(rel(r["baseMean"], ro["baseMean"]).max())
    S["coupling"] = float(max(abs(r["trend_a0"] - ro["trend_a0"]) / ro["trend_a0"], abs(r["trend_a1"] - ro["trend_a1"]) / ro["trend_a1"]))
    S["vld_rel"] = float(abs(r["varLogDispEsts"] - ro["varLogDispEsts"]) / ro["varLogDispEsts"])
    say("   aggregated counts bit-exact: %s ; FullMean sums max rel %.2e ; size factors max rel %.2e ; theta %s / %s ; "
        "theta-grid deviances max rel %.2e" % (S["counts_exact"], S["fullmean_max_rel"], S["sf_max_rel"], r["theta"], ro["theta"], S["dev_max_rel"]))
    say("   free run: trend coefficients rel diff %.2e ; varLogDispEsts rel diff %.2e ; dispPriorVar %.9g / %.9g" % (
        S["coupling"], S["vld_rel"], r["dispPriorVar"], ro["dispPriorVar"]))

    gm, mm = ro["geneMargin"], ro["mapMargin"]
    with np.errstate(invalid="ignore"):
        noisy = (gm < MARGIN_NOISE) | (mm < MARGIN_NOISE)
    allzero = np.isnan(gm)
    clean = ~noisy & ~allzero
    S["n"], S["n_clean"], S["n_noisy"] = int(n), int(clean.sum()), int(noisy.sum())
    say("-- shared global scalars (theta, trend, varLogDispEsts, dispPriorVar from the oracle): per-region agreement")
    say("   oracle decision margins below %g rounding errors: gene-wise search %d rows (%d of them with an estimate above the 1e-6 "
        "floor), MAP search %d rows, either %d of %d" % (MARGIN_NOISE, int((gm < MARGIN_NOISE).sum()),
                                                        int(((gm < MARGIN_NOISE) & (ro["dispGeneEst"] >= 1e-6)).sum()),
                                                        int((mm < MARGIN_NOISE).sum()), S["n_noisy"], n))
    say("   %-16s %10s %9s %9s %13s | %-24s | %s" % ("column", "max rel", "#>1e-6", "#>1e-5", "frac<=1e-6", "clean rows: max rel, #>1e-6",
                                                       "rounding-decided rows: #>1e-6"))
    bad = np.zeros(n, bool)
    S["clean_bad"], S["clean_max_rel"] = {}, {}
    errs = {}
    for nm, a, b, sc in columns(rs, ro, p):
        e = rel(a, b, sc)
        errs[nm] = e
        bad |= e > TOL
        S["clean_bad"][nm] = int((e[clean] > TOL).sum())
        S["clean_max_rel"][nm] = float(e[clean].max()) if clean.any() else 0.0
        say("   %-16s %10.2e %9d %9d %13.8f | %10.2e %13d | %d" % (nm, e.max(), (e > TOL).sum(), (e > 1e-5).sum(), (e <= TOL).mean(),
                                                                  S["clean_max_rel"][nm], S["clean_bad"][nm], int((e[noisy] > TOL).sum())))
    S["na_pattern_equal"] = bool(np.array_equal(np.isnan(rs["pvalue"]), np.isnan(ro["pvalue"])))
    S["rows_bad"] = int(bad.sum())
    S["rows_bad_clean"] = int((bad & clean).sum())
    S["rows_bad_allzero"] = int((bad & allzero).sum())
    idx = np.flatnonzero(bad)
    say("   regions with any column beyond 1e-6: %d of %d (%.2e); among the %d clean-margin regions: %d" % (
        len(idx), n, len(idx) / max(n, 1), S["n_clean"], S["rows_bad_clean"]))
    for i in idx[:60]:
        say("      region %8d  margin gene %-9.3g MAP %-9.3g | geneEst %.6e / %.6e trips %d/%d | MAP %.6e / %.6e trips %d/%d | flags %d/%d | "
            "p rel %.2e z %.2f" % (i, gm[i], mm[i], rs["dispGeneEst"][i], ro["dispGeneEst"][i], rs["dispGeneIter"][i], ro["dispGeneIter"][i],
                                   rs["dispMAP"][i], ro["dispMAP"][i], rs["dispIter"][i], ro["dispIter"][i], rs["flags"][i] & 63, ro["flags"][i],
                                   errs["pvalue"][i], ro["stat"][i]))
    S["betaIter_equal"] = float((rs["betaIter"] == ro["betaIter"]).mean())
    S["flags_equal"] = float(((rs["flags"] & 63) == ro["flags"]).mean())
    say("   trip counts equal: dispGeneIter %.6f  dispIter %.6f  betaIter %.6f ; flags equal %.6f" % (
        (rs["dispGeneIter"] == ro["dispGeneIter"]).mean(), (rs["dispIter"] == ro["dispIter"]).mean(), S["betaIter_equal"], S["flags_equal"]))

    say("-- free run (each side fits its own trend and MAD): what the coupling through the global fits does to the same columns")
    say("   %-16s %10s %9s %9s %13s" % ("column", "max rel", "#>1e-6", "#>1e-5", "frac<=1e-6"))
    for nm, a, b, sc in columns(r, ro, p):
        e = rel(a, b, sc)
        say("   %-16s %10.2e %9d %9d %13.8f" % (nm, e.max(), (e > TOL).sum(), (e > 1e-5).sum(), (e <= TOL).mean()))
    adj = engine.results_adjust(r["baseMean"], r["maxCooks"], r["flags"], r["pvalue"], d.S, p)
    res_o = O.results(ro, Ko, d.X)
    with np.errstate(invalid="ignore"):
        sg, so = adj["padj"] < 0.05, res_o["padj"] < 0.05
        near = np.abs(res_o["padj"] - 0.05) < 1e-5
    S["padj_na_equal"] = bool(np.array_equal(np.isnan(adj["padj"]), np.isnan(res_o["padj"])))
    S["sig"] = (int(sg.sum()), int(so.sum()))
    S["sig_differ"] = int(((sg | near) != (so | near)).sum())
    S["filter_index"] = (int(adj["filterIndex"]), int(res_o["filterIndex"]) + 1)
    say("   results(): filter index %d / %d ; padj NA pattern equal %s ; significant calls (padj < 0.05): %d / %d, differing %d" % (
        S["filter_index"][0], S["filter_index"][1], S["padj_na_equal"], S["sig"][0], S["sig"][1], S["sig_differ"]))
    return S


def assert_parity(S, all_rows=False, noisy_share=0.0):
    """the gate.  all_rows: no branch flip is tolerated at all (small inputs).  noisy_share: flips also allowed for this
    share of the rounding-decided rows (inputs where a large part of the searches is decided by rounding)"""
    assert S["counts_exact"], "aggregated counts must be bit-exact"
    assert S["fullmean_na_equal"] and S["fullmean_max_rel"] < 1e-14
    assert S["sf_max_rel"] < 1e-12
    assert S["theta"][0] == S["theta"][1]
    assert S["dev_max_rel"] < 1e-5
    assert S["nf_max_rel"] <= TOL and S["baseMean_max_rel"] <= TOL
    # per region, with shared global scalars: every clean-margin region within 1e-6 in every column
    assert S["na_pattern_equal"] and S["rows_bad_allzero"] == 0
    assert S["rows_bad_clean"] == 0, ("clean-margin regions beyond 1e-6", S["clean_bad"], S["clean_max_rel"])
    # rounding-decided regions: a bounded number of branch flips
    limit = 0 if all_rows else int(FLIP_BOUND * S["n"] + noisy_share * S["n_noisy"]) + 2
    assert S["rows_bad"] <= limit, ("branch flips", S["rows_bad"], limit)
    assert S["betaIter_equal"] >= 1.0 - 2 * FLIP_BOUND - noisy_share * S["n_noisy"] / max(S["n"], 1)
    # free run: bounded coupling, same calls
    assert S["coupling"] < (1e-9 if all_rows else COUPLING_BOUND), ("trend coefficients", S["coupling"])
    assert S["padj_na_equal"] and S["sig_differ"] == 0, "significant-interaction calls differ"
    assert S["filter_index"][0] == S["filter_index"][1]
