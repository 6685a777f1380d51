"""Known-answer tests of the CPU oracle (oracle/chicdiff_oracle.c).  The reference has no tests and cannot run
here (R), so each restated piece is pinned against an independent computation: SciPy special functions and
distributions, NumPy linear algebra, and bounded scalar / Newton optimisers of the same likelihoods."""
import ctypes as C

import numpy as np
import pytest
from scipy import optimize, special, stats

from chicdiff_b200 import synth
from oracle import oracle as O

X2 = np.array([[1, 0]] * 3 + [[1, 1]] * 3, float)


def _ptr(a):
    return a.ctypes.data


def test_special_functions():
    L = O.lib()
    rng = np.random.default_rng(0)
    xs = np.concatenate([np.exp(rng.uniform(np.log(1e-3), np.log(1e9), 3000)), [0.5, 1, 1.5, 2, 10, 15, 100]])
    for x in xs:
        dg = special.digamma(x)
        assert abs(L.orc_digamma(x) - dg) <= 2e-14 * max(1.0, abs(dg))
        assert abs(L.orc_trigamma(x) - special.polygamma(1, x)) <= 1e-14 * special.polygamma(1, x)
    assert abs(L.orc_trigamma(2.0) - 0.6449340668482264) < 1e-15       # df = 4 (3-vs-3 final fit)
    assert abs(L.orc_trigamma(2.5) - 0.4903577561002349) < 1e-15       # df = 5 (3-vs-3 theta grid)
    for (pr, d1, d2) in [(0.99, 2, 4), (0.99, 3, 13), (0.99, 2, 2), (0.99, 1, 5)]:
        assert abs(L.orc_qf(pr, d1, d2) - stats.f.ppf(pr, d1, d2)) < 1e-9 * stats.f.ppf(pr, d1, d2)
    assert abs(L.orc_qf(0.99, 2, 4) - 18.0) < 1e-10


def test_dnbinom_mu():
    L = O.lib()
    rng = np.random.default_rng(1)
    for _ in range(5000):
        mu = np.exp(rng.uniform(np.log(0.01), np.log(1e4)))
        size = np.exp(rng.uniform(np.log(0.05), np.log(1e5)))
        x = float(rng.poisson(mu * rng.gamma(2, .5)))
        a = L.orc_dnbinom_mu_log(x, size, mu)
        b = stats.nbinom.logpmf(x, size, size / (size + mu))
        assert abs(a - b) <= 1e-9 * max(1.0, abs(b))
    # huge size: Poisson limit, where the plain lgamma formula cancels badly
    for x, mu in [(0.0, 0.0105), (3.0, 2.5), (40.0, 55.0)]:
        a = L.orc_dnbinom_mu_log(x, 1e8, mu)
        b = stats.poisson.logpmf(x, mu)
        assert abs(a - b) < 1e-6 * max(1.0, abs(b))


def _lp(la, y, mu, X, pm=0.0, ps=1.0, use_prior=0):
    return O.lib().orc_log_posterior(la, len(y), X.shape[1], _ptr(X), _ptr(y), _ptr(mu), pm, ps, use_prior, 1)


def _dlp(la, y, mu, X, pm=0.0, ps=1.0, use_prior=0):
    return O.lib().orc_dlog_posterior(la, len(y), X.shape[1], _ptr(X), _ptr(y), _ptr(mu), pm, ps, use_prior, 1)


def test_log_posterior_against_scipy():
    rng = np.random.default_rng(2)
    for _ in range(500):
        mu = np.exp(rng.uniform(np.log(0.5), np.log(1e3), 6))
        y = rng.poisson(mu * rng.gamma(2, .5, 6)).astype(float)
        la = rng.uniform(-10, 2)
        al = np.exp(la)
        r = 1 / al
        ref = np.sum(stats.nbinom.logpmf(y, r, r / (r + mu)) + special.gammaln(y + 1) - y * np.log(mu)) \
            - 0.5 * np.log(np.linalg.det(X2.T @ np.diag(1 / (1 / mu + al)) @ X2))
        assert abs(_lp(la, y, mu, X2) - ref) < 1e-8 * max(1.0, abs(ref))
        h = 1e-5
        num = (_lp(la + h, y, mu, X2) - _lp(la - h, y, mu, X2)) / (2 * h)
        assert abs(_dlp(la, y, mu, X2) - num) < 1e-4 * max(1.0, abs(num))
        # prior terms
        assert abs(_lp(la, y, mu, X2, -1.0, 0.7, 1) - (_lp(la, y, mu, X2) - 0.5 * (la + 1.0) ** 2 / 0.7)) < 1e-9
        assert abs(_dlp(la, y, mu, X2, -1.0, 0.7, 1) - (_dlp(la, y, mu, X2) - (la + 1.0) / 0.7)) < 1e-9


@pytest.fixture(scope="module")
def tiny():
    d = synth.generate("tiny")
    K, FM = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
    return d, K, FM


def test_aggregate_matches_numpy(tiny):
    d, K, FM = tiny
    Kn = np.add.reduceat(d.N_rows.astype(np.int64), d.row_off[:-1], axis=1)
    assert np.array_equal(K, Kn)
    FMn = np.add.reduceat(d.FM_rows, d.row_off[:-1], axis=1)
    assert np.array_equal(np.isnan(FM), np.isnan(FMn))
    ok = ~np.isnan(FMn)
    assert np.max(np.abs(FM[ok] - FMn[ok]) / FMn[ok]) < 1e-14
    assert np.isnan(FM).any(), "generator must exercise NA poisoning (s_j = NA baits)"


def test_aggregate_edge_cases():
    # empty region, single-row region, NA poisoning and integer overflow -> NA_integer_
    row_off = np.array([0, 0, 1, 4, 6], np.int64)
    N = np.array([[5, 1, 2, 3, 2147483647, 1]], np.int32)
    FMr = np.array([[0.5, 1.0, np.nan, 2.0, 1.0, 1.0]])
    K, FM = O.aggregate(row_off, N, FMr)
    assert K.tolist() == [[0, 5, 6, -2147483648]]
    assert FM[0, 0] == 0.0 and FM[0, 1] == 0.5 and np.isnan(FM[0, 2]) and FM[0, 3] == 2.0


def test_na_and_negative_counts_are_refused(tiny):
    """DESeqDataSetFromMatrix (chicdiff.R:1556-1559) stops on NA and negative counts; so does the oracle, whether the NA
    comes from a region sum beyond the int32 range (NA_integer_ = INT32_MIN) or the counts are handed over as they are"""
    import parity
    X, row_off, N, FMr = parity.aggregate_edge_rows()
    K, FM = O.aggregate(row_off, N, FMr)
    assert K[2, 6] == -2147483648
    with pytest.raises(ValueError, match=O.NEGATIVE_COUNTS):
        O.region_test(K, FM, X)
    d, K, FM = tiny
    O.region_test(K, FM, d.X, theta=0.5)                                   # the clean matrix runs
    for v in (-1, -3, -2147483648):
        Kb = K.copy()
        Kb[2, 5] = v
        with pytest.raises(ValueError, match=O.NEGATIVE_COUNTS):
            O.size_factors(Kb)
        with pytest.raises(ValueError, match=O.NEGATIVE_COUNTS):
            O.region_test(Kb, FM, d.X, theta=0.5)
        with pytest.raises(RuntimeError, match=O.NEGATIVE_COUNTS):
            O.deseq(Kb, np.ones(Kb.shape), d.X, prior_var=1.0)


def test_size_factors_against_numpy(tiny):
    d, K, FM = tiny
    sf = O.size_factors(K)
    Kf = K.astype(float)
    with np.errstate(divide="ignore"):
        lg = np.log(Kf).mean(axis=0)
    keep = np.isfinite(lg)
    ref = np.array([np.exp(np.median((np.log(Kf[s][keep & (Kf[s] > 0)]) - lg[keep & (Kf[s] > 0)]))) for s in range(d.S)])
    assert np.max(np.abs(sf - ref) / ref) < 1e-13
    with pytest.raises(ValueError):
        O.size_factors(np.array([[0, 1], [1, 0]], np.int32))


def test_norm_factors_against_numpy(tiny):
    d, K, FM = tiny
    sf = O.size_factors(K)
    with np.errstate(invalid="ignore"):
        m3 = FM / np.exp(np.log(FM).mean(axis=0))
    na = np.isnan(m3).any(axis=0)
    m3[:, na] = sf[:, None]
    assert na.any()
    assert np.allclose(O.norm_factors(FM, sf, "fullmean"), m3, rtol=1e-13, atol=0)
    for th in (0.0, 0.25, 1.0):
        sc = m3 * (1 - th) + sf[:, None] * th
        sc = sc / np.exp(np.log(sc).mean(axis=0))
        assert np.allclose(O.norm_factors(FM, sf, "combined", th), sc, rtol=1e-13, atol=0)
    assert np.allclose(O.norm_factors(FM, sf, "standard"), np.repeat(sf[:, None], d.n, axis=1))


@pytest.fixture(scope="module")
def tiny_fit(tiny):
    d, K, FM = tiny
    return O.region_test(K, FM, d.X)


def test_pipeline_runs_and_is_sane(tiny, tiny_fit):
    d, K, FM = tiny
    r = tiny_fit
    assert r["theta"] in (0, .25, .5, .75, 1)
    assert len(r["deviances"]) == 5 and np.all(np.isfinite(r["deviances"]))
    assert r["trend_a0"] > 0 and r["trend_a1"] > 0
    assert r["dispPriorVar"] >= 0.25
    nz = r["allZero"] == 0
    assert nz.all()
    for k in ("dispGeneEst", "dispFit", "dispMAP", "dispersion", "pvalue", "stat", "deviance"):
        assert np.all(np.isfinite(r[k][nz])), k
    assert np.all((r["dispersion"] >= 1e-8) & (r["dispersion"] <= 10))
    assert np.all((r["pvalue"] >= 0) & (r["pvalue"] <= 1))
    # true effects are recovered: strong positive correlation on regions with a planted fold change
    planted = d.true_lfc != 0
    assert np.corrcoef(r["beta"][1][planted], d.true_lfc[planted])[0, 1] > 0.6


def test_gene_dispersion_is_a_maximum_of_the_cox_reid_likelihood(tiny, tiny_fit):
    """fitDisp's answer must be the maximiser of the posterior it climbs (checked with a bounded scalar solver)."""
    d, K, FM = tiny
    r = tiny_fit
    conv = (r["dispGeneIter"] > 1) & (r["dispGeneIter"] < 100) & ((r["flags"] & (O.FLAG_GENE_GRID | O.FLAG_GENE_NOINCREASE)) == 0)
    idx = np.flatnonzero(conv & (r["dispGeneEst"] > 1e-6) & (r["dispGeneEst"] < 9.9))[:150]
    assert len(idx) > 50
    worse = 0
    for i in idx:
        y = K[:, i].astype(float)
        mu = np.ascontiguousarray(r["mu"][:, i])
        f = lambda la: -_lp(la, y, mu, d.X)
        la_hat = np.log(r["dispGeneEst"][i])
        opt = optimize.minimize_scalar(f, bounds=(la_hat - 3, la_hat + 3), method="bounded", options=dict(xatol=1e-10))
        # the line search stops when the posterior gains < 1e-6: it sits within that of the optimum
        assert f(la_hat) - opt.fun < 1e-4
        worse += f(la_hat) - opt.fun > 2e-6
    assert worse <= 0.1 * len(idx)


def test_irls_beta_maximises_the_penalised_likelihood(tiny, tiny_fit):
    d, K, FM = tiny
    r = tiny_fit
    L = O.lib()
    lam = 1e-6 / np.log(2) ** 2
    idx = np.flatnonzero(r["betaConv"] == 1)[:60]
    for i in idx:
        y = K[:, i].astype(float)
        nf = r["nf"][:, i]
        alpha = r["dispersion"][i]

        def negll(b):
            mu = nf * np.exp(d.X @ b)
            return -sum(L.orc_dnbinom_mu_log(yy, 1 / alpha, m) for yy, m in zip(y, mu)) + 0.5 * lam * np.sum(b ** 2)
        b_hat = r["beta"][:, i] * np.log(2)
        if np.any(nf * np.exp(d.X @ b_hat) < 0.5):
            continue                      # the minmu floor changes the fixed point (all-zero condition)
        opt = optimize.minimize(negll, b_hat, method="Nelder-Mead", options=dict(xatol=1e-9, fatol=1e-12, maxiter=4000))
        assert negll(b_hat) - opt.fun < 1e-6
        # standard error = sqrt of the sandwich diagonal ~ inverse Fisher information
        mu = nf * np.exp(d.X @ b_hat)
        W = mu / (1 + alpha * mu)
        cov = np.linalg.inv(d.X.T @ np.diag(W) @ d.X + lam * np.eye(2))
        assert abs(r["betaSE"][1, i] - np.sqrt(cov[1, 1]) / np.log(2)) < 1e-5 * r["betaSE"][1, i]


def test_trend_is_the_gamma_glm_fit(tiny_fit):
    """parametricDispersionFit: at convergence (a0, a1) solve the Gamma(identity) score equations on the kept rows."""
    r = tiny_fit
    use = r["dispGeneEst"] > 1e-6
    m, dsp = r["baseMean"][use], r["dispGeneEst"][use]
    a0, a1 = r["trend_a0"], r["trend_a1"]
    ratio = dsp / (a0 + a1 / m)
    good = (ratio > 1e-4) & (ratio < 15)
    mu = a0 + a1 / m[good]
    score0 = np.sum((dsp[good] - mu) / mu ** 2)
    score1 = np.sum((dsp[good] - mu) / mu ** 2 / m[good])
    scale = np.sum(1 / mu ** 2)
    assert abs(score0) / scale < 1e-3 and abs(score1) / scale < 1e-3
    resid = np.log(r["dispGeneEst"][use]) - np.log(r["dispFit"][use])
    mad = 1.4826 * np.median(np.abs(resid - np.median(resid)))
    assert abs(mad ** 2 - r["varLogDispEsts"]) < 1e-12
    assert abs(r["dispPriorVar"] - max(r["varLogDispEsts"] - special.polygamma(1, 2.0), 0.25)) < 1e-12


def test_theta_grid_na_and_intercept_shortcut(tiny):
    d, K, FM = tiny
    K0 = K.copy()
    K0[:, 7] = 0                                  # an all-zero region poisons the theta-grid sum (chicdiff.R:1647)
    with pytest.raises(ValueError):
        O.region_test(K0, FM, d.X)
    r = O.region_test(K0, FM, d.X, theta=0.5)     # ... so theta is inherited for such sets (chicdiff.R:331)
    assert r["allZero"][7] == 1 and np.isnan(r["pvalue"][7]) and np.isnan(r["dispersion"][7])
    # theta = 1 / 0 collapse to standard / fullmean (chicdiff.R:1511-1521)
    sf = O.size_factors(K)
    r1 = O.region_test(K, FM, d.X, theta=1)
    assert np.allclose(r1["nf"], np.repeat(sf[:, None], d.n, axis=1))


def test_results_cooks_and_filtering(tiny, tiny_fit):
    d, K, FM = tiny
    res = O.results(tiny_fit, K, d.X)
    assert abs(res["cooksCutoff"] - 18.0) < 1e-9
    ok = ~np.isnan(res["padj"])
    assert ok.sum() > 0 and np.all(res["padj"][ok] >= res["pvalue"][ok] - 1e-15)
    assert np.all(res["baseMean"][~ok & ~np.isnan(res["pvalue"])] < res["filterThreshold"])


def test_region_universe_against_generator(tiny):
    """two independent restatements of getRegionUniverse (the generator's and oracle.region_universe) agree"""
    d, K, FM = tiny
    row_off, row_bait, row_oe = O.region_universe(d.region_bait, d.region_seed, 5, d.frag_chr)
    assert np.array_equal(row_off, d.row_off) and np.array_equal(row_bait, d.row_bait) and np.array_equal(row_oe, d.row_oe)
    d23 = synth.generate("c3", n_regions=30000)            # 23 chromosomes: exercises the same-chromosome trimming
    row_off, row_bait, row_oe = O.region_universe(d23.region_bait, d23.region_seed, 5, d23.frag_chr)
    assert np.array_equal(row_off, d23.row_off) and np.array_equal(row_oe, d23.row_oe)
    with pytest.raises(ValueError):
        O.region_universe([10], [10], 5, d.frag_chr)


def test_replicate_tables_from_chicago_table(tiny):
    """Host adapter: the look-up tables built from a reference-shaped CHiCAGO table (per-bait / per-other-end
    first values, Tmean table, .chicEstimateDistFun) equal the generator's own tables wherever the table says
    anything, and the distance function is recovered from its binned samples."""
    from chicdiff_b200 import api
    d, K, FM = tiny
    ids = np.arange(1, len(d.frag_chr) + 1)
    for s in (0, 3):
        x = synth.chicago_table(d, s)
        t = O.replicate_tables(x, ids, synth.chinput_table(d, s))
        g = d.extra["tables"][s]
        baits = np.unique(x["baitID"]); oes = np.unique(x["otherEndID"])
        assert np.array_equal(np.isnan(t["s_j"][baits - 1]), np.isnan(g["s_j"][baits - 1]))
        okb = ~np.isnan(g["s_j"][baits - 1])
        assert np.array_equal(t["s_j"][baits - 1][okb], g["s_j"][baits - 1][okb])
        assert np.array_equal(t["s_i"][oes - 1], g["s_i"][oes - 1])
        assert np.isnan(t["s_i"][np.setdiff1d(ids, oes) - 1]).all()
        assert np.array_equal(t["tblb"][baits - 1], g["tblb"][baits - 1]) and np.array_equal(t["tlb"][oes - 1], g["tlb"][oes - 1])
        seen = ~np.isnan(t["tmean"])
        assert seen.sum() >= 20 and np.array_equal(t["tmean"][seen], g["tmean"][seen])
        assert np.array_equal(t["cnt_off"], g["cnt_off"]) and np.array_equal(t["cnt_N"], g["cnt_N"])
        assert np.max(np.abs(t["distfun"][:4] - g["distfun"][:4])) < 1e-7           # cubic recovered from 75 bin means
        assert abs(t["distfun"][4] - np.log(10000)) < 1e-12
    # .chicEstimateDistFun on its own: C1 continuation at both ends
    p = api.chicEstimateDistFun(x["distbin"], x["refBinMean"])
    f = lambda l: p[0] + p[1] * l + p[2] * l * l + p[3] * l ** 3
    for l, (a0, b0) in ((p[4], p[6:8]), (p[5], p[8:10])):
        assert abs(f(l) - (a0 + b0 * l)) < 1e-9
