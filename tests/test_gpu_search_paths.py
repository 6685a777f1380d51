"""The rare paths of the dispersion line search (csrc/dispersion.cu) and counts at the edges of the device arithmetic,
against the CPU oracle.

The parity inputs of tests/test_gpu_parity.py never park a MAP search (no MAP search there runs more than 24 trips),
never refit one on the grid, never fill the park and pick the lane-per-region resume kernel only for S = 6, p <= 2
without a prior.  A flat MAP prior (a large caller-supplied disp_prior_var, which DESeq2 accepts for any design) makes
the MAP searches as long as the gene-wise ones, so ordinary data reach all of these paths.  Every case first shows from
the oracle alone that its path is taken, then holds the CUDA path to parity.assert_parity (tests/parity.py) and
compares the number of MAP grid refits.
"""
import copy

import numpy as np
import pytest

import parity
from chicdiff_b200 import engine, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TRIP_CAP = 24                     # kFitDispTripCap: pass 1 parks a search still running after this many trips
INT32_MIN = -2147483648


def park_capacity(nv):
    """regions one line-search launch can park (cd_region_test)"""
    return nv // 4 + 4096


def lane_resume(nv, S):
    """whether launch_fit_disp resumes the parked searches one per lane (True) or sample-parallel in tiles (False)"""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    G = 8 if S <= 8 else (16 if S <= 16 else 32)
    return nv * 0.04 * G > sms * 1024.0


_DATA, _ORACLE = {}, {}


def data(name, p4=False, **kw):
    """synth.generate, once per session; p4: the 4-column design of test_other_designs (intercept, two nuisance
    covariates, condition) on the same counts"""
    key = (name, tuple(sorted(kw.items())))
    if key not in _DATA:
        _DATA[key] = synth.generate(name, **kw)
    d = _DATA[key]
    if p4:
        d = copy.copy(d)
        S = d.S
        d.X = np.column_stack([np.ones(S), np.arange(S) % 2, (np.arange(S) // 2) % 2, d.X[:, -1]]).astype(float)
    return d


def oracle(key, d, prior=None, prior_grid=None, **kw):
    """the oracle's run of a case, once per session"""
    if key not in _ORACLE:
        K, FM = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
        _ORACLE[key] = parity.oracle_region_test(K, FM, d.X, prior, prior_grid, **kw)
    return _ORACLE[key]


def map_grid(ro):
    return int(((ro["flags"] & O.FLAG_MAP_GRID) != 0).sum())


# With a flat prior (1e3) the MAP posterior is nearly flat, and far more of the search's comparisons are decided by
# rounding (oracle margin below parity.MARGIN_NOISE) than with an estimated prior: 4-6 % of the regions here.  Every
# clean-margin region must still agree to 1e-6; branch flips stay confined to the rounding-decided regions (measured on
# a B200: 0.6-3 % of them), and are bounded by 5 % of those.  The same holds for the crafted regions of
# test_edge_counts_through_set_aggregated, whose huge and identical counts are rounding-decided by construction.
FLAT_PRIOR_NOISY_SHARE = 0.05


def check(d, t, noisy_share=0.0):
    """parity gate, then the MAP search paths of the shared-scalar run against the oracle's"""
    report = []
    S = parity.compare(d, t, report)
    try:
        parity.assert_parity(S, noisy_share=noisy_share)
    except AssertionError:
        print("\n".join(report))
        raise
    ro, rs = t["oracle"], t["shared"]
    bound = int(parity.FLIP_BOUND * d.n) + 2
    assert abs(rs["n_map_grid"] - map_grid(ro)) <= bound, (rs["n_map_grid"], map_grid(ro))
    assert abs(int((rs["dispIter"] > TRIP_CAP).sum()) - int((ro["dispIter"] > TRIP_CAP).sum())) <= bound
    return S


def run(d, ro, prior=None, prior_grid=None, **kw):
    t = parity.run_three(d, prior=prior, prior_grid=prior_grid, oracle=ro, **kw)
    check(d, t, FLAT_PRIOR_NOISY_SHARE if prior == 1e3 else 0.0)
    return t


# ---- MAP park, tile resume, grid refit -------------------------------------------------------------------------------

@pytest.mark.parametrize("prior", [10.0, 1e3])
def test_map_park_tile_resume_and_grid_refit(prior):
    """c1 (2-vs-2, 28 k regions) at theta = 0.5: thousands of MAP searches are parked and resumed by the tile kernel with
    the prior reloaded; with the flat prior thousands more reach 100 trips and are refitted on the grid around dispFit"""
    d = data("c1")
    ro = oracle(("c1", prior), d, prior=prior, theta=0.5)
    parked = int((ro["dispIter"] > TRIP_CAP).sum())
    assert 1000 < parked < park_capacity(d.n) and not lane_resume(d.n, d.S)
    assert map_grid(ro) >= (50 if prior == 10.0 else 5000)
    run(d, ro, prior=prior, theta=0.5)


@pytest.mark.parametrize("grid_len", [pytest.param(2, marks=pytest.mark.xfail(strict=True, reason=(
                                          "open finding: with two grid points, 92 of 28 470 rounding-decided regions land on "
                                          "the other grid point than the oracle's, and 49 significance calls of the free "
                                          "run differ"))), 7, 32])
def test_map_grid_refit_lengths(grid_len):
    """fitDispGrid with disp_grid_len points: the ends of the accepted range and a length that is not the default"""
    d = data("c1")
    ro = oracle(("c1", 1e3, grid_len), d, prior=1e3, theta=0.5, disp_grid_len=grid_len)
    assert map_grid(ro) > 5000
    run(d, ro, prior=1e3, theta=0.5, disp_grid_len=grid_len)


def test_park_overflow():
    """c2 at full size with a flat prior: more MAP searches run past the trip cap than the park holds, so lanes whose
    slot is taken keep searching in the first pass"""
    d = data("c2")
    ro = oracle(("c2", 1e3), d, prior=1e3, theta=0.5)
    assert int((ro["dispIter"] > TRIP_CAP).sum()) > park_capacity(d.n)
    assert not lane_resume(d.n, d.S)
    run(d, ro, prior=1e3, theta=0.5)


# ---- lane-per-region resume with a prior -----------------------------------------------------------------------------

def test_lane_resume_theta_grid_with_prior():
    """the theta grid of c2 (5 fits of ~100 k regions = ~500 k virtual regions, design ~ 1) with a flat prior: the MAP
    searches of the grid are resumed one per lane, each with the prior of its own fit.  Only the grid's total deviances
    leave the library; they decide theta."""
    d = data("c2")
    assert lane_resume(5 * d.n, d.S)
    # one fit of the grid, from the oracle: its MAP searches do run past the trip cap
    K, FM = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
    nf = O.norm_factors(FM, O.size_factors(K), "combined", 0.5)
    r1 = O.deseq(K, nf, np.ones((d.S, 1)), prior_var=1e3)
    assert int((r1["dispIter"] > TRIP_CAP).sum()) > 1000
    ro = oracle(("c2 grid", 1e3), d, prior=1e3, prior_grid=1e3)
    assert ro["deviances"] is not None
    run(d, ro, prior=1e3, prior_grid=1e3)


@pytest.mark.parametrize("case", ["c2_500k_p2", "c4_8v8_p3",
                                  pytest.param("c4_8v8_p4", marks=pytest.mark.xfail(strict=True, reason=(
                                      "open finding: with p = 4 and the flat prior, 11 of 245 817 clean-margin regions get "
                                      "coefficients that differ from the oracle's (dispersions agree); not yet explained"))),
                                  "16v16_p2"])
def test_lane_resume_with_prior(case):
    """the final fit resumed one region per lane: S = 4 (p = 2), S = 16 (p = 3 and p = 4) and S = 32"""
    d = {"c2_500k_p2": lambda: data("c2", n_regions=500000),
         "c4_8v8_p3": lambda: data("c4", n_regions=260000),
         "c4_8v8_p4": lambda: data("c4", p4=True, n_regions=260000),
         "16v16_p2": lambda: data("c3", n_regions=140000, reps=(16, 16))}[case]()
    assert d.X.shape[1] == int(case[-1])
    ro = oracle((case, 1e3), d, prior=1e3, theta=0.5)
    assert lane_resume(d.n, d.S)
    assert int((ro["dispIter"] > TRIP_CAP).sum()) > 100 and map_grid(ro) > 100
    run(d, ro, prior=1e3, theta=0.5)


# ---- counts at the edges, injected into aggregated matrices ----------------------------------------------------------

def crafted_regions(K, FM, rng):
    """a few hundred regions whose counts sit where the device arithmetic changes branch, with FullMean columns taken
    from random regions of the base set; -> (K, FM, dict of column indices per kind)"""
    S = K.shape[0]
    cols, kinds = [], {}

    def add(kind, k):
        kinds.setdefault(kind, []).append(len(cols))
        cols.append(np.asarray(k, np.int64))
    # the end of the log-factorial table (wald.cu: kLfactN = 4096 entries)
    for k in ([4095, 4096, 4097, 4095], [4096, 4096, 4096, 4097], [4097, 4095, 4096, 4096], [4094, 4095, 4096, 4097]):
        add("lfact", k[:S] + [4096] * (S - 4))
    for _ in range(36):
        add("lfact", rng.integers(4093, 4100, S))
    # 1e6 .. 2^31 - 1: the overflow branch of the device's gamma rational functions
    for _ in range(60):
        v = np.exp(rng.uniform(np.log(1e6), np.log(2.0e9))) * np.exp(rng.normal(0, 0.2, S))
        add("huge", np.minimum(np.rint(v), 2147483647))
    add("huge", [2147483647] * S)
    add("huge", [2147483647, 2147483646, 2000000000, 2147483647][:S] + [2147483647] * (S - 4))
    # every replicate zero but one; a single count of 1
    for s in range(S):
        for c in (1, 2, 7, 50, 1000):
            k = np.zeros(S, np.int64)
            k[s] = c
            add("one_nonzero", k)
    # the same count in every replicate: the gene-wise dispersion goes to the floor
    for c in (1, 3, 10, 100, 5000, 10 ** 6):
        for _ in range(5):
            add("identical", [c] * S)
    # one replicate 1000 times the others: a Cook's outlier
    for s in range(S):
        for _ in range(8):
            base = rng.integers(5, 60)
            k = rng.integers(base // 2 + 1, base * 2, S)
            k[s] = 1000 * base
            add("outlier", k)
    m = len(cols)
    Kc = np.stack(cols, axis=1)
    src = rng.integers(0, K.shape[1], m)
    FMc = FM[:, src].copy()
    # a zero FullMean in one replicate (its normalisation row is replaced by the size factors)
    for j in range(40):
        k = K[:, src[j]].copy()
        Kc = np.concatenate([Kc, k[:, None]], axis=1)
        f = FM[:, src[j]].copy()
        f[j % S] = 0.0
        FMc = np.concatenate([FMc, f[:, None]], axis=1)
        kinds.setdefault("zero_fullmean", []).append(m + j)
    assert Kc.min() >= 0 and Kc.max() <= 2147483647
    # mixed into the base set at random places
    n0 = K.shape[1]
    Kall = np.concatenate([K, Kc.astype(np.int32)], axis=1)
    FMall = np.concatenate([FM, FMc], axis=1)
    perm = rng.permutation(Kall.shape[1])
    where = np.empty_like(perm)
    where[perm] = np.arange(len(perm))
    kinds = {k: where[n0 + np.asarray(v)] for k, v in kinds.items()}
    return Kall[:, perm], FMall[:, perm], kinds


@pytest.mark.parametrize("base", ["c1", "c3_30k"])
def test_edge_counts_through_set_aggregated(base):
    """c1 (2-vs-2, prior 0.5 as in test_c1_shape_2v2_with_given_prior_variance) or a 30 k-region 3-vs-3 subset of c3,
    plus ~300 crafted regions, handed over with cd_set_aggregated: the trend is still fitted on ordinary data, and every
    crafted region is held to the same per-region gate"""
    d = data("c1") if base == "c1" else data("c3", n_regions=30000)
    prior = 0.5 if base == "c1" else None
    K, FM = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
    Kx, FMx, kinds = crafted_regions(K, FM, np.random.default_rng(11))
    ro = parity.oracle_region_test(Kx, FMx, d.X, prior, theta=0.5)
    # the crafted regions do what they are there for
    assert (ro["dispGeneEst"][kinds["identical"]] < 1e-6).mean() > 0.4
    for k in kinds:
        assert np.isfinite(ro["pvalue"][kinds[k]]).all(), k
    if d.S - d.X.shape[1] > 2:                  # with 2 residual degrees of freedom the cut-off (99) is out of reach
        cutoff = O.lib().orc_qf(0.99, float(d.X.shape[1]), float(d.S - d.X.shape[1]))
        assert (ro["maxCooks"][kinds["outlier"]] > cutoff).sum() >= 5
    t = parity.run_three_aggregated(Kx, FMx, d.X, prior=prior, oracle=ro, theta=0.5)
    assert np.array_equal(t["K"], Kx)
    report = []
    S = parity.compare(t["inputs"], t, report)
    try:
        parity.assert_parity(S, noisy_share=FLAT_PRIOR_NOISY_SHARE)
        # the crafted regions themselves: every column within 1e-6 unless the oracle marks the row rounding-decided
        rs = t["shared"]
        rows = np.concatenate(list(kinds.values()))
        with np.errstate(invalid="ignore"):
            noisy = (ro["geneMargin"] < parity.MARGIN_NOISE) | (ro["mapMargin"] < parity.MARGIN_NOISE)
        for nm, a, b, sc in parity.columns(rs, ro, d.X.shape[1]):
            e = parity.rel(a, b, sc)[rows]
            assert (e[~noisy[rows]] <= parity.TOL).all(), (nm, rows[~noisy[rows] & (e > parity.TOL)][:10])
    except AssertionError:
        print("\n".join(report))
        raise


# ---- NA and negative counts are refused ------------------------------------------------------------------------------

def test_na_and_negative_counts_are_refused():
    """DESeqDataSetFromMatrix (chicdiff.R:1556-1559) stops on NA and negative counts.  An aggregated sum beyond the int32
    range is NA_integer_; it and a negative count handed over with cd_set_aggregated must be refused, and the context
    must take the next, clean matrix as if nothing had happened."""
    X, row_off, N, FMr = parity.aggregate_edge_rows()
    e = engine.Engine(0)
    e.set_design(X)
    e.set_regions(row_off)
    for s in range(4):
        e.set_sample_rows(s, N[s], FMr[s])
    K, FM = e.aggregate()
    assert K[2, 6] == INT32_MIN
    with pytest.raises(engine.ChicdiffError, match="NA or negative"):
        e.region_test()
    with pytest.raises(engine.ChicdiffError, match="NA or negative"):
        e.region_test(theta=0.5, disp_prior_var=0.5)
    e.close()
    d = data("tiny")
    Ko, FMo = O.aggregate(d.row_off, d.N_rows, d.FM_rows)
    e = engine.Engine(0)
    e.set_design(d.X)
    ref = None
    for v in (None, -1, INT32_MIN, None):
        Kb = Ko.copy()
        if v is not None:
            Kb[2, 5] = v
        e.set_aggregated(Kb, FMo)
        if v is None:
            r = e.region_test(theta=0.5)
            if ref is None:
                ref = r
            for k in ("pvalue", "dispersion", "maxCooks"):
                assert np.array_equal(r[k], ref[k], equal_nan=True), k
        else:
            with pytest.raises(engine.ChicdiffError, match="NA or negative"):
                e.region_test(theta=0.5)
    e.close()


def test_na_counts_refused_by_every_shard():
    """cd_multi over 2 GPUs with the overflowing sum in one shard only: both shards must return the error (the clean one
    must not wait for the other in the next collective).  Skipped on a 1-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d = data("tiny")
    N = d.N_rows.copy()
    m = engine.MultiEngine(2)
    m.set_design(d.X)
    m.set_regions(d.row_off, d.region_bait)
    b = m.shards()
    i = int(b[1]) + 3                                     # a region of the second shard
    lo = d.row_off[i]
    N[2, lo] = 2147483647
    N[2, lo + 1] = 5
    for s in range(d.S):
        m.set_sample_rows(s, N[s], d.FM_rows[s])
    K, _ = m.aggregate()
    assert K[2, i] == INT32_MIN and (K[:, :b[1]] >= 0).all()
    with pytest.raises(engine.ChicdiffError, match="NA or negative"):
        m.region_test(theta=0.5)
    # the clean counts run afterwards on the same contexts
    for s in range(d.S):
        m.set_sample_rows(s, d.N_rows[s], d.FM_rows[s])
    m.aggregate()
    assert np.isfinite(m.region_test(theta=0.5)["pvalue"]).any()
    m.close()
