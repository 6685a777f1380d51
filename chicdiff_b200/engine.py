"""ctypes binding of libchicdiff_b200.so (include/chicdiff_b200.h).

This is the Python stand-in for the R ``.Call`` glue (R/r_glue.c): it only marshals NumPy
arrays to the C ABI.  There is no CPU implementation behind it: if the shared library or a
CUDA device is missing every call raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# (CHICDIFF_B200_LIB: development hook to load another build of the same library, e.g. to compare two builds'
# outputs and timings; scripts/results_resident_check.py uses it)
_LIB_PATH = os.environ.get("CHICDIFF_B200_LIB") or os.path.join(_HERE, "libchicdiff_b200.so")
_lib = None

CD_NORM = {"standard": 0, "fullmean": 1, "combined": 2}
FLAG_ALLZERO, FLAG_GENE_GRID, FLAG_MAP_GRID, FLAG_BETA_NOCONV, FLAG_OUTLIER, FLAG_GENE_NOINCREASE, FLAG_COOKS_KEEP = \
    1, 2, 4, 8, 16, 32, 64

EXPORTED = ["cd_version", "cd_create", "cd_destroy", "cd_last_error", "cd_comm_unique_id", "cd_comm_init", "cd_comm_info", "cd_results_resident", "cd_results_device", "cd_ihw_apply",
            "cd_plan_shards", "cd_set_design", "cd_set_regions", "cd_set_sample_rows", "cd_set_rows_device",
            "cd_set_aggregated", "cd_aggregate", "cd_region_test", "cd_results_adjust", "cd_launch_count",
            "cd_device_buffers", "cd_last_timings", "cd_last_search_counts", "cd_get_dims", "cd_last_rendezvous", "cd_ihw_apply_device",
            "cd_prior_var_small_df", "cd_prior_var_hist", "cd_prior_var_from_hist", "cd_prior_var_debug_stream", "cd_prior_var_debug_curve",
            "cd_multi_create", "cd_multi_destroy", "cd_multi_last_error", "cd_multi_gpus", "cd_multi_set_design", "cd_multi_set_regions",
            "cd_multi_get_shards", "cd_multi_set_sample_rows", "cd_multi_aggregate", "cd_multi_region_test", "cd_multi_last_timings", "cd_timer_start", "cd_timer_stop", "cd_measure_fp64_peak",
            "cd_set_rmap", "cd_set_region_rows", "cd_set_sample_tables", "cd_build_sample_tables", "cd_get_sample_tables", "cd_assemble", "cd_get_sample_rows", "cd_get_sample_bmean", "cd_region_universe", "cd_get_region_universe", "cd_countput", "cd_get_countput", "cd_parse_chinput", "cd_get_chinput"]


class ChicdiffError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("chicdiff_b200 error %d: %s" % (code, msg))
        self.code = code


PRIOR_VAR_FN = C.CFUNCTYPE(C.c_double, C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_double))


class CdOptions(C.Structure):
    _fields_ = [("norm", C.c_int), ("theta", C.c_double), ("theta_grid", C.POINTER(C.c_double)),
                ("n_theta_grid", C.c_int), ("disp_prior_var", C.c_double), ("disp_prior_var_grid", C.c_double),
                ("disp_grid_len", C.c_int), ("prior_var_fn", PRIOR_VAR_FN), ("prior_var_user", C.c_void_p),
                ("trend_a0", C.c_double), ("trend_a1", C.c_double), ("var_log_disp", C.c_double)]


class CdSampleTables(C.Structure):
    _fields_ = [("s_j", C.c_void_p), ("tblb", C.c_void_p), ("s_i", C.c_void_p), ("tlb", C.c_void_p),
                ("n_tblb", C.c_int), ("n_tlb", C.c_int), ("tmean", C.c_void_p), ("distfun", C.c_double * 10),
                ("cnt_off", C.c_void_p), ("cnt_oe", C.c_void_p), ("cnt_N", C.c_void_p)]


class CdChicagoTable(C.Structure):
    _fields_ = [("rows", C.c_int64), ("baitID", C.c_void_p), ("otherEndID", C.c_void_p), ("s_j", C.c_void_p), ("s_i", C.c_void_p),
                ("tblb", C.c_void_p), ("tlb", C.c_void_p), ("Tmean", C.c_void_p), ("N", C.c_void_p), ("n_tblb", C.c_int),
                ("n_tlb", C.c_int), ("distfun", C.c_double * 10), ("cnt_rows", C.c_int64), ("cnt_baitID", C.c_void_p),
                ("cnt_otherEndID", C.c_void_p), ("cnt_N", C.c_void_p)]


class CdChicagoRows(C.Structure):
    _fields_ = [("rows", C.c_int64), ("baitID", C.c_void_p), ("otherEndID", C.c_void_p), ("N", C.c_void_p),
                ("Bmean", C.c_void_p), ("score", C.c_void_p)]


_RES_PTRS = ["baseMean", "baseVar", "dispGeneEst", "dispFit", "dispMAP", "dispersion", "log2FoldChange", "lfcSE",
             "beta", "betaSE", "stat", "pvalue", "deviance", "maxCooks", "normFactors", "mu",
             "dispGeneIter", "dispIter", "betaIter", "flags"]


class CdResults(C.Structure):
    _fields_ = ([(k, C.c_void_p) for k in _RES_PTRS] +
                [("sizeFactors", C.c_double * 32), ("theta", C.c_double), ("deviances", C.c_double * 16),
                 ("n_deviances", C.c_int), ("trend_a0", C.c_double), ("trend_a1", C.c_double),
                 ("varLogDispEsts", C.c_double), ("dispPriorVar", C.c_double), ("n_nonzero", C.c_int64),
                 ("n_gene_grid", C.c_int64), ("n_map_grid", C.c_int64), ("n_beta_noconv", C.c_int64)])


def load_library():
    """Loads the in-tree shared library; raises if it was not built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ChicdiffError(-2, "libchicdiff_b200.so is not built (run `python -m chicdiff_b200.build`); "
                                "there is no CPU fallback")
    L = C.CDLL(_LIB_PATH)
    L.cd_version.restype = C.c_char_p
    L.cd_last_error.restype = C.c_char_p
    L.cd_last_error.argtypes = [C.c_void_p]
    L.cd_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.cd_destroy.argtypes = [C.c_void_p]
    L.cd_destroy.restype = None
    L.cd_comm_unique_id.argtypes = [C.c_void_p, C.c_char_p]
    L.cd_comm_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p]
    L.cd_results_resident.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_comm_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.cd_plan_shards.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.cd_set_design.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.cd_set_regions.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.cd_set_sample_rows.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_set_rows_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_set_aggregated.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_aggregate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_region_test.argtypes = [C.c_void_p, C.POINTER(CdOptions), C.POINTER(CdResults)]
    L.cd_results_adjust.argtypes = [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    L.cd_launch_count.argtypes = [C.c_void_p]
    L.cd_launch_count.restype = C.c_int64
    L.cd_device_buffers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    L.cd_last_timings.argtypes = [C.c_void_p, C.c_void_p]
    L.cd_set_rmap.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_set_region_rows.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_set_sample_tables.argtypes = [C.c_void_p, C.c_int, C.POINTER(CdSampleTables)]
    L.cd_build_sample_tables.argtypes = [C.c_void_p, C.c_int, C.POINTER(CdChicagoTable)]
    L.cd_get_sample_tables.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
    L.cd_get_dims.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]
    L.cd_assemble.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_get_sample_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.cd_get_sample_bmean.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.cd_region_universe.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64)]
    L.cd_get_region_universe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_parse_chinput.argtypes = [C.c_void_p, C.c_char_p, C.c_int64, C.POINTER(C.c_int64)]
    L.cd_get_chinput.argtypes = [C.c_void_p] + [C.c_void_p] * 5
    L.cd_countput.argtypes = [C.c_void_p, C.c_int, C.POINTER(CdChicagoRows), C.POINTER(C.c_int64)]
    L.cd_get_countput.argtypes = [C.c_void_p] + [C.c_void_p] * 6
    L.cd_timer_start.argtypes = [C.c_void_p]
    L.cd_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.cd_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.cd_multi_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p]
    L.cd_multi_destroy.argtypes = [C.c_void_p]
    L.cd_multi_destroy.restype = None
    L.cd_multi_last_error.restype = C.c_char_p
    L.cd_multi_last_error.argtypes = [C.c_void_p]
    L.cd_multi_gpus.argtypes = [C.c_void_p]
    L.cd_multi_set_design.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.cd_multi_set_regions.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_multi_get_shards.argtypes = [C.c_void_p, C.c_void_p]
    L.cd_multi_set_sample_rows.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
    L.cd_multi_aggregate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.cd_multi_region_test.argtypes = [C.c_void_p, C.POINTER(CdOptions), C.POINTER(CdResults)]
    L.cd_multi_last_timings.argtypes = [C.c_void_p, C.c_void_p]
    _lib = L
    return L


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def plan_shards(region_bait, row_off, nshards):
    """Contiguous, bait-aligned, row-balanced partition of the regions (cd_plan_shards)."""
    L = load_library()
    region_bait = np.ascontiguousarray(region_bait, dtype=np.int32)
    row_off = np.ascontiguousarray(row_off, dtype=np.int64)
    bounds = np.zeros(nshards + 1, np.int64)
    rc = L.cd_plan_shards(len(region_bait), _ptr(region_bait), _ptr(row_off), nshards, _ptr(bounds))
    if rc != 0:
        raise ChicdiffError(rc, "cd_plan_shards: bad arguments")
    return bounds


def ihw_apply(avDist, pvalue, minLogDist, maxLogDist, avWeights):
    """IHWcorrection()'s "apply to test data" block (cd_ihw_apply, chicdiff.R:2038-2049); rows stay in input order."""
    L = load_library()
    avDist = np.ascontiguousarray(avDist, dtype=np.float64)
    pvalue = np.ascontiguousarray(pvalue, dtype=np.float64)
    lo = np.ascontiguousarray(minLogDist, dtype=np.float64)
    hi = np.ascontiguousarray(maxLogDist, dtype=np.float64)
    w = np.ascontiguousarray(avWeights, dtype=np.float64)
    n = len(avDist)
    group = np.empty(n, np.int32)
    weight, wp, wpadj = np.empty(n), np.empty(n), np.empty(n)
    L.cd_ihw_apply.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]
    rc = L.cd_ihw_apply(n, _ptr(avDist), _ptr(pvalue), len(w), _ptr(lo), _ptr(hi), _ptr(w), _ptr(group), _ptr(weight), _ptr(wp),
                        _ptr(wpadj))
    if rc != 0:
        raise ChicdiffError(rc, "cd_ihw_apply: bad arguments or non-unique breaks")
    return dict(group=group, weight=weight, weighted_pvalue=wp, weighted_padj=wpadj)


def results_adjust(baseMean, maxCooks, flags, pvalue, S, p):
    """DESeq2 results(): Cook's cutoff, independent filtering and BH (cd_results_adjust)."""
    L = load_library()
    baseMean = np.ascontiguousarray(baseMean, dtype=np.float64)
    n = len(baseMean)
    pv = np.array(pvalue, dtype=np.float64, copy=True)
    mc = None if maxCooks is None else np.ascontiguousarray(maxCooks, dtype=np.float64)
    fl = None if flags is None else np.ascontiguousarray(flags, dtype=np.uint8)
    padj = np.empty(n, np.float64)
    sc = np.zeros(4, np.float64)
    rc = L.cd_results_adjust(n, S, p, _ptr(baseMean), _ptr(mc), _ptr(fl), _ptr(pv), _ptr(padj), _ptr(sc))
    if rc != 0:
        raise ChicdiffError(rc, "cd_results_adjust: bad arguments")
    return dict(pvalue=pv, padj=padj, cooksCutoff=sc[0], filterThreshold=sc[1], filterTheta=sc[2], filterIndex=int(sc[3]))


class Engine:
    """One context = one GPU (cd_ctx)."""

    def __init__(self, device=0):
        self._L = load_library()
        h = C.c_void_p()
        rc = self._L.cd_create(C.byref(h), device)
        if rc != 0:
            raise ChicdiffError(rc, self._L.cd_last_error(None).decode())
        self._h = h
        self.S = self.p = None
        self.n = 0
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            self._L.cd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise ChicdiffError(rc, self._L.cd_last_error(self._h).decode())

    # -- multi-GPU -------------------------------------------------------------------------
    def comm_unique_id(self):
        buf = C.create_string_buffer(128)
        self._check(self._L.cd_comm_unique_id(self._h, buf))
        return buf.raw

    def comm_init(self, nranks, rank, uid):
        self._check(self._L.cd_comm_init(self._h, nranks, rank, C.create_string_buffer(uid, 128)))

    def comm_info(self):
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        self._check(self._L.cd_comm_info(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return dict(nranks=a.value, rank=b.value, peer_memory_allreduce=bool(c.value & 1), peer_memory_medians=bool(c.value & 2))

    def results_resident(self):
        """results() (Cook's cutoff, independent filtering, BH) on the arrays of the last region_test, on the device
        (cd_results_resident); same keys as results_adjust()."""
        n = self.n
        pv, padj, sc = np.empty(n), np.empty(n), np.zeros(4)
        self._check(self._L.cd_results_resident(self._h, pv.ctypes.data, padj.ctypes.data, sc.ctypes.data))
        return dict(pvalue=pv, padj=padj, cooksCutoff=sc[0], filterThreshold=sc[1], filterTheta=sc[2], filterIndex=int(sc[3]))

    def results_device(self, baseMean, maxCooks, flags, pvalue, S, p):
        """results() on the given columns with the device routine of results_resident() (cd_results_device); arguments
        and keys as results_adjust().  The columns are copied to this context's GPU; pvalue is not modified."""
        baseMean = np.ascontiguousarray(baseMean, dtype=np.float64)
        n = len(baseMean)
        pvalue = np.ascontiguousarray(pvalue, dtype=np.float64)
        mc = None if maxCooks is None else np.ascontiguousarray(maxCooks, dtype=np.float64)
        fl = None if flags is None else np.ascontiguousarray(flags, dtype=np.uint8)
        if len(pvalue) != n or (mc is not None and len(mc) != n) or (fl is not None and len(fl) != n):
            raise ValueError("results_device: columns of different lengths")
        pv, padj, sc = np.empty(n), np.empty(n), np.zeros(4)
        self._L.cd_results_device.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int] + [C.c_void_p] * 7
        self._check(self._L.cd_results_device(self._h, n, S, p, _ptr(baseMean), _ptr(mc), _ptr(fl), _ptr(pvalue), _ptr(pv),
                                               _ptr(padj), _ptr(sc)))
        return dict(pvalue=pv, padj=padj, cooksCutoff=sc[0], filterThreshold=sc[1], filterTheta=sc[2], filterIndex=int(sc[3]))

    # -- setup ------------------------------------------------------------------------------
    def set_design(self, X):
        X = np.ascontiguousarray(X, dtype=np.float64)
        self.S, self.p = X.shape
        self._check(self._L.cd_set_design(self._h, self.S, self.p, _ptr(X)))

    def set_regions(self, row_off):
        row_off = np.ascontiguousarray(row_off, dtype=np.int64)
        self.n = len(row_off) - 1
        self._check(self._L.cd_set_regions(self._h, self.n, _ptr(row_off)))

    def set_sample_rows(self, s, N, fullmean):
        N = np.ascontiguousarray(N, dtype=np.int32)
        fullmean = np.ascontiguousarray(fullmean, dtype=np.float64)
        self._keep = [N, fullmean]        # the copy is asynchronous on the context's stream
        self._check(self._L.cd_set_sample_rows(self._h, s, len(N), _ptr(N), _ptr(fullmean)))

    def set_sample_rows_ptr(self, s, R, N_ptr, fm_ptr):
        self._check(self._L.cd_set_sample_rows(self._h, s, R, C.c_void_p(N_ptr), C.c_void_p(fm_ptr)))

    def set_rows_device(self, R, N_dev_ptr, fm_dev_ptr):
        self._check(self._L.cd_set_rows_device(self._h, R, C.c_void_p(N_dev_ptr), C.c_void_p(fm_dev_ptr)))

    def set_aggregated(self, K, fullmean):
        K = np.ascontiguousarray(K, dtype=np.int32)
        fullmean = np.ascontiguousarray(fullmean, dtype=np.float64)
        self.n = K.shape[1]
        self._check(self._L.cd_set_aggregated(self._h, self.n, _ptr(K), _ptr(fullmean)))

    # -- per-replicate assembly fused with stage 1 ------------------------------------------------
    def set_rmap(self, chr_codes, start, end, frag_id0=1):
        a = [np.ascontiguousarray(x, dtype=np.int32) for x in (chr_codes, start, end)]
        self._F = len(a[0])
        self._check(self._L.cd_set_rmap(self._h, len(a[0]), frag_id0, _ptr(a[0]), _ptr(a[1]), _ptr(a[2])))

    def region_universe(self, peak_bait, peak_oe, ru_expand=5, fetch=True):
        """getRegionUniverse on the device; returns (row_off, row_bait, row_oe) when fetch."""
        pb = np.ascontiguousarray(peak_bait, dtype=np.int32)
        po = np.ascontiguousarray(peak_oe, dtype=np.int32)
        R = C.c_int64()
        self._check(self._L.cd_region_universe(self._h, len(pb), _ptr(pb), _ptr(po), int(ru_expand), C.byref(R)))
        self.n = len(pb)
        if not fetch:
            return R.value
        off = np.empty(self.n + 1, np.int64)
        rb = np.empty(R.value, np.int32)
        ro = np.empty(R.value, np.int32)
        self._check(self._L.cd_get_region_universe(self._h, _ptr(off), _ptr(rb), _ptr(ro)))
        return off, rb, ro

    def parse_chinput(self, data):
        """bytes of a .chinput file -> dict(baitID, otherEndID, N, otherEndLen, distSign) (cd_parse_chinput)."""
        m = C.c_int64()
        self._check(self._L.cd_parse_chinput(self._h, data, len(data), C.byref(m)))
        g = m.value
        out = dict(baitID=np.empty(g, np.int32), otherEndID=np.empty(g, np.int32), N=np.empty(g, np.int32),
                   otherEndLen=np.empty(g, np.int32), distSign=np.empty(g, np.float64))
        self._check(self._L.cd_get_chinput(self._h, *[_ptr(out[k]) for k in ("baitID", "otherEndID", "N", "otherEndLen", "distSign")]))
        return out

    def countput(self, reps):
        """reps: list of dicts (baitID, otherEndID, N, Bmean, score) of ONE condition's replicates ->
        dict(baitID, otherEndID, Nav, Bav, score, oeID_mid) in first-appearance order (cd_countput)."""
        arr = (CdChicagoRows * len(reps))()
        keep = []
        for k, r in enumerate(reps):
            cols = [np.ascontiguousarray(r["baitID"], dtype=np.int32), np.ascontiguousarray(r["otherEndID"], dtype=np.int32),
                    np.ascontiguousarray(r["N"], dtype=np.int32), np.ascontiguousarray(r["Bmean"], dtype=np.float64),
                    np.ascontiguousarray(r["score"], dtype=np.float64)]
            keep.append(cols)
            arr[k].rows = len(cols[0])
            arr[k].baitID, arr[k].otherEndID, arr[k].N, arr[k].Bmean, arr[k].score = [c.ctypes.data for c in cols]
        G = C.c_int64()
        self._check(self._L.cd_countput(self._h, len(reps), arr, C.byref(G)))
        g = G.value
        out = dict(baitID=np.empty(g, np.int32), otherEndID=np.empty(g, np.int32), Nav=np.empty(g), Bav=np.empty(g),
                   score=np.empty(g), oeID_mid=np.empty(g))
        self._check(self._L.cd_get_countput(self._h, *[_ptr(out[k]) for k in ("baitID", "otherEndID", "Nav", "Bav", "score", "oeID_mid")]))
        return out

    def set_region_rows(self, row_bait, row_oe):
        rb = np.ascontiguousarray(row_bait, dtype=np.int32)
        ro = np.ascontiguousarray(row_oe, dtype=np.int32)
        self._keep_rows = [rb, ro]
        self._check(self._L.cd_set_region_rows(self._h, len(rb), _ptr(rb), _ptr(ro)))

    @staticmethod
    def pack_sample_tables(tab, pin=None):
        """dict (s_j, tblb, s_i, tlb, tmean, distfun, cnt_off, cnt_oe, cnt_N) -> (CdSampleTables, keep-alive list)."""
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        keep = [f64(tab["s_j"]), i32(tab["tblb"]), f64(tab["s_i"]), i32(tab["tlb"]), f64(tab["tmean"]),
                np.ascontiguousarray(tab["cnt_off"], dtype=np.int64), i32(tab["cnt_oe"]), i32(tab["cnt_N"])]
        if pin is not None:
            keep = [pin(k) for k in keep]
        t = CdSampleTables()
        ptr = (lambda a: a.data_ptr()) if pin is not None else (lambda a: a.ctypes.data)
        t.s_j, t.tblb, t.s_i, t.tlb, t.tmean, t.cnt_off, t.cnt_oe, t.cnt_N = [ptr(k) for k in keep]
        t.n_tblb, t.n_tlb = np.asarray(tab["tmean"]).shape
        for k, v in enumerate(np.asarray(tab["distfun"], dtype=np.float64)):
            t.distfun[k] = float(v)
        return t, keep

    def set_sample_tables(self, s, tab):
        t, keep = tab if isinstance(tab, tuple) else self.pack_sample_tables(tab)
        self._keep_tabs = getattr(self, "_keep_tabs", {})
        self._keep_tabs[s] = keep
        self._check(self._L.cd_set_sample_tables(self._h, s, C.byref(t)))

    def build_sample_tables(self, s, t):
        """One replicate's raw CHiCAGO columns (api.chicago_columns) -> the per-fragment tables, built on the device
        (cd_build_sample_tables): first (s_j, tblb) per bait, first (s_i, tlb) per other end, first Tmean per bin pair, counts."""
        c = CdChicagoTable()
        keep = {k: np.ascontiguousarray(t[k], dtype=dt) for k, dt in (("baitID", np.int32), ("otherEndID", np.int32), ("s_j", np.float64),
                ("s_i", np.float64), ("tblb", np.int32), ("tlb", np.int32), ("Tmean", np.float64))}
        c.rows = len(keep["baitID"])
        for k, v in keep.items():
            setattr(c, k, v.ctypes.data)
        if t.get("N") is not None:
            keep["N"] = np.ascontiguousarray(t["N"], dtype=np.int32)
            c.N = keep["N"].ctypes.data
        c.n_tblb, c.n_tlb = int(t["n_tblb"]), int(t["n_tlb"])
        for k, v in enumerate(np.asarray(t["distfun"], dtype=np.float64)):
            c.distfun[k] = float(v)
        if t.get("cnt_baitID") is not None:
            for k in ("cnt_baitID", "cnt_otherEndID", "cnt_N"):
                keep[k] = np.ascontiguousarray(t[k], dtype=np.int32)
                setattr(c, k, keep[k].ctypes.data)
            c.cnt_rows = len(keep["cnt_baitID"])
        self._check(self._L.cd_build_sample_tables(self._h, s, C.byref(c)))
        self._table_shapes = getattr(self, "_table_shapes", {})
        self._table_shapes[s] = (c.n_tblb, c.n_tlb)

    def get_sample_tables(self, s, F=None):
        """the tables of replicate s as they stand on the device (cd_get_sample_tables)"""
        if F is None:
            F = self._F
        nt = self._table_shapes[s]
        out = dict(s_j=np.empty(F), tblb=np.empty(F, np.int32), s_i=np.empty(F), tlb=np.empty(F, np.int32),
                   tmean=np.empty(nt), cnt_off=np.empty(F + 1, np.int64))
        self._check(self._L.cd_get_sample_tables(self._h, s, _ptr(out["s_j"]), _ptr(out["tblb"]), _ptr(out["s_i"]), _ptr(out["tlb"]),
                                                 _ptr(out["tmean"]), _ptr(out["cnt_off"]), None, None))
        m = int(out["cnt_off"][-1])
        out["cnt_oe"], out["cnt_N"] = np.empty(m, np.int32), np.empty(m, np.int32)
        self._check(self._L.cd_get_sample_tables(self._h, s, None, None, None, None, None, None, _ptr(out["cnt_oe"]), _ptr(out["cnt_N"])))
        return out

    def assemble(self, keep_rows=False, fetch=True):
        if fetch:
            K = np.empty((self.S, self.n), np.int32)
            FM = np.empty((self.S, self.n), np.float64)
            av = np.empty(self.n, np.float64)
            self._check(self._L.cd_assemble(self._h, int(keep_rows), _ptr(K), _ptr(FM), _ptr(av)))
            return K, FM, av
        self._check(self._L.cd_assemble(self._h, int(keep_rows), None, None, None))
        return None

    def get_sample_rows(self, s, R):
        N = np.empty(R, np.int32)
        FM = np.empty(R, np.float64)
        self._check(self._L.cd_get_sample_rows(self._h, s, _ptr(N), _ptr(FM)))
        return N, FM

    def get_sample_bmean(self, s, R):
        B = np.empty(R, np.float64)
        self._check(self._L.cd_get_sample_bmean(self._h, s, _ptr(B)))
        return B

    # -- stages -----------------------------------------------------------------------------
    def aggregate(self, fetch=True):
        if fetch:
            K = np.empty((self.S, self.n), np.int32)
            FM = np.empty((self.S, self.n), np.float64)
            self._check(self._L.cd_aggregate(self._h, _ptr(K), _ptr(FM)))
            return K, FM
        self._check(self._L.cd_aggregate(self._h, None, None))
        return None

    def region_test(self, norm="combined", theta=None, theta_grid=None, disp_prior_var=None,
                    disp_prior_var_grid=None, disp_grid_len=20, fetch="all", prior_var_fn=None, trend=None,
                    var_log_disp=None, out=None):
        """cd_region_test.  fetch: "all" | "table" (columns of the output table only) | "none".
        out: optional dict of preallocated result arrays by column name (page-locked ones make the device-to-host copies
        plain DMA transfers; pageable NumPy arrays are staged by the driver at a fraction of the bus rate).
        prior_var_fn(df, residuals) -> dispPriorVar is asked once per dispersion fit whose design has S - p <= 3 and no
        disp_prior_var* given (the place where an R front end evaluates DESeq2's Monte-Carlo rule)."""
        n, S, p = self.n, self.S, self.p
        opt = CdOptions()
        opt.norm = CD_NORM[norm]
        opt.theta = float("nan") if theta is None else float(theta)
        grid = None
        if theta_grid is not None:
            grid = np.ascontiguousarray(theta_grid, dtype=np.float64)
            opt.theta_grid = grid.ctypes.data_as(C.POINTER(C.c_double))
            opt.n_theta_grid = len(grid)
        opt.disp_prior_var = float("nan") if disp_prior_var is None else float(disp_prior_var)
        opt.disp_prior_var_grid = float("nan") if disp_prior_var_grid is None else float(disp_prior_var_grid)
        opt.disp_grid_len = disp_grid_len
        nan = float("nan")
        opt.trend_a0, opt.trend_a1 = (nan, nan) if trend is None else (float(trend[0]), float(trend[1]))
        opt.var_log_disp = nan if var_log_disp is None else float(var_log_disp)
        cb_error = []
        if prior_var_fn is not None:
            def _cb(_user, df, m, ptr):
                try:
                    return float(prior_var_fn(int(df), np.ctypeslib.as_array(ptr, shape=(int(m),)).copy()))
                except Exception as ex:              # never unwind through the C frames
                    cb_error.append(ex)
                    return float("nan")
            cb = PRIOR_VAR_FN(_cb)                   # kept alive by this frame for the duration of the call
            opt.prior_var_fn = cb
        res = CdResults()
        arrays = {}
        shapes = dict(beta=(p, n), betaSE=(p, n), normFactors=(S, n), mu=(S, n))
        dtypes = dict(dispGeneIter=np.int32, dispIter=np.int32, betaIter=np.int32, flags=np.uint8)
        if fetch == "all":
            want = _RES_PTRS
        elif fetch == "table":
            want = ["baseMean", "log2FoldChange", "lfcSE", "stat", "pvalue", "maxCooks", "flags"]
        else:
            want = []
        for k in want:
            shape, dtype = shapes.get(k, (n,)), dtypes.get(k, np.float64)
            if out is not None and k in out:
                a = out[k]                           # the caller's buffer (e.g. page-locked memory: the copy is a plain DMA then)
                if a.shape != shape or a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
                    raise ValueError("out[%r]: expected a C-contiguous %s array of shape %s" % (k, np.dtype(dtype).name, shape))
                arrays[k] = a
            else:
                arrays[k] = np.empty(shape, dtype)
            setattr(res, k, arrays[k].ctypes.data)
        rc = self._region_test_entry()(self._h, C.byref(opt), C.byref(res))
        if cb_error:
            raise cb_error[0]
        self._check(rc)
        out = dict(arrays)
        out["sizeFactors"] = np.array(res.sizeFactors[:S])
        out["theta"] = None if res.theta != res.theta else res.theta
        out["deviances"] = np.array(res.deviances[:res.n_deviances]) if res.n_deviances else None
        for k in ("trend_a0", "trend_a1", "varLogDispEsts", "dispPriorVar", "n_nonzero", "n_gene_grid", "n_map_grid",
                  "n_beta_noconv"):
            out[k] = getattr(res, k)
        return out

    def _region_test_entry(self):
        return self._L.cd_region_test

    # -- introspection ------------------------------------------------------------------------
    def launch_count(self):
        return int(self._L.cd_launch_count(self._h))

    def timer_start(self):
        self._check(self._L.cd_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_double()
        self._check(self._L.cd_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def measure_fp64_peak(self):
        t = C.c_double()
        self._check(self._L.cd_measure_fp64_peak(self._h, C.byref(t)))
        return t.value

    def last_search_counts(self):
        """[(evaluations, design columns, regions searched)] of the dispersion line-search launches of the last region_test"""
        k = C.c_int()
        ev, pc, rg = (C.c_int64 * 16)(), (C.c_int * 16)(), (C.c_int64 * 16)()
        self._L.cd_last_search_counts.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_void_p]
        self._check(self._L.cd_last_search_counts(self._h, C.byref(k), ev, pc, rg))
        return [(int(ev[i]), int(pc[i]), int(rg[i])) for i in range(k.value)]

    def last_timings(self):
        t = np.zeros(8, np.float64)
        self._L.cd_last_timings(self._h, _ptr(t))
        return t

    def ihw_apply_device(self, pvalue, minLogDist, maxLogDist, avWeights, avDist=None):
        """cd_ihw_apply_device: IHWcorrection()'s "apply to test data" block on this context's GPU.  avDist=None uses the
        avDist column cd_assemble left on the device."""
        pvalue = np.ascontiguousarray(pvalue, dtype=np.float64)
        n = len(pvalue)
        av = None if avDist is None else np.ascontiguousarray(avDist, dtype=np.float64)
        lo = np.ascontiguousarray(minLogDist, dtype=np.float64)
        hi = np.ascontiguousarray(maxLogDist, dtype=np.float64)
        w = np.ascontiguousarray(avWeights, dtype=np.float64)
        group = np.empty(n, np.int32)
        weight, wp, wpadj = np.empty(n), np.empty(n), np.empty(n)
        self._L.cd_ihw_apply_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 7
        self._check(self._L.cd_ihw_apply_device(self._h, n, _ptr(av), _ptr(pvalue), len(w), _ptr(lo), _ptr(hi), _ptr(w),
                                                _ptr(group), _ptr(weight), _ptr(wp), _ptr(wpadj)))
        return dict(group=group, weight=weight, weighted_pvalue=wp, weighted_padj=wpadj)

    def last_rendezvous(self):
        """(trend passes, SM cycles waited for peers, SM cycles waited for the own slot, the first-pass part of the peers'
        figure) of the last region_test"""
        a, b, c, d = C.c_double(), C.c_double(), C.c_double(), C.c_double()
        self._L.cd_last_rendezvous.argtypes = [C.c_void_p] + [C.POINTER(C.c_double)] * 4
        self._check(self._L.cd_last_rendezvous(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value


class MultiEngine(Engine):
    """Several GPUs from this one process (cd_multi_*): same calls as Engine on the whole problem; the library cuts the
    regions into bait-aligned shards, one per device, and runs one host thread per device inside every call."""

    def __init__(self, n_gpus, device_ids=None):
        self._L = load_library()
        h = C.c_void_p()
        ids = None if device_ids is None else np.ascontiguousarray(device_ids, dtype=np.int32)
        rc = self._L.cd_multi_create(C.byref(h), int(n_gpus), _ptr(ids))
        if rc != 0:
            raise ChicdiffError(rc, self._L.cd_multi_last_error(None).decode())
        self._h = h
        self.S = self.p = None
        self.n = 0
        self.n_gpus = int(n_gpus)
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            self._L.cd_multi_destroy(self._h)
            self._h = None

    def _check(self, rc):
        if rc != 0:
            raise ChicdiffError(rc, self._L.cd_multi_last_error(self._h).decode())

    def set_design(self, X):
        X = np.ascontiguousarray(X, dtype=np.float64)
        self.S, self.p = X.shape
        self._check(self._L.cd_multi_set_design(self._h, self.S, self.p, _ptr(X)))

    def set_regions(self, row_off, region_bait):
        row_off = np.ascontiguousarray(row_off, dtype=np.int64)
        region_bait = np.ascontiguousarray(region_bait, dtype=np.int32)
        self.n = len(row_off) - 1
        self._check(self._L.cd_multi_set_regions(self._h, self.n, _ptr(row_off), _ptr(region_bait)))

    def shards(self):
        b = np.zeros(self.n_gpus + 1, np.int64)
        self._check(self._L.cd_multi_get_shards(self._h, _ptr(b)))
        return b

    def set_sample_rows(self, s, N, fullmean):
        N = np.ascontiguousarray(N, dtype=np.int32)
        fullmean = np.ascontiguousarray(fullmean, dtype=np.float64)
        self._keep.append((N, fullmean))            # uploads are asynchronous until the next aggregate
        self._check(self._L.cd_multi_set_sample_rows(self._h, s, len(N), _ptr(N), _ptr(fullmean)))

    def aggregate(self, fetch=True):
        K = np.empty((self.S, self.n), np.int32) if fetch else None
        FM = np.empty((self.S, self.n), np.float64) if fetch else None
        self._check(self._L.cd_multi_aggregate(self._h, _ptr(K), _ptr(FM)))
        self._keep = []
        return (K, FM) if fetch else None

    def _region_test_entry(self):
        return self._L.cd_multi_region_test

    def last_timings(self):
        t = np.zeros(8, np.float64)
        self._L.cd_multi_last_timings(self._h, _ptr(t))
        return t
