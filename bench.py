#!/usr/bin/env python
"""bench.py -- regions tested per second through the Chicdiff hot path (aggregation + offsets + NB GLM +
dispersion + Wald, with the default norm="combined" theta grid) on synthetic genome-wide 3-vs-3 PCHi-C data
(BASELINE.json configs[2], the configuration the metric's target is quoted on; it fits one GPU).

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
    python bench.py --gpus 1 --steps K --dump-outputs DIR      # ... and the outputs of the last step as DIR/<name>.npy
    python bench.py --impl reference --gpus N --steps K ...    # CPU restatement of the reference (oracle port)
    python bench.py --sweep                                     # region-count sweep (BASELINE.json configs[4])

One step = one pass of DESeq2Wrap's numeric core over one synthetic batch: cd_aggregate + cd_region_test
(size factors, 5 intercept-only theta-grid fits, final dispersion fit, IRLS, Cook's, Wald).
`value` times steps whose inputs are already resident in HBM; `e2e` times the same step through the host-
buffer C-ABI calls, with the pinned-host -> device copy of every input column and the device -> host read of
the output-table columns inside the timed region (the upload of batch k+1 is issued before the region test of
batch k, so it crosses the bus under that test: cd_set_sample_rows is asynchronous on the context's copy stream).
Under torchrun each rank owns a genome-wide set of its own (weak scaling: regions are partitioned by bait, the
global steps exchange sums and counters only); with more than one rank the line also carries a `strong` object:
ONE genome-wide set cut by cd_plan_shards over the ranks, timed the same way and checked against a single-GPU run of
the whole set on rank 0.  Inputs (1.7 GB per rank) are far larger than L2 (126 MB), so no explicit L2 flush is needed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only; the benchmark leaves it as it found it


class stdout_to_stderr:
    """NCCL prints its version banner on stdout when the first communicator comes up; stdout must carry only
    the one JSON line, so file descriptor 1 points at stderr while the communicators are created."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


METRIC = "regions tested/sec (agg+NB GLM+dispersion+Wald)"
UNIT = "regions/s"
WORKLOADS = {"tiny": "synthetic 3-vs-3, one small chromosome (smoke size)",
             "c1": "synthetic chr19-shaped 2-vs-2 PCHi-C (BASELINE configs[0] shape)",
             "c2": "synthetic 2-vs-2 PCHi-C, 1 chromosome (BASELINE configs[1])",
             "c3": "synthetic genome-wide 3-vs-3 PCHi-C (BASELINE configs[2])",
             "c4": "synthetic genome-wide 8-vs-8 PCHi-C with batch covariate, 3-column GLM (BASELINE configs[3])"}


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def read_flop_table():
    """FP64 flop per line-search evaluation by design columns, counted by ncu on this workload
    (scripts/flop_probe.py + scripts/flop_per_eval.py); None when the file is missing."""
    path = os.path.join(ROOT, "profiles", "r02_fit_disp_flop_per_eval.json")
    try:
        with open(path) as fh:
            return json.load(fh), "profiles/r02_fit_disp_flop_per_eval.json"
    except Exception:
        return None, None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_data(workload, n_regions, seed):
    from chicdiff_b200 import synth
    return synth.generate(workload, n_regions=n_regions, seed_offset=1000 * seed)


def cpu_reference_rate(d, sample_regions, threads):
    """Times the oracle port (CPU restatement of the reference) on the first `sample_regions` regions."""
    from oracle import oracle as O
    m = min(sample_regions, d.n)
    r_hi = int(d.row_off[m])
    row_off = d.row_off[: m + 1]
    N = np.ascontiguousarray(d.N_rows[:, :r_hi])
    FMr = np.ascontiguousarray(d.FM_rows[:, :r_hi])
    t0 = time.perf_counter()
    K, FM = O.aggregate(row_off, N, FMr)
    O.region_test(K, FM, d.X, nthreads=threads)
    dt = time.perf_counter() - t0
    return m / dt, dt, m


def workload_label(args, d):
    return "%s: %d regions, %d region rows, %d samples, %d design columns per GPU" % (
        WORKLOADS.get(args.workload, args.workload), d.n, d.R, d.S, int(d.X.shape[1]))


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    threads = os.cpu_count() or 1
    d = make_data(args.workload, args.regions, 0)
    # bounded sample: the whole --steps K run should end within a few minutes whatever K is.  A small probe gives the
    # rate of this box; the per-step sample is what fits ~150 s / K, between 20 000 regions and --cpu-sample
    probe_rate, _, _ = cpu_reference_rate(d, min(args.cpu_sample, 20000), threads)
    sample = int(max(20000, min(args.cpu_sample, probe_rate * 150.0 / max(args.steps, 1))))
    sample = min(sample, d.n)
    times = []
    m = 0
    for _ in range(args.steps):
        rate, dt, m = cpu_reference_rate(d, sample, threads)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = m / (ms * 1e-3)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOADS.get(args.workload, args.workload), "regions_per_step": m,
                       "samples": d.S, "design_columns": int(d.X.shape[1]), "norm": "combined", "theta_grid": 5},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "first %d of %d regions of the same synthetic set, full DESeq2Wrap numerics "
                                       "(aggregation, size factors, 5 theta-grid fits, final fit), OpenMP over regions" % (m, d.n)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(index):
    """Pins this process to the CPU cores next to its GPU (NVML's ideal affinity) before any pinned host buffer is
    allocated, so that the buffers land on that NUMA node and eight ranks' host->device copies do not all cross the
    socket interconnect.  Best effort: returns the number of cores, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


class Runner:
    """one rank's context + the timing helpers"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from chicdiff_b200 import engine
        self.torch, self.dist, self.engine = torch, dist, engine
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; chicdiff_b200 has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.affinity = bind_to_gpu_numa_node(self.local_rank)
        self.e = engine.Engine(self.local_rank)
        if self.world > 1:
            with stdout_to_stderr():
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
                uid = [self.e.comm_unique_id() if self.rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                self.e.comm_init(self.world, self.rank, uid[0])
                dist.barrier()
                torch.cuda.synchronize()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, e=None):
        """K steps bracketed by barrier + synchronize; device time from CUDA events on the context's stream, max over ranks"""
        e = e or self.e
        self.barrier()
        e.timer_start()
        t0 = time.perf_counter()
        tm = np.zeros(8)
        for k in range(steps):
            fn(k, steps)
            tm += e.last_timings()
        dev_ms = e.timer_stop()
        wall_ms = (time.perf_counter() - t0) * 1e3
        self.barrier()
        t = self.torch.tensor([dev_ms, wall_ms], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]) / steps, float(t[1]) / steps, tm / steps

    def total(self, x):
        t = self.torch.tensor([x], dtype=self.torch.int64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t)
        return int(t)


def fp64_roofline(e, d, fit_ms, fp64_peak, flop_tab, flop_src):
    """achieved FP64 rate of the line-search kernels: evaluations counted on the device in this run x flop per
    evaluation (ncu instruction counts of the same kernels, committed) / their CUDA-event time in this run"""
    calls = e.last_search_counts()
    evals = sum(c[0] for c in calls)
    out = {"bound": "fp64", "kernel": "fit_disp_kernel (dispersion line searches: %.0f %% of the step)" % 0.0,
           "unit": "TFLOP/s", "peak": fp64_peak, "peak_source": "DFMA loop timed in this run (cd_measure_fp64_peak); DFMA = 2 flop",
           "evaluations_per_step": int(evals), "replicates": d.S, "kernel_ms_per_step": fit_ms,
           "achieved": None, "frac": None, "traffic": None, "flop_source": flop_src}
    if flop_tab is not None and flop_tab.get("S") == d.S:
        flop = inst = 0.0
        ok = True
        for ev, p, _ in calls:
            ent = flop_tab["per_design_columns"].get(str(p))
            if ent is None:
                ok = False
                break
            flop += ev * ent["flop_per_evaluation"]
            inst += ev * ent.get("fp64_instructions_per_evaluation", float("nan"))
        if ok and fit_ms > 0:
            out["achieved"] = flop / (fit_ms * 1e-3) / 1e12
            out["frac"] = out["achieved"] / fp64_peak if fp64_peak else None
            out["algorithmic_flop_per_step"] = flop
            out["flop_per_evaluation"] = {p: v["flop_per_evaluation"] for p, v in flop_tab["per_design_columns"].items()}
            if fp64_peak and inst == inst:
                # DFMA, DMUL and DADD all take one slot of the FP64 pipe: its utilisation is what bounds the kernel; the
                # flop fraction above counts a DADD or DMUL as half a DFMA
                out["fp64_pipe_frac"] = inst / (fit_ms * 1e-3) / (fp64_peak * 1e12 / 2)
                out["fma_share_of_fp64_instructions"] = (flop - inst) / inst
    return out


def hbm_roofline(d, agg_ms, peaks, peak_src):
    W = d.R / max(d.n, 1)
    agg_bytes = d.n * (W * d.S * 12 + 8 + d.S * 12)          # DESIGN.md: rows read once + CSR offsets + outputs written
    achieved = agg_bytes / (agg_ms * 1e-3) / 1e9 if agg_ms > 0 else None
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_aggregate_traffic.json")) as fh:
            t = json.load(fh)
        if t.get("regions") == d.n and t.get("S") == d.S:
            traffic = t["dram_bytes_per_launch"]
    except Exception:
        pass
    return {"bound": "hbm", "kernel": "aggregate_kernel", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"] if achieved else None, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": agg_bytes, "kernel_ms": agg_ms}


def stage_dict(tm):
    return {"aggregate": tm[0], "region_test": tm[1], "fit_disp_kernels": tm[2], "wald_kernels": tm[3],
            "grid_refits": tm[4], "trend_and_mad": tm[5], "size_factors": tm[6]}


DUMP_BUDGET = 60 * 2 ** 20          # bytes of per-region arrays in one dump (the whole dump stays under 64 MB)


def dump_outputs(path, r, n):
    """Writes what Engine.region_test returned as path/<name>.npy in float64 (integer columns are exact in float64;
    a scalar that is None, such as theta without a grid, becomes NaN).  When the per-region arrays of all n regions
    exceed DUMP_BUDGET, they are cut to the same seeded sample of regions on every run with the same arguments, and
    the sampled region indices go to region_index.npy."""
    per_region = {k: v for k, v in r.items()
                  if isinstance(v, np.ndarray) and v.shape[-1] == n and k not in ("sizeFactors", "deviances")}
    width = sum(v.size // n for v in per_region.values())
    m = min(n, DUMP_BUDGET // (8 * (width + 1)))
    idx = None if m == n else np.sort(np.random.default_rng(20261020).choice(n, m, replace=False))
    os.makedirs(path, exist_ok=True)
    for k, v in r.items():
        if k in per_region:
            v = v if idx is None else v[..., idx]
        elif v is None:
            v = np.nan
        np.save(os.path.join(path, k + ".npy"), np.asarray(v, dtype=np.float64))
    if idx is not None:
        np.save(os.path.join(path, "region_index.npy"), idx.astype(np.float64))


def run_strong(R, args, d_full):
    """ONE genome-wide set partitioned by bait over the ranks (the north-star configuration), timed like the main line and
    checked against a single-GPU run of the whole set on rank 0."""
    from chicdiff_b200 import parallel
    torch, dist, e = R.torch, R.dist, R.e
    d = d_full
    bounds = parallel.shard_slices(d.region_bait, d.row_off, R.world)
    off, (Nl, FMl), (lo, hi) = parallel.take_shard(d.row_off, [d.N_rows, d.FM_rows], bounds, R.rank)
    n_loc, R_loc = hi - lo, int(off[-1])
    e.set_regions(off)
    N_dev = torch.from_numpy(Nl).cuda()
    FM_dev = torch.from_numpy(FMl).cuda()
    e.set_rows_device(R_loc, N_dev.data_ptr(), FM_dev.data_ptr())

    def step(k, steps):
        e.aggregate(fetch=False)
        e.region_test(fetch="none")

    for _ in range(3):
        step(0, 1)
    ms, _, tm = R.timed(step, args.steps)
    e.aggregate(fetch=False)
    r = e.region_test(fetch="table")
    sizes = [int(bounds[k + 1] - bounds[k]) for k in range(R.world)]

    def gather_pvalues(res):
        """p-values of all shards on every rank, in region order (rank order = region order; shards are ragged)"""
        m = max(sizes)
        pad = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
        pad[: sizes[R.rank]] = torch.from_numpy(res["pvalue"]).cuda()
        padded = [torch.empty(m, dtype=torch.float64, device="cuda") for _ in sizes]
        dist.all_gather(padded, pad)
        return torch.cat([q[:k] for q, k in zip(padded, sizes)]).cpu().numpy()

    pv = gather_pvalues(r)
    # the same set on one GPU (rank 0, a context of its own without communicator); its global scalars go to every rank
    box = [None]
    e1 = r1 = None
    one_ms = None
    if R.rank == 0:
        e1 = R.engine.Engine(R.local_rank)
        e1.set_design(d.X); e1.set_regions(d.row_off)
        for s in range(d.S):
            e1.set_sample_rows(s, d.N_rows[s], d.FM_rows[s])
        e1.aggregate(fetch=False)
        for _ in range(2):
            r1 = e1.region_test(fetch="table")
        e1.aggregate(fetch=False)
        r1 = e1.region_test(fetch="table")
        one_ms = e1.last_timings()[0] + e1.last_timings()[1]
        box[0] = (r1["theta"], r1["trend_a0"], r1["trend_a1"], r1["varLogDispEsts"], r1["dispPriorVar"])
    dist.broadcast_object_list(box, src=0)
    th, a0, a1, vld, pvar = box[0]
    # second sharded run with the single-GPU run's global scalars: per-region numbers then depend on the region's data only
    rs = e.region_test(fetch="table", theta_grid=[th], trend=(a0, a1), var_log_disp=vld, disp_prior_var=pvar)
    pv_shared = gather_pvalues(rs)
    out = None
    if R.rank == 0:
        with np.errstate(invalid="ignore", divide="ignore"):
            rel = np.abs(pv - r1["pvalue"]) / np.maximum(np.abs(r1["pvalue"]), 1e-300)
            rel_s = np.abs(pv_shared - r1["pvalue"]) / np.maximum(np.abs(r1["pvalue"]), 1e-300)
        rel[np.isnan(rel)] = 0.0
        rel_s[np.isnan(rel_s)] = 0.0
        adj_s = R.engine.results_adjust(r1["baseMean"], r1["maxCooks"], r1["flags"], pv, d.S, int(d.X.shape[1]))
        adj_1 = R.engine.results_adjust(r1["baseMean"], r1["maxCooks"], r1["flags"], r1["pvalue"], d.S, int(d.X.shape[1]))
        with np.errstate(invalid="ignore"):
            same_calls = bool(np.array_equal(adj_s["padj"] < 0.05, adj_1["padj"] < 0.05))
        out = {"what": "ONE genome-wide set (%d regions) partitioned by bait over %d GPUs (cd_plan_shards), inputs resident" % (d.n, R.world),
               "ms_per_step": ms, "value": d.n / (ms * 1e-3), "unit": UNIT, "regions_per_gpu": sizes,
               "one_gpu_ms_per_step_same_set": one_ms, "speedup_vs_one_gpu": one_ms / ms,
               "stage_ms": stage_dict(tm),
               "check_vs_single_gpu": {"what": "p-values of the sharded run against a single-GPU run of the same set.  free: each run fits its own "
                                               "dispersion trend (the sharded sums add up in another order; one region whose line search takes "
                                               "the other branch of a rounding-level comparison moves the trend by ~1e-6 and with it every far-tail "
                                               "p-value); shared_scalars: the sharded run repeated with the single-GPU run's trend / MAD / prior, "
                                               "which leaves only per-region differences (DESIGN.md section 5)",
                                       "free": {"pvalue_max_rel": float(rel.max()), "regions_beyond_1e-6": int((rel > 1e-6).sum())},
                                       "shared_scalars": {"pvalue_max_rel": float(rel_s.max()), "regions_beyond_1e-6": int((rel_s > 1e-6).sum())},
                                       "pvalue_checksum_sharded": float(np.nansum(pv)), "pvalue_checksum_single": float(np.nansum(r1["pvalue"])),
                                       "theta_equal": bool(r["theta"] == r1["theta"]),
                                       "significant_calls_identical": same_calls}}
        e1.close()
    R.barrier()
    return out


def run_sweep(R, args):
    """region-count sweep (BASELINE.json configs[4]): ms/step, regions/s, stage split and both roofline fractions per size.
    Sizes up to ~2 M regions per GPU are generated directly; larger ones replicate a 2.1 M-region set on the device
    (tiles of the same regions: the trip-count distribution, and with it the timing per region, is that of the base set)."""
    torch, e = R.torch, R.e
    peaks, peak_src = read_peaks()
    flop_tab, flop_src = read_flop_table()
    fp64_peak = e.measure_fp64_peak()
    if args.sweep_sizes:
        totals = [int(float(x)) for x in args.sweep_sizes.split(",")]
    else:
        totals = [100000, 1000000, 10000000] if R.world == 1 else [10000000, 100000000]
    points = []
    for total in totals:
        per_rank = total // R.world
        tiles = 1
        gen = per_rank
        if per_rank > 3000000:
            tiles = max(1, int(round(per_rank / 2135814.0)))
            gen = None                                  # the full c3 set
        d = make_data("c3", gen, R.rank)
        S, n0, R0 = d.S, d.n, d.R
        e.set_design(d.X)
        N_dev = torch.from_numpy(d.N_rows).cuda()
        FM_dev = torch.from_numpy(d.FM_rows).cuda()
        row_off = d.row_off
        if tiles > 1:
            N_dev = N_dev.repeat(1, tiles).contiguous()
            FM_dev = FM_dev.repeat(1, tiles).contiguous()
            row_off = np.concatenate([[0]] + [d.row_off[1:] + k * R0 for k in range(tiles)]).astype(np.int64)
        n, Rr = n0 * tiles, R0 * tiles
        e.set_regions(row_off)
        e.set_rows_device(Rr, N_dev.data_ptr(), FM_dev.data_ptr())

        def step(k, steps):
            e.aggregate(fetch=False)
            e.region_test(fetch="none")

        for _ in range(2):
            step(0, 1)
        l0 = e.launch_count()
        ms, _, tm = R.timed(step, args.steps)
        launches = (e.launch_count() - l0) // args.steps
        n_tot = R.total(n)
        if R.rank == 0:
            class _D:
                pass
            dd = _D(); dd.n, dd.R, dd.S = n, Rr, S
            fr = fp64_roofline(e, d, tm[2], fp64_peak, flop_tab, flop_src)
            hb = hbm_roofline(dd, tm[0], peaks, peak_src)
            points.append({"regions_total": n_tot, "regions_per_gpu": n, "tiles_of_base_set": tiles, "n_gpus": R.world,
                           "ms_per_step": ms, "value": n_tot / (ms * 1e-3), "launches_per_step": int(launches),
                           "stage_ms": stage_dict(tm), "fit_disp_fp64_frac": fr["frac"], "fit_disp_tflops": fr["achieved"],
                           "aggregate_hbm_frac": hb["frac"], "aggregate_gbs": hb["achieved"]})
        del N_dev, FM_dev
        torch.cuda.empty_cache()
    if R.rank == 0:
        print(json.dumps({"metric": METRIC, "unit": UNIT, "sweep": points, "n_gpus": R.world, "steps": args.steps,
                          "scaling": "one set partitioned by bait over the ranks (each rank generates its own partition)",
                          "fp64_peak_tflops_measured": fp64_peak, "hbm_peak_gbs": peaks["hbm_gbs"]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed section")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--regions", type=int, default=None, help="override the number of regions per rank")
    ap.add_argument("--cpu-sample", type=int, default=600000, help="regions in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sub-line of a multi-rank run")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default): every rank owns a genome-wide set of its own; strong: ONE set, regions partitioned by "
                         "bait across the ranks (cd_plan_shards)")
    ap.add_argument("--sweep", action="store_true", help="region-count sweep instead of the bench line")
    ap.add_argument("--sweep-sizes", default=None, help="comma-separated total region counts")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last device-resident step returned (rank 0's regions) as DIR/<name>.npy, float64, "
                         "at most 64 MB: a fixed seeded sample of the regions when all of them would not fit")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sweep or args.impl != "cuda"):
        ap.error("--dump-outputs applies to the bench line of the CUDA path")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    R = Runner(args)
    torch, dist, e, engine = R.torch, R.dist, R.e, R.engine
    if args.sweep:
        run_sweep(R, args)
        e.close()
        if world > 1:
            dist.destroy_process_group()
        return

    d = make_data(args.workload, args.regions, rank if args.scaling == "weak" else 0)
    d_full = d
    if args.scaling == "strong" and world > 1:
        # one genome-wide set, regions partitioned by bait (every rank generates the same set and keeps its shard)
        from chicdiff_b200 import parallel
        import copy
        bounds = parallel.shard_slices(d.region_bait, d.row_off, world)
        off, (Nl, FMl, rb, ro), (lo, hi) = parallel.take_shard(d.row_off, [d.N_rows, d.FM_rows, d.row_bait, d.row_oe], bounds, rank)
        d = copy.copy(d_full)
        d.row_off, d.N_rows, d.FM_rows, d.row_bait, d.row_oe = off, Nl, FMl, rb, ro
        d.region_bait, d.region_seed, d.true_lfc = d.region_bait[lo:hi], d.region_seed[lo:hi], d.true_lfc[lo:hi]
        d.extra = {}
    S, p, n, Rr = d.S, int(d.X.shape[1]), d.n, d.R
    e.set_design(d.X)
    e.set_regions(d.row_off)

    # pinned host copies of the inputs (what the R glue would hand over) and device-resident copies
    N_host = torch.from_numpy(d.N_rows).pin_memory()
    FM_host = torch.from_numpy(d.FM_rows).pin_memory()
    N_dev = N_host.cuda(non_blocking=True)
    FM_dev = FM_host.cuda(non_blocking=True)
    torch.cuda.synchronize()
    fp64_peak = e.measure_fp64_peak()

    def step_resident(k, steps):
        e.aggregate(fetch=False)
        return e.region_test(fetch="none")

    def upload():
        for s in range(S):
            e.set_sample_rows_ptr(s, Rr, N_host[s].data_ptr(), FM_host[s].data_ptr())

    # result columns of a step land in page-locked host memory (allocated once, like the input rows)
    table_out = {k: torch.empty(n, dtype=torch.float64).pin_memory().numpy() for k in
                 ("baseMean", "log2FoldChange", "lfcSE", "stat", "pvalue", "maxCooks")}
    table_out["flags"] = torch.empty(n, dtype=torch.uint8).pin_memory().numpy()

    def step_e2e(k, steps):
        # batch k's rows were uploaded during batch k-1's region test (or just now for the first batch); batch k+1's
        # upload is issued before this batch's region test and crosses the bus under it
        if k == 0:
            upload()
        e.aggregate(fetch=False)
        if k + 1 < steps:
            upload()
        return e.region_test(fetch="table", out=table_out)

    # device-resident steps
    e.set_rows_device(Rr, N_dev.data_ptr(), FM_dev.data_ptr())
    for _ in range(max(args.warmup, 3)):
        step_resident(0, 1)
    launches0 = e.launch_count()
    sampler = ClockSampler(R.local_rank) if rank == 0 else None
    dev_ms, wall_ms, tm = R.timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    launches = (e.launch_count() - launches0) / args.steps
    rendezvous = None
    if world > 1:
        passes, wait_peers, wait_self, wait_first = e.last_rendezvous()
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        launches_trend = 2                      # theta-grid batch + final fit
        rendezvous = {"what": "trend-fit passes of one step: every pass ends with an all-reduce of 8 sums per fit through NVLink peer-memory "
                              "mailboxes inside the kernel; wait = SM cycles CTA 0 of this rank spent polling for a peer's sequence word, "
                              "per pass and peer.  The first pass of a launch absorbs the ranks' different arrival times from their line "
                              "searches (skew); the later passes start together, so their wait is the exchange itself",
                      "trend_passes_per_step": passes, "trend_launches_per_step": launches_trend, "ranks": world,
                      "mean_wait_us_per_pass_and_peer": wait_peers / max(passes * (world - 1), 1) / mhz,
                      "first_pass_wait_us_per_launch_and_peer": wait_first / max(launches_trend * (world - 1), 1) / mhz,
                      "later_pass_wait_us_per_pass_and_peer": (wait_peers - wait_first) / max((passes - launches_trend) * (world - 1), 1) / mhz,
                      "own_slot_us_per_pass": wait_self / max(passes, 1) / mhz,
                      "median_kernel_exchanges_per_step": 8 * 5}
        # how different the ranks are: the line-search time and the DFMA peak of every rank (the step ends with the slowest)
        spread = torch.tensor([tm[2], fp64_peak or 0.0, dev_ms], dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(spread) for _ in range(world)]
        R.dist.all_gather(allr, spread)
        rendezvous["fit_disp_ms_per_rank"] = [round(float(t[0]), 3) for t in allr]
        rendezvous["fp64_peak_tflops_per_rank"] = [round(float(t[1]), 2) for t in allr]
    flop_tab, flop_src = read_flop_table()
    fp64 = fp64_roofline(e, d, tm[2], fp64_peak, flop_tab, flop_src)
    fp64["kernel"] = "fit_disp_kernel (dispersion line searches: %.0f %% of the step)" % (100.0 * tm[2] / dev_ms)

    if args.dump_outputs:
        # the timed step once more on the same resident inputs, its outputs fetched this time.  Its reductions run in a
        # fixed order (no floating-point atomics), so this is what the last timed step computed.  Collective on all ranks.
        e.aggregate(fetch=False)
        r_dump = e.region_test(fetch="all")
        if rank == 0:
            dump_outputs(args.dump_outputs, r_dump, n)

    # end-to-end steps (host buffers in, table columns out)
    e.set_regions(d.row_off)
    step_e2e(0, 1)
    step_e2e(0, 1)
    e2e_dev_ms, e2e_wall_ms, _ = R.timed(step_e2e, args.steps)

    # the upload alone, all ranks at once: what the host side of this box delivers to N GPUs together (the e2e step cannot
    # be shorter than this; at N = 8 it is what bounds it)
    def step_upload(k, steps):
        upload()
        e.aggregate(fetch=False)
    up_ms, _, _ = R.timed(step_upload, args.steps)

    # the same step started one stage earlier: per-replicate CHiCAGO tables -> fused assembly + aggregation
    # (cd_assemble) -> region test.  Reported beside the main line, not instead of it.
    asm = None
    if "tables" in d.extra:
        pin = lambda a: torch.from_numpy(a).pin_memory()
        packed = [engine.Engine.pack_sample_tables(t, pin=pin) for t in d.extra["tables"]]
        asm_h2d = sum(int(k.numel() * k.element_size()) for _, keep in packed for k in keep)
        e.set_rmap(d.frag_chr, d.frag_start, d.frag_end, 1)
        e.set_regions(d.row_off)
        e.set_region_rows(d.row_bait, d.row_oe)
        for si in range(S):
            e.set_sample_tables(si, packed[si])

        def step_asm_resident(k, steps):
            e.assemble(fetch=False)
            return e.region_test(fetch="none")

        def upload_tables():
            for si in range(S):
                e.set_sample_tables(si, packed[si])

        def step_asm_e2e(k, steps):
            # pipelined like the main e2e step: the tables of batch k+1 cross the bus under batch k's region test
            if k == 0:
                upload_tables()
            e.assemble(fetch=False)
            if k + 1 < steps:
                upload_tables()
            return e.region_test(fetch="table", out=table_out)

        for _ in range(2):
            step_asm_resident(0, 1)
        a_dev_ms, _, a_tm = R.timed(step_asm_resident, args.steps)
        for _ in range(2):
            step_asm_e2e(0, 1)
        a_e2e_ms, _, _ = R.timed(step_asm_e2e, args.steps)
        asm = {"what": "per-replicate CHiCAGO tables (s_j, s_i, tblb/tlb, Tmean table, distance function, sparse counts) -> cd_assemble "
                       "(joins + Bmean/Tmean + count merge + region sums in one kernel) -> cd_region_test",
               "ms_per_step": a_dev_ms, "assemble_kernel_ms": a_tm[0], "e2e_ms_per_step": a_e2e_ms, "h2d_bytes_per_step": asm_h2d}

    # the "next" step after the Wald test, outside the metric: results() (Cook's cutoff, independent filtering, BH) on the
    # arrays still in device memory, beside the host routine on the same columns
    res_step = None
    if world == 1:
        r_tab = e.region_test(fetch="table")
        e.results_resident()
        t0 = time.perf_counter()
        for _ in range(3):
            adj_dev = e.results_resident()
        res_dev_ms = (time.perf_counter() - t0) / 3 * 1e3
        t0 = time.perf_counter()
        adj_host = engine.results_adjust(r_tab["baseMean"], r_tab["maxCooks"], r_tab["flags"], r_tab["pvalue"], S, p)
        res_host_ms = (time.perf_counter() - t0) * 1e3
        res_step = {"what": "results(): cd_results_resident (device sorts + prefix counts, padj and filtered p-values copied to the "
                            "host) vs cd_results_adjust (host) on the same columns",
                    "device_wall_ms": res_dev_ms, "host_wall_ms": res_host_ms,
                    "identical": bool(np.array_equal(adj_dev["padj"], adj_host["padj"], equal_nan=True)),
                    "d2h_bytes": int(n * 16)}

    n_tot = R.total(n)

    # north-star configuration: one set over all ranks, with a correctness bit against the single-GPU run
    strong = None
    if world > 1 and args.scaling == "weak" and not args.no_strong:
        d0 = d if rank == 0 else make_data(args.workload, args.regions, 0)      # rank 0's weak set is the seed-0 set
        strong = run_strong(R, args, d0)

    if rank == 0:
        peaks, peak_src = read_peaks()
        value = n_tot / (dev_ms * 1e-3)
        info = e.comm_info()
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": dev_ms, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_label(args, d),
                           "regions_total": n_tot, "design_columns": p, "norm": "combined", "theta_grid": 5,
                           "fits_per_step": 6, "host_cores_bound_to_this_gpu": R.affinity, "l2": "inputs (%.2f GB per GPU) larger than L2; no flush" % ((N_host.numel() * 4 + FM_host.numel() * 8) / 1e9),
                           "parallelism": "regions sharded by bait, %d rank(s); global steps by all-reduce only (trend sums and median "
                                          "histograms: %s; offsets sums, deviances: NCCL); nothing is gathered"
                                          % (world, "inside the kernels over NVLink peer memory" if info["peer_memory_allreduce"] else "single rank")},
                "wall_ms_per_step": wall_ms,
                "stage_ms": stage_dict(tm),
                "roofline": fp64,
                "roofline_hbm": hbm_roofline(d, tm[0], peaks, peak_src),
                "e2e": {"value": n_tot / (e2e_dev_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_dev_ms, "wall_ms_per_step": e2e_wall_ms,
                        "steps": args.steps,
                        "h2d_bytes_per_step": int(N_host.numel() * 4 + FM_host.numel() * 8),
                        "d2h_bytes_per_step": int(n * (6 * 8 + 1)),
                        "upload_alone": {"what": "cd_set_sample_rows of one batch + cd_aggregate and nothing else, all ranks at "
                                                 "the same time (max over ranks): the floor the host-to-device path sets for a step",
                                         "ms": up_ms, "gbs_per_gpu": (N_host.numel() * 4 + FM_host.numel() * 8) / (up_ms * 1e-3) / 1e9,
                                         "gbs_all_gpus": world * (N_host.numel() * 4 + FM_host.numel() * 8) / (up_ms * 1e-3) / 1e9},
                        "pipelined": "the upload of batch k+1 is issued before the region test of batch k (asynchronous "
                                     "cd_set_sample_rows on the context's copy stream, double-buffered rows); every step uploads its "
                                     "own rows inside the timed region"},
                "gpu_launches": int(round(launches * args.steps)), "gpu_launches_per_step": launches, "clocks": clocks}
        if asm is not None:
            asm["value"] = n_tot / (asm["ms_per_step"] * 1e-3)
            asm["e2e_value"] = n_tot / (asm["e2e_ms_per_step"] * 1e-3)
            line["assembly_path"] = asm
        if res_step is not None:
            line["results_step"] = res_step
        if strong is not None:
            line["strong"] = strong
        if rendezvous is not None:
            line["rendezvous"] = rendezvous
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            rate, dt, m = cpu_reference_rate(d, args.cpu_sample, threads)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "first %d of %d regions of the same synthetic set (%.1f s), full DESeq2Wrap numerics, "
                                              "OpenMP over regions on all host cores" % (m, n, dt)}
            # the reference's DESeq2 loops are single-threaded and Chicdiff never enables BiocParallel: one core as well
            rate1, dt1, m1 = cpu_reference_rate(d, max(2000, args.cpu_sample // 16), 1)
            line["cpu_baseline_single_thread"] = {"value": rate1, "unit": UNIT, "cores": 1, "kind": "port",
                                                  "sample": "first %d regions (%.1f s)" % (m1, dt1)}
        print(json.dumps(line), flush=True)
    e.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
