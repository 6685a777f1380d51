"""results_resident() of two builds of the library on the bench workload: padj, filtered p-values, scalars and launch count.

Runs the bench's flagship inputs (synthetic C3, seed 0, 2.14 M regions unless --regions says otherwise) through
aggregate, region_test and results_resident() once per library, each in a child process of its own (the library path
is fixed at import), and compares what results_resident() returned bit for bit.  For a change to the results() code
that must not change its outputs on this workload:

    python scripts/results_resident_check.py --before OLD/libchicdiff_b200.so [--after NEW/libchicdiff_b200.so]

Prints one JSON line; exits 1 when the outputs or the launch count differ.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_one(out_path, regions):
    sys.path.insert(0, ROOT)
    from chicdiff_b200 import engine, synth
    d = synth.generate("c3", n_regions=regions, seed_offset=0)
    e = engine.Engine(0)
    e.set_design(d.X)
    e.set_regions(d.row_off)
    for s in range(d.S):
        e.set_sample_rows(s, d.N_rows[s], d.FM_rows[s])
    e.aggregate()
    e.region_test()
    before = e.launch_count()
    adj = e.results_resident()
    launches = e.launch_count() - before
    np.savez(out_path, pvalue=adj["pvalue"], padj=adj["padj"],
             scalars=np.array([adj["cooksCutoff"], adj["filterThreshold"], adj["filterTheta"], adj["filterIndex"]]),
             launches=np.array([launches]), lib=np.array([engine._LIB_PATH]))
    e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--before", required=True, help="library built from the earlier code")
    ap.add_argument("--after", default=os.path.join(ROOT, "chicdiff_b200", "libchicdiff_b200.so"))
    ap.add_argument("--regions", type=int, default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        run_one(a.child, a.regions)
        return 0
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for tag, lib in (("before", a.before), ("after", a.after)):
            out = os.path.join(tmp, tag + ".npz")
            env = dict(os.environ, CHICDIFF_B200_LIB=os.path.abspath(lib), PYTHONDONTWRITEBYTECODE="1")
            cmd = [sys.executable, os.path.abspath(__file__), "--before", a.before, "--child", out]
            if a.regions:
                cmd += ["--regions", str(a.regions)]
            subprocess.run(cmd, check=True, env=env)
            res[tag] = dict(np.load(out))
    b, f = res["before"], res["after"]
    bits = lambda x: np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    nan_same = lambda x, y: np.array_equal(np.isnan(x), np.isnan(y))
    padj_identical = nan_same(b["padj"], f["padj"]) and np.array_equal(bits(b["padj"])[~np.isnan(b["padj"])],
                                                                     bits(f["padj"])[~np.isnan(f["padj"])])
    pv_identical = nan_same(b["pvalue"], f["pvalue"]) and np.array_equal(bits(b["pvalue"])[~np.isnan(b["pvalue"])],
                                                                       bits(f["pvalue"])[~np.isnan(f["pvalue"])])
    out = dict(regions=int(len(f["padj"])), padj_identical=bool(padj_identical), pvalue_identical=bool(pv_identical),
               scalars_before=b["scalars"].tolist(), scalars_after=f["scalars"].tolist(),
               launches_before=int(b["launches"][0]), launches_after=int(f["launches"][0]),
               padj_non_na=int(np.count_nonzero(~np.isnan(f["padj"]))))
    ok = padj_identical and pv_identical and out["scalars_before"] == out["scalars_after"] and \
        out["launches_before"] == out["launches_after"]
    out["identical"] = bool(ok)
    print(json.dumps(out))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
