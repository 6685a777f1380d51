"""Search for inputs on which the 0-based and the 1-based index of quantile(type = 7) give different filter cut-offs.

results() takes its 50 filter cut-offs from quantile(baseMean, theta), which R (quantile.default, type 7 branch)
computes as
    index <- 1 + (n - 1) * probs;  lo <- floor(index);  hi <- ceiling(index)
    qs <- x[lo];  i <- which(index > lo & x[hi] != qs);  h <- (index - lo)[i];  qs[i] <- (1 - h) * qs[i] + h * x[hi[i]]
A 0-based restatement index0 = (n - 1) * probs, h0 = index0 - floor(index0) differs from it only through the rounding
of 1 + (n - 1) * probs, which drops the last bit of (n - 1) * probs when that lies in [2^j - 1, 2^j).  Such a
difference in h moves the interpolated cut by an ulp or so.  It changes the rows kept (baseMean >= cut) only when the
cut lands on a data value: sorted values q = x[lo] and qh = x[hi] are neighbours, so the only values that can switch
sides are q (cut == q in one version, q + ulp in the other) and qh.

For every (n, number of zero baseMeans, theta) visited this finds the h of both versions and, where they differ, tries
q = 1 and qh = 1 + d * 2^-52 for the d around 1 / (2 h) where the rounding of the interpolation changes.  A hit is a
dataset (n, nzero, k, q, qh) on which the two versions keep a different set of rows at cut-off k.

    python scripts/quantile_index_search.py [--nmax 10000000] [--pairs 20000000] [--seed 1]
prints the hits found (or the closest candidates) as JSON lines.
"""
import argparse
import json

import numpy as np

NT = 50


def r_lower(nzero, n):
    """mean(filter == 0): R sums the logical in long double and divides by n in long double, then rounds to double."""
    return (np.asarray(nzero, dtype=np.longdouble) / np.asarray(n, dtype=np.longdouble)).astype(np.float64)


def r_theta(lower):
    """seq(lower, upper, length.out = 50): c(from, from + (1:48) * ((to - from) / 49), to)."""
    lower = np.asarray(lower, dtype=np.float64)
    upper = np.where(lower < .95, .95, 1.0)
    k = np.arange(NT, dtype=np.float64)
    th = lower[..., None] + k * ((upper - lower) / (NT - 1))[..., None]
    th[..., -1] = upper
    th[..., 0] = lower
    return th


def interp(h, q, qh):
    return (1.0 - h) * q + h * qh


def crossing(h1, h0):
    """For pairs (h1, h0) with h1 != h0, a qh = 1 + d * 2^-52 (q = 1) on which the two cuts keep different rows, or 0."""
    q = 1.0
    out = np.zeros(len(h1))
    for hh in (h1, h0):
        with np.errstate(divide="ignore"):
            d0 = np.floor(0.5 / np.where(hh > 0, hh, np.inf))
        for dd in range(-3, 4):
            d = d0 + dd
            ok = (d >= 1) & (d < 2.0 ** 52) & (out == 0)
            qh = q + d * 2.0 ** -52
            c1 = np.where(h1 > 0, interp(h1, q, qh), q)
            c0 = np.where(h0 > 0, interp(h0, q, qh), q)
            diff = ((c1 <= q) != (c0 <= q)) | ((c1 <= qh) != (c0 <= qh))
            out = np.where(ok & diff, qh, out)
    return out


def scan(n, nzero):
    """n, nzero: 1-d arrays of equal length.  Returns (n, nzero, k, h1, h0, qh) of the hits, and the candidates with
    h1 != h0 sorted by h (smallest first) for the record."""
    n = np.asarray(n, dtype=np.int64)
    nzero = np.asarray(nzero, dtype=np.int64)
    th = r_theta(r_lower(nzero, n))                                      # (m, 50)
    x = (n - 1).astype(np.float64)[:, None] * th
    i1 = 1.0 + x
    lo1 = np.floor(i1)
    h1 = i1 - lo1
    lo0 = np.floor(x)
    h0 = x - lo0
    # the 1-based version reads x[lo1] (1-based) = sorted position lo1 - 1; when the positions differ h1 is 0 and
    # the two cuts are the same value x[lo0 + 1] or an interpolation towards it that cannot pass it
    same_pos = (lo1 - 1) == lo0
    diff = same_pos & (h1 != h0)
    r, k = np.nonzero(diff)
    if len(r) == 0:
        return [], []
    qh = crossing(h1[r, k], h0[r, k])
    hit = qh > 0
    hits = [dict(n=int(n[a]), nzero=int(nzero[a]), k=int(b), h_r=float(c), h_0based=float(d), q=1.0, qh=float(e))
            for a, b, c, d, e in zip(r[hit], k[hit], h1[r[hit], k[hit]], h0[r[hit], k[hit]], qh[hit])]
    o = np.argsort(np.minimum(h1[r, k], h0[r, k]))[:5]
    near = [dict(n=int(n[r[i]]), nzero=int(nzero[r[i]]), k=int(k[i]), h_r=float(h1[r[i], k[i]]), h_0based=float(h0[r[i], k[i]]))
            for i in o]
    return hits, near


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmin", type=int, default=2)
    ap.add_argument("--nmax", type=int, default=10_000_000)
    ap.add_argument("--pairs", type=int, default=20_000_000, help="random (n, nzero) pairs with nzero > 0")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--max-hits", type=int, default=20)
    a = ap.parse_args()
    hits, near = [], []
    step = 200_000
    for s in range(a.nmin, a.nmax + 1, step):                            # no zero baseMean: lower = 0
        n = np.arange(s, min(s + step, a.nmax + 1))
        h, nr = scan(n, np.zeros_like(n))
        hits += h
        near += nr
        if len(hits) >= a.max_hits:
            break
    rng = np.random.default_rng(a.seed)
    done = 0
    while done < a.pairs and len(hits) < a.max_hits:                     # some zero baseMeans: lower = nzero / n
        m = min(step, a.pairs - done)
        n = rng.integers(a.nmin, a.nmax + 1, m)
        nzero = (rng.random(m) * 0.95 * n).astype(np.int64)
        h, nr = scan(n, nzero)
        hits += h
        near += nr
        done += m
    for h in hits[:a.max_hits]:
        print(json.dumps(dict(hit=True, **h)))
    if not hits:
        near.sort(key=lambda d: min(d["h_r"], d["h_0based"]))
        for d in near[:5]:
            print(json.dumps(dict(hit=False, **d)))


if __name__ == "__main__":
    main()
