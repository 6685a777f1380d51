"""The input codecs beside the device .chinput parser: the .Rds reader (chicdiff_b200/rds.py) and the Arrow cache
(chicdiff_b200/cache.py).  The reader is exercised on chicagoData-like objects built by tests/rds_writer.py."""
import os

import numpy as np
import pytest

import rds_writer
from chicdiff_b200 import cache, rds


def _table(n=5000, seed=0):
    rng = np.random.default_rng(seed)
    labels = ["(0,1]", "(1,2]", "(2,3]", "(3,5]"]
    tlb = [labels[k] for k in rng.integers(0, 4, n)]
    tlb[3] = None
    N = rng.poisson(3, n).astype(np.int32)
    N[7] = rds_writer.NA_INT
    s_i = rng.gamma(2.0, 0.5, n)
    s_i[11] = np.nan
    return [("baitID", "int", rng.integers(1, 900, n).astype(np.int32)),
            ("otherEndID", "int", rng.integers(1, 90000, n).astype(np.int32)),
            ("s_j", "real", rng.gamma(2.0, 0.5, n)),
            ("s_i", "real", s_i),
            ("N", "int", N),
            ("tlb", "str", tlb),
            ("tblb", "factor", (rng.integers(1, 5, n).astype(np.int32), labels)),
            ("Tmean", "real", rng.uniform(0, 1e-3, n)),
            ("isBait2bait", "lgl", rng.integers(0, 2, n).astype(np.int32)),
            ("ids", "deferred", rng.integers(1, 1000, n).astype(np.int32)),
            ("score", "real", rng.uniform(0, 12, n))]


def test_rds_reader_on_a_chicago_object(tmp_path):
    cols = _table()
    path = str(tmp_path / "rep1.Rds")
    rds_writer.chicago_data(path, cols, dict(binsize=20000, maxLBrownEst=1.5e6), dict(rmapfile="x.rmap", removeAdjacent=True))
    t = rds.chicago_table(path)
    assert t["settings"]["rmapfile"] == ["x.rmap"] and t["params"]["binsize"][0] == 20000
    c = t["columns"]
    assert list(c) == [name for name, _, _ in cols]
    by = {name: (kind, v) for name, kind, v in cols}
    for name in ("baitID", "otherEndID", "N", "isBait2bait"):
        assert c[name].dtype == np.int32 and np.array_equal(c[name], by[name][1])
    assert c["N"][7] == rds.NA_INTEGER
    for name in ("s_j", "s_i", "Tmean", "score"):
        assert np.array_equal(c[name], by[name][1], equal_nan=True)         # bit for bit (XDR doubles are IEEE)
    assert list(c["tlb"]) == by["tlb"][1] and c["tlb"][3] is None
    codes, labels = by["tblb"][1]
    assert list(c["tblb"]) == [labels[k - 1] for k in codes]
    assert list(c["ids"]) == [str(int(v)) for v in by["ids"][1]]             # ALTREP deferred string
    obj = rds.read_rds(path)
    assert obj.kind == "S4" and obj.klass() == ["chicagoData"]
    rn = rds.unwrap(obj.attrs["x"].attrs["row.names"])
    assert np.array_equal(rn, np.arange(1, len(c["N"]) + 1))                 # ALTREP compact sequence
    # the bare data.table (what a peak matrix or an exported table is), uncompressed
    w = rds_writer.W()
    rds_writer.data_table(w, cols[:5], altrep_rownames=False)
    p2 = str(tmp_path / "table.Rds")
    open(p2, "wb").write(w.bytes())
    assert list(rds.chicago_table(p2)["columns"]) == ["baitID", "otherEndID", "s_j", "s_i", "N"]
    with pytest.raises(rds.RdsError):
        open(p2, "wb").write(w.bytes()[:-9])
        rds.read_rds(p2)
    with pytest.raises(rds.RdsError):
        open(p2, "wb").write(b"A\n2\n")
        rds.read_rds(p2)


def test_arrow_cache_round_trip_and_invalidation(tmp_path):
    cols = _table(20000, seed=1)
    path = str(tmp_path / "rep2.Rds")
    rds_writer.chicago_data(path, cols, {}, {})
    first = cache.load_or_build(path)
    assert os.path.exists(path + ".arrow")
    assert set(first) == set(cache.CHICAGO_COLUMNS) & {name for name, _, _ in cols}
    direct = rds.chicago_table(path)["columns"]
    calls = []
    second = cache.load_or_build(path, reader=lambda p: calls.append(p) or direct)
    assert calls == []                                                         # served from the cache, source not decoded
    for k, v in first.items():
        if v.dtype == object:
            assert list(v) == list(direct[k]) == list(second[k])
        else:
            assert v.dtype == direct[k].dtype and np.array_equal(v, direct[k], equal_nan=True)
            assert np.array_equal(second[k], v, equal_nan=True)
            assert not second[k].flags.writeable                              # a view of the mapped file, not a copy
    assert first["N"][7] == rds.NA_INTEGER and np.isnan(first["s_i"][11]) and first["tlb"][3] is None
    # a changed source invalidates the cache
    cols2 = _table(1000, seed=2)
    rds_writer.chicago_data(path, cols2, {}, {})
    os.utime(path, ns=(1, 1))
    third = cache.load_or_build(path)
    assert len(third["N"]) == 1000
    # any reader can sit behind the cache (e.g. the device .chinput parser's columns)
    other = str(tmp_path / "counts.chinput")
    open(other, "w").write("x")
    got = cache.load_or_build(other, columns=None, reader=lambda p: dict(baitID=np.arange(5, dtype=np.int32), N=np.ones(5, np.int32)))
    assert np.array_equal(got["baitID"], np.arange(5))


def test_mirror_reads_replicates_through_the_cache(tmp_path):
    """api.read_chicago_tables: the readRDS loop of the reference's front end, {condition: [files]} -> tables"""
    from chicdiff_b200 import api
    files = {}
    for cond, seeds in (("CD4", (3, 4)), ("Mono", (5,))):
        files[cond] = []
        for sd in seeds:
            p = str(tmp_path / ("%s_%d.Rds" % (cond, sd)))
            rds_writer.chicago_data(p, _table(300, seed=sd), {}, {})
            files[cond].append(p)
    a = api.read_chicago_tables(files)
    b = api.read_chicago_tables(files, use_cache=False)
    assert list(a) == ["CD4", "Mono"] and [len(v) for v in a.values()] == [2, 1]
    for cond in a:
        for ta, tb in zip(a[cond], b[cond]):
            assert ta["name"] == tb["name"] and set(ta) == set(tb)
            for k in ta:
                if k == "name":
                    continue
                if ta[k].dtype == object:
                    assert list(ta[k]) == list(tb[k])
                else:
                    assert np.array_equal(ta[k], tb[k], equal_nan=True)
    codes, levels = api.label_codes(a["CD4"][0]["tlb"])
    assert codes[3] == -1 and levels == sorted(levels)

