"""bench.py --dump-outputs: the arrays written for a materialised QuerySpec (host side, no GPU)."""
import numpy as np

import bench
from sybil_b200 import engine as E


class _Hist:
    """The Histogram interface of engine.Hist over fixed values."""

    def __init__(self, n):
        self.n, self.Values = n, np.arange(1002, dtype=np.int64) * n

    def TotalCount(self):
        return self.n

    def Sum(self):
        return self.n * 700

    def Min(self):
        return 30

    def Max(self):
        return 23500

    def Mean(self):
        return 700.0

    def StdDev(self):
        return 1.5

    def GetPercentiles(self):
        return list(range(100))


def _result(key, n, hist=True):
    r = E.Result()
    r.GroupByKey, r.Count, r.Samples = key, n, n
    if hist:
        r.Hists["lat"] = _Hist(n)
    return r


def _query_spec(ngroups, time_buckets=()):
    qs = E.QuerySpec(Aggregations=[E.Aggregation("lat", 0, "hist")])
    qs.Sorted = [_result("g%d\t" % i, ngroups - i, hist=i != 1) for i in range(ngroups)]
    qs.Cumulative = _result("TOTAL\t", sum(r.Count for r in qs.Sorted))
    qs.MatchedCount, qs.NumGroups = qs.Cumulative.Count, ngroups
    qs.TimeResults = {tb: {"b\t": _result("b\t", 2), "a\t": _result("a\t", 1)} for tb in time_buckets}
    return qs


def test_arrays_hold_every_group_field_as_float64():
    a = bench.result_arrays(_query_spec(3, time_buckets=(7200, 3600)))
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["scalars"].tolist() == [6, 3, 0, 0]
    assert a["groups_count"].tolist() == [6, 3, 2, 1]  # Cumulative, then the sorted groups
    assert a["groups_lat_buckets"].shape == (4, 1002) and a["groups_lat_percentiles"].shape == (4, 100)
    assert np.isnan(a["groups_lat_sum"][2]) and np.isnan(a["groups_lat_buckets"][2]).all()  # no histogram
    assert a["groups_lat_sum"][1] == 3 * 700
    assert a["time_bucket"].tolist() == [3600, 3600, 7200, 7200]
    assert a["time_count"].tolist() == [1, 2, 1, 2]  # buckets ascending, groups by key
    assert len(set(a["groups_key_crc32"])) == 4


def test_large_outputs_keep_a_fixed_sample_within_the_limit():
    a = bench.result_arrays(_query_spec(500, time_buckets=(0,)))
    limit = 1 << 20
    assert sum(v.nbytes for v in a.values()) > limit
    s1 = bench.sample_rows(dict(a), limit)
    s2 = bench.sample_rows(dict(bench.result_arrays(_query_spec(500, time_buckets=(0,)))), limit)
    assert sum(v.nbytes for v in s1.values()) <= limit
    assert s1.keys() == s2.keys() and all(np.array_equal(s1[k], s2[k], equal_nan=True) for k in s1)
    rows = s1["groups_rows"].astype(np.int64)
    assert 0 < len(rows) < 501 and np.array_equal(s1["groups_count"], a["groups_count"][rows])
    assert len(s1["time_rows"]) == len(s1["time_count"]) >= 1
