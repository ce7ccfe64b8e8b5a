"""Cold spells without a GPU: the cold accounting of k_intensity (hdp_b200/csrc/intensity.h: intensity_e with the deficit) replayed
on the CPU by tests/cold_host.cpp against the heatwave oracle on negated inputs - cold(x, thr) must equal warm(-x, -thr) bit for
bit - plus the HDP_B200_COLD flag of the C ABI (its value, the unchanged ABI version, how the entry points decode it) and the
Python layer around it (season swap, variable names and attributes).  The kernels themselves are checked by
tests/test_gpu_cold.py on the GPU."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import intensity_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def replay(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("cold") / "libcold_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-shared", "-fPIC", "-I",
                    os.path.join(ROOT, "hdp_b200", "csrc"), os.path.join(ROOT, "tests", "cold_host.cpp"), "-o", so], check=True)
    L = ctypes.CDLL(so)
    p = ctypes.c_void_p
    L.cold_host_cell.argtypes = [p, p, p, ctypes.c_int64, p, ctypes.c_int, p, ctypes.c_int, ctypes.c_int, p]

    def run(x, thr, doy_map, defs, seasons, cold=True):
        x = np.ascontiguousarray(x, np.float32)
        thr = np.ascontiguousarray(thr, np.float64)
        dm = np.ascontiguousarray(doy_map, np.int32)
        df = np.ascontiguousarray(defs, np.int32).reshape(-1, 3)
        sn = np.ascontiguousarray(seasons, np.int32).reshape(-1, 2)
        out = np.full((3, df.shape[0], sn.shape[0]), -7.0, np.float32)
        rc = L.cold_host_cell(x.ctypes.data, thr.ctypes.data, dm.ctypes.data, x.size, df.ctypes.data, df.shape[0],
                              sn.ctypes.data, sn.shape[0], int(cold), out.ctypes.data)
        return rc, out
    return run


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def neg(x, thr):
    return -np.asarray(x, np.float32), -np.asarray(thr, np.float64)


def check(replay, x, thr, dm, defs, seasons):
    """The cold replay against both heatwave oracles on (-x, -thr); returns it."""
    rc, got = replay(x, thr, dm, defs, seasons)
    assert rc == 0
    nx, nt = neg(x, thr)
    want = np.stack([intensity_oracle.np_intensity(nx, nt, dm, *d, seasons) for d in defs], axis=1)      # [3, D, Y]
    assert np.array_equal(bits(got), bits(want)), (got, want)
    want_c = np.stack([intensity_oracle.heatwave_intensity(nx, nt, dm, *d, seasons) for d in defs], axis=1)
    assert np.array_equal(bits(got), bits(want_c))
    return got


def test_negation_identity():
    # thr - x == (-x) - (-thr) bit for bit, and x < thr <=> -x > -thr, for float32 x against float64 thr (the oracle's premise)
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.normal(0, 30, 20000), [np.nan, np.inf, -np.inf, 0.0, -0.0, 3.4e38, -3.4e38]]).astype(np.float32)
    thr = np.concatenate([rng.normal(0, 30, 20000), [np.nan, np.inf, -np.inf, -0.0, 0.0, 1e300, -1e300]])
    thr[::7] = x[::7].astype(np.float64)                            # ties
    thr[1::7] = np.nextafter(x[1::7].astype(np.float64), np.inf)
    thr[2::7] = np.nextafter(x[2::7].astype(np.float64), -np.inf)
    xd = x.astype(np.float64)
    with np.errstate(invalid="ignore"):
        assert np.array_equal(xd < thr, -xd > -thr)
        d1, d2 = thr - xd, (-xd) - (-thr)
    assert np.array_equal(np.isnan(d1), np.isnan(d2))
    ok = ~np.isnan(d1)
    assert np.array_equal((d1[ok] + 0.0).view(np.uint64), (d2[ok] + 0.0).view(np.uint64))


def test_hand_case(replay):
    thr = np.array([-1.0])
    T = 24
    x = np.zeros(T, np.float32)
    x[2:7] = [-1.5, -2.25, -3.0, -1.75, -2.5]                       # one 5-day cold spell
    x[8] = -2.0                                                     # break day 7 -> 1-day run 8 (a sub-event of [3, 1, 1])
    x[15:24] = -1.25                                                # a run open at the end of the series
    defs = [[3, 0, 0], [3, 1, 1], [1, 0, 0]]
    seasons = [[0, 4], [4, 12], [12, 30]]
    got = check(replay, x, thr, np.zeros(T), defs, seasons)
    assert got[0, 0, 0] == np.float32(0.5 + 1.25) and got[2, 0, 0] == np.float32(1.25)      # days 2, 3 of the spell
    assert got[0, 0, 1] == np.float32(2.0 + 0.75 + 1.5) and got[0, 1, 1] == np.float32(4.25 + 1.0)
    assert got[1, 0, 2] == np.float32(0.25) and got[0, 2, 2] == np.float32(9 * 0.25)


def test_nan_and_infinite_samples_and_thresholds(replay):
    x = np.array([-2, -2, np.nan, -2, -2, -2, -np.inf, -2, -2, np.inf, -2, -2, -2, -5], np.float32)
    thr = np.array([-1.0, np.nan, -np.inf, np.inf])
    dm = np.zeros(x.size, np.int64)
    dm[11] = 1                                                     # NaN threshold: never cold
    got = check(replay, x, thr, dm, [[2, 0, 0], [3, 0, 0]], [[0, 14]])
    assert np.isinf(got[:, :, 0]).all()                            # -inf is cold: CSC, CSI, CSP are inf
    dm[:] = 2                                                      # nothing is below -inf
    got = check(replay, x, thr, dm, [[1, 0, 0]], [[0, 14]])
    assert (got == 0).all()
    dm[:] = 3                                                      # every finite and -inf sample is below +inf: deficit inf
    got = check(replay, x, thr, dm, [[1, 0, 0]], [[0, 14]])
    assert np.isinf(got).all()


@pytest.mark.parametrize("T", [1, 31, 32, 33, 97, 400, 1500])
def test_random_series_many_definitions(replay, T):
    rng = np.random.default_rng(T + 5)
    for trial in range(12):
        n_doy = int(rng.integers(1, 40))
        dm = np.arange(T) % n_doy
        if trial % 3 == 0:
            dm = (np.arange(T) * 3) % n_doy                           # days of year that are not consecutive: short words
        thr = rng.normal(0.0, 1.0, n_doy)
        z = rng.standard_normal(T)
        for t in range(1, T):
            z[t] = 0.7 * z[t - 1] + 0.7 * z[t]
        x = (z + rng.uniform(-1, 1)).astype(np.float32)
        if trial % 4 == 1:
            x[rng.integers(0, T, max(1, T // 20))] = np.nan
        if trial % 4 == 2:
            x[rng.integers(0, T, max(1, T // 30))] = rng.choice([np.inf, -np.inf], max(1, T // 30))
            thr[rng.integers(0, n_doy)] = rng.choice([np.nan, np.inf, -np.inf])
        if trial % 6 == 3:
            k = rng.integers(0, T, max(1, T // 10))                   # thresholds a float64 ulp off the samples
            thr[dm[k]] = np.nextafter(x[k].astype(np.float64), rng.choice([np.inf, -np.inf]))
        D = int(rng.integers(1, 33))
        defs = np.stack([rng.integers(0, 7, D), rng.integers(0, 4, D), rng.integers(0, 4, D)], axis=1)
        Y = int(rng.integers(1, 9))
        cuts = np.sort(rng.integers(0, T + 10, 2 * Y))
        seasons = cuts.reshape(Y, 2)[rng.permutation(Y)]               # disjoint, in any order
        seasons = np.where((seasons < T) & (rng.random(seasons.shape) < 0.3), seasons - T, seasons)
        got = check(replay, x, thr, dm, defs, seasons)
        assert (got >= 0).all()                                        # a deficit is positive on every cold-spell day
        rc, warm = replay(x, thr, dm, defs, seasons, cold=False)       # the replay's heatwave direction is the heatwave oracle
        assert rc == 0 and np.array_equal(bits(warm), bits(np.stack(
            [intensity_oracle.np_intensity(x, thr, dm, *d, seasons) for d in defs], axis=1)))


# ------------------------------------------------------------------------------------------------ the C ABI
def test_abi_flag_and_version():
    with open(os.path.join(ROOT, "include", "hdp_b200.h")) as f:
        header = f.read()
    assert re.search(r"^#define HDP_B200_COLD 0x100$", header, re.M)
    assert re.search(r"^#define HDP_B200_ABI_VERSION 6$", header, re.M)
    from hdp_b200 import _core, _lib
    assert _core.COLD == 0x100
    assert _core.COLD_METRIC_NAMES == ("CSF", "CSN", "CSD", "CSA") and _core.COLD_INTENSITY_NAMES == ("CSC", "CSI", "CSP")
    assert _lib.lib().hdp_b200_abi_version() == 6


def test_entry_points_decode_the_flag():
    # an empty run (C = 0) gets as far as the argument checks and returns before it touches a device
    from hdp_b200 import _lib
    L = _lib.lib()
    defs = np.array([[3, 0, 0]], np.int32)
    seas = np.zeros((1, 2), np.int32)
    ws = np.zeros(1 << 20, np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)              # noqa: E731

    def metrics(unit):
        return L.hdp_b200_metrics(None, 0, 0, 1, 1, None, 1, 1, None, p(defs), 1, p(seas), p(seas), 1, None, None,
                                  p(ws), ws.size, None, unit)

    def intensity(unit):
        return L.hdp_b200_intensity(None, 0, 0, 1, 1, None, 1, 1, None, p(defs), 1, p(seas), p(seas), 1, None, None, None,
                                    p(ws), ws.size, None, unit)
    for fn in (metrics, intensity):
        for unit in (0, 1, 2, 0x100, 0x101, 0x102):
            assert fn(unit) == 0, (fn, unit)
        for unit in (3, 0x103, 0x200, 0x300, -1, 0x100 | 0x80):
            assert fn(unit) == -1, (fn, unit)
    # thresholds have no direction
    ti, wr, q = np.zeros((1, 1), np.int32), np.zeros((1, 1), np.int32), np.array([0.05])
    for unit, rc in ((0, 0), (0x100, -1), (0x102, -1)):
        assert L.hdp_b200_thresholds(None, 0, 1, 1, 1, p(ti), p(wr), 1, 1, 1, p(q), 1, None, p(ws), ws.size, None, unit) == rc
    assert L.hdp_b200_thresholds_workspace_bytes(0, 1, 1, 1, 1, 1, 1, 1, 0) >= 0


# ------------------------------------------------------------------------------------------------ the Python layer
@pytest.fixture
def fake_pass(monkeypatch):
    """_core.metrics_host / intensity_host replaced by recorders that fill every plane i with i + 1 (metrics) or i + 0.5
    (intensity): the metric layer's tables, flags and names can then be checked without a device."""
    from hdp_b200 import _core
    calls = []

    def metrics_host(x, thr, dm, defs, north, south, is_south, out=None, units=None, *, cold=False):
        calls.append(dict(north=np.asarray(north), south=np.asarray(south), cold=cold, intensity=False))
        P, D, Y, C = thr.shape[2], len(defs), len(north), x.shape[1]
        return np.broadcast_to(np.arange(1, 5, dtype=np.uint16)[:, None, None, None, None], (4, P, D, Y, C)).copy()

    def intensity_host(x, thr, dm, defs, north, south, is_south, out=None, metrics_out=None, units=None, *, cold=False):
        met = metrics_host(x, thr, dm, defs, north, south, is_south, cold=cold)
        calls[-1]["intensity"] = True
        metrics_out[...] = met
        return np.broadcast_to((np.arange(3, dtype=np.float32) + 0.5)[:, None, None, None, None], (3,) + met.shape[1:]).copy()
    monkeypatch.setattr(_core, "metrics_host", metrics_host)
    monkeypatch.setattr(_core, "intensity_host", intensity_host)
    return calls


def _measure_and_threshold():
    from hdp_b200 import utils, xr
    m = utils.generate_test_warming_dataarray("2000-01-01", "2003-12-31", grid_shape=(2, 3)).astype(np.float32)
    lat, lon = xr.coord_values(m, "lat"), xr.coord_values(m, "lon")
    thr = xr.DataArray(np.zeros((2, 3, 365, 2)), dims=["lon", "lat", "doy", "percentile"],
                       coords={"lon": lon, "lat": lat, "doy": np.arange(1, 366), "percentile": np.array([0.05, 0.1])}, name="t",
                       attrs={})
    return m, thr


@pytest.mark.parametrize("intensity", [False, True])
def test_metric_layer_cold_variables_and_seasons(fake_pass, intensity):
    from hdp_b200 import _tables as tb, metric, utils, xr
    m, thr = _measure_and_threshold()
    defs = [[3, 0, 0], [3, 1, 1]]
    warm = metric.compute_individual_metrics(m, thr, defs, check_variables=False, intensity=intensity)
    cold = metric.compute_individual_metrics(m, thr, defs, check_variables=False, intensity=intensity, cold=True)
    st = tb.hemisphere_ranges(utils.time_axis_of(m))
    w, c = fake_pass
    assert not w["cold"] and np.array_equal(w["north"], st.north) and np.array_equal(w["south"], st.south)
    assert c["cold"] and np.array_equal(c["north"], st.south) and np.array_equal(c["south"], st.north)   # the swapped tables
    assert w["intensity"] == c["intensity"] == intensity
    names = ["CSF", "CSN", "CSD", "CSA"] + (["CSC", "CSI", "CSP"] if intensity else [])
    assert sorted(cold.keys()) == sorted(names)
    assert sorted(warm.keys()) == sorted(["HWF", "HWN", "HWD", "HWA"] + (["HWC", "HWI", "HWP"] if intensity else []))
    for cn, wn in zip(names, ["HWF", "HWN", "HWD", "HWA", "HWC", "HWI", "HWP"]):
        a, b = cold[cn], warm[wn]
        assert tuple(a.dims) == tuple(b.dims) and a.shape == b.shape and xr.values_of(a).dtype == xr.values_of(b).dtype
        assert np.array_equal(xr.values_of(a), xr.values_of(b))                           # the same plane of the output
        for d in a.dims:
            assert repr(xr.coord_values(a, d)) == repr(xr.coord_values(b, d))             # (small coordinates, time stamps too)
        assert re.sub(r"\(\d{4}-\d\d-\d\d \d\d:\d\d\) ", "", a.attrs["history"]) == \
            re.sub(r"\(\d{4}-\d\d-\d\d \d\d:\d\d\) ", "", b.attrs["history"])
        attrs = {**metric.COLD_METRIC_ATTRS, **metric.COLD_INTENSITY_ATTRS}[cn]
        assert all(a.attrs[k] == v for k, v in attrs.items())
        assert "cold spell" in a.attrs["description"] and "heat" not in a.attrs["description"].lower()
    assert cold["CSF"].attrs["long_name"] == "Cold Spell Frequency"
    assert cold["definition"].attrs["first_number"] == "Minimum number of consecutively cold days"
    assert warm["definition"].attrs["first_number"] == "Minimum number of consecutively hot days"
    assert cold.attrs["hdp_type"] == "metric" and cold.attrs["description"].startswith("Cold spell metric dataset")
    assert cold["CSF"].attrs["description"] == "Number of days that fall within a cold spell during a cold season"
    if intensity:
        assert cold["CSC"].attrs["units"] == m.attrs["units"] and "deficit" in cold["CSC"].attrs["description"]


def test_group_metrics_cold_names(fake_pass):
    from hdp_b200 import metric
    m, thr = _measure_and_threshold()
    m.attrs["baseline_variable"] = thr.attrs["baseline_variable"] = "t"
    ds = metric.compute_group_metrics({"t": m}, {"t_threshold": thr}, [[3, 0, 0]], check_variables=False, cold=True, intensity=True)
    assert sorted(ds.keys()) == sorted(f"t.t_threshold.{n}" for n in ("CSF", "CSN", "CSD", "CSA", "CSC", "CSI", "CSP"))
    assert [c["cold"] for c in fake_pass] == [True]
