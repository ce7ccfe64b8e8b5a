"""Trend statistics without a GPU: the NumPy oracle of tests/trend_oracle.py against scipy.stats.theilslopes and kendalltau, the
stdlib normal quantile against scipy's, the g++ replay of hdp_b200/csrc/trend.h (tests/trend_host.cpp) against the oracle bit for bit,
the argument checks of _core and the metric layer with the replay in place of the device call.  The kernel itself is checked by
tests/test_gpu_trend.py."""
import ctypes
import math
import os
import subprocess
from statistics import NormalDist

import numpy as np
import pytest

from conftest import bits_equal
from trend_oracle import NAMES, ranks, series, trend_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
scipy_stats = pytest.importorskip("scipy.stats")
from scipy.special import ndtri  # noqa: E402

ZQ = NormalDist().inv_cdf(0.025)


@pytest.fixture(scope="module")
def replay(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("trend") / "libtrend_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-shared", "-fPIC", "-I",
                    os.path.join(ROOT, "hdp_b200", "csrc"), os.path.join(ROOT, "tests", "trend_host.cpp"), "-o", so], check=True)
    L = ctypes.CDLL(so)
    L.trend_host.restype = ctypes.c_int
    L.trend_host.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                             ctypes.c_double, ctypes.c_void_p]

    def run(x, zq=ZQ, missing=None):
        x = np.ascontiguousarray(x)
        rows, Y, C = x.shape
        out = np.empty((8, rows, C))
        dtype = 1 if x.dtype == np.uint16 else 2
        rc = L.trend_host(x.ctypes.data, dtype, rows, Y, C, -1 if missing is None else missing, zq, out.ctypes.data)
        assert rc == 0
        return out
    return run


def random_series(rng, kind, Y, C):
    """[1, Y, C] uint16 or float32 series of one kind, with ties, gaps and the degenerate columns the contract names."""
    if kind == "poisson":
        x = rng.poisson(rng.uniform(0.2, 6, C)[None, :] + 0.03 * np.arange(Y)[:, None]).astype(np.uint16)
        x[rng.random((Y, C)) < 0.1] = 0xFFFF
    elif kind == "high":
        x = (65534 - rng.integers(0, 4, (Y, C))).astype(np.uint16)
    elif kind == "float":
        x = (rng.standard_normal((Y, C)) + 0.02 * np.arange(Y)[:, None]).astype(np.float32)
        x[rng.random((Y, C)) < 0.1] = np.nan
        x[rng.random((Y, C)) < 0.03] = np.inf
        x[rng.random((Y, C)) < 0.03] = -np.inf
        x[rng.random((Y, C)) < 0.05] = 0.0
        x[rng.random((Y, C)) < 0.05] = -0.0
        x[:, 0] = np.round(x[:, 0])                                 # ties
    if x.dtype == np.uint16:
        x[:, -1] = 0xFFFF                                           # empty with the sentinel
        if C > 1:
            x[:, -2] = 7                                            # all equal
        if C > 2:
            x[:, -3] = 0xFFFF
            x[Y // 2, -3] = 3                                       # one valid season
    else:
        x[:, -1] = np.nan
        if C > 1:
            x[:, -2] = 1.5
        if C > 2:
            x[:, -3] = np.nan
            x[Y // 2, -3] = 2.0
    return x[None]


def test_stdlib_quantile_matches_ndtri():
    for alpha in (0.001, 0.01, 0.05, 0.1, 0.2, 0.5, 0.9):
        zq = NormalDist().inv_cdf(alpha / 2)
        assert abs(zq - ndtri(alpha / 2)) <= 1e-15 * abs(zq)


@pytest.mark.parametrize("seed", range(4))
def test_oracle_against_scipy(seed):
    rng = np.random.default_rng(seed)
    for Y in (2, 3, 5, 17, 40, 86):
        for kind in ("poisson", "float"):
            x = random_series(rng, kind, Y, 6)[0]
            for c in range(x.shape[1]):
                y = x[:, c]
                miss = 0xFFFF if kind == "poisson" else None
                o = series(y, ZQ, miss if y.dtype == np.uint16 else None)
                valid = np.isfinite(y) if y.dtype != np.uint16 else y != 0xFFFF
                idx = np.flatnonzero(valid)
                v = y[idx].astype(np.float64)
                assert o[7] == idx.size
                if idx.size < 2:
                    assert np.isnan(o[[0, 1, 2, 3, 6]]).all() and o[4] == 0 and o[5] == 0
                    continue
                zq = ndtri(0.025)
                res = scipy_stats.theilslopes(v, idx.astype(np.float64), alpha=0.95)
                assert math.isclose(o[0], res[0], rel_tol=1e-12, abs_tol=1e-300)
                assert math.isclose(o[1], res[1], rel_tol=1e-12, abs_tol=1e-12)
                mine = series(y, zq, miss if y.dtype == np.uint16 else None)
                # scipy scales the variance by 1/18. instead of dividing by 18: where that last bit moves rint across a half the ranks
                # differ; such a series is left out
                N = idx.size * (idx.size - 1) // 2
                scaled = 1 / 18. * (mine[5] * 18.0)
                if ranks(N, mine[5], zq) == ranks(N, scaled, zq):
                    assert mine[2] == res[2] and mine[3] == res[3]
                # Mann-Kendall against kendalltau (x = season index has no ties): tau-b and the asymptotic p-value without continuity
                t = np.unique(v, return_counts=True)[1]
                n0, n2 = N, int((t * (t - 1) // 2).sum())
                if idx.size < 3 or n0 - n2 == 0:                      # kendalltau's asymptotic variance divides by n - 2
                    continue
                kt = scipy_stats.kendalltau(idx, v, method="asymptotic")
                assert math.isclose(kt.statistic, o[4] / math.sqrt(n0 * (n0 - n2)), rel_tol=1e-12, abs_tol=1e-15)
                assert math.isclose(kt.pvalue, math.erfc(abs(o[4]) / math.sqrt(o[5]) / math.sqrt(2)), rel_tol=1e-9, abs_tol=1e-300)


def test_oracle_median_and_rank_rules():
    # odd N (n = 3): the middle slope; even N (n = 4): the mean of the two middle ones
    y = np.array([0, 1, 3], np.float32)                             # slopes 1, 1.5, 2
    assert series(y, ZQ)[0] == 1.5
    y = np.array([0, 1, 3, 4], np.float32)                          # slopes 1, 1.5, 4/3, 2, 1.5, 1 -> sorted 1 1 4/3 1.5 1.5 2
    assert series(y, ZQ)[0] == (4 / 3 + 1.5) * 0.5
    # CI ranks at both clamps: n = 2 has N = 1, both bounds the one slope
    o = series(np.array([2, 5], np.uint16), ZQ)
    assert o[0] == o[2] == o[3] == 3.0


@pytest.mark.parametrize("kind", ["poisson", "high", "float"])
@pytest.mark.parametrize("Y", [1, 2, 3, 4, 33, 86, 251, 512])
def test_replay_matches_oracle(replay, kind, Y):
    rng = np.random.default_rng(Y * 7 + len(kind))
    C = 5 if Y >= 251 else 9
    x = random_series(rng, kind, Y, C)
    miss = 0xFFFF if x.dtype == np.uint16 and kind != "high" else None
    got = replay(x, missing=miss)
    want = trend_batch(x, ZQ, miss)
    for q, name in enumerate(NAMES):
        assert bits_equal(got[q], want[q]), name


def test_replay_signed_zero_and_alpha(replay):
    x = np.array([[0.0, -0.0, 0.0, -0.0, 1.0], [-0.0, 0.0, -0.0, 0.0, -1.0]], np.float32).T[None]
    for alpha in (0.01, 0.05, 0.5):
        zq = NormalDist().inv_cdf(alpha / 2)
        got, want = replay(x, zq), trend_batch(x, zq)
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(got), nan) and np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64))


def test_core_trend_arguments():
    from hdp_b200 import _core
    code, rows, Y, C, miss, zq = _core._trend_args("uint16", (6, 10, 86, 100), 0xFFFF, 0.05)
    assert (code, rows, Y, C, miss) == (_core.DTYPE_U16, 60, 86, 100, 0xFFFF) and zq == NormalDist().inv_cdf(0.025)
    assert _core._trend_args("float32", (3, 2, 7), None, 0.1)[:5] == (_core.DTYPE_F32, 3, 2, 7, -1)
    assert _core._trend_args("uint16", (5, 4), None, 0.05)[1:5] == (1, 5, 4, -1)
    with pytest.raises(ValueError):
        _core._trend_args("float32", (2, 3), 0xFFFF, 0.05)
    with pytest.raises(ValueError):
        _core._trend_args("uint16", (2, 3), 70000, 0.05)
    with pytest.raises(ValueError):
        _core._trend_args("uint16", (2, 3), None, 1.0)
    with pytest.raises(TypeError):
        _core._trend_args("float64", (2, 3), None, 0.05)
    with pytest.raises(ValueError):
        _core._trend_args("uint16", (3,), None, 0.05)
    assert _core.TREND_NAMES == NAMES


def test_metric_layer_with_replay(replay, monkeypatch):
    from hdp_b200 import _core, metric, xr
    calls = []

    def trend_host(values, *, missing=None, alpha=0.05):
        calls.append((values.dtype, values.shape, missing, np.shares_memory(values, src_u16)))
        flat = values.reshape(-1, *values.shape[-2:])
        return replay(flat, NormalDist().inv_cdf(alpha / 2), missing).reshape(8, *values.shape[:-2], values.shape[-1])
    monkeypatch.setattr(_core, "trend_host", trend_host)

    rng = np.random.default_rng(5)
    P, D, Y, nlat, nlon = 2, 3, 20, 2, 3
    src_u16 = rng.poisson(3, (P, D, Y, nlat * nlon)).astype(np.uint16)
    hwf = src_u16.transpose(0, 1, 3, 2).reshape(P, D, nlat, nlon, Y)                   # the metric layer's view of [P, D, Y, C]
    hwo = np.where(rng.random(hwf.shape) < 0.2, np.nan, rng.integers(0, 100, hwf.shape)).astype(np.float32)
    hwc = rng.standard_normal((2, P, D, nlat, nlon, Y)).astype(np.float32)
    hwc[0, 0, 0, 0, 0, :3] = np.inf
    coords = {"percentile": np.array([0.9, 0.95]), "definition": ["3-0-0", "3-1-1", "4-0-0"], "lat": np.array([-10.0, 10.0]),
              "lon": np.array([0.0, 1.0, 2.0]), "time": np.arange(Y)}
    dims = ["percentile", "definition", "lat", "lon", "time"]
    ds = xr.Dataset({
        "HWF": xr.DataArray(hwf, dims=dims, coords=coords, attrs={"units": "heatwave days"}),
        "HWO": xr.DataArray(hwo, dims=dims, coords=coords, attrs={"units": "days"}),
        "HWC": xr.DataArray(hwc, dims=["measure", *dims], coords={**coords, "measure": ["tmax", "tmin"]}, attrs={"units": "degC"}),
    })
    out = metric.compute_metric_trends(ds, alpha=0.1)
    assert sorted(out.keys()) == sorted(f"{v}_{s}" for v in ("HWF", "HWO", "HWC") for s in NAMES)
    assert out.attrs["alpha"] == 0.1 and "Theil-Sen" in out.attrs["trend_method"]
    assert calls[0][:3] == (np.uint16, (P, D, Y, nlat * nlon), None) and calls[0][3]                 # a view, no copy
    assert calls[1][0] == np.float32 and calls[2][1] == (2, P, D, Y, nlat * nlon)
    zq = NormalDist().inv_cdf(0.05)
    want = trend_batch(src_u16.reshape(P * D, Y, -1), zq)
    for q, s in enumerate(NAMES):
        a = out[f"HWF_{s}"]
        assert tuple(a.dims) == ("percentile", "definition", "lat", "lon")
        assert bits_equal(np.asarray(xr.values_of(a)), want[q].reshape(P, D, nlat, nlon))
        assert "time" not in a.coords and np.array_equal(xr.coord_values(a, "lon"), coords["lon"])
    assert tuple(out["HWC_slope"].dims) == ("measure", "percentile", "definition", "lat", "lon")
    want_c = trend_batch(np.moveaxis(hwc, -1, 3).reshape(2 * P * D, Y, -1), zq)
    assert bits_equal(np.asarray(xr.values_of(out["HWC_slope"])).reshape(2 * P * D, -1), want_c[0])
    assert out["HWC_n"].values[0, 0, 0, 0, 0] == Y - 3
    want_o = trend_batch(np.moveaxis(hwo, -1, 2).reshape(P * D, Y, -1), zq)
    assert bits_equal(np.asarray(xr.values_of(out["HWO_slope"])).reshape(P * D, -1), want_o[0])
    assert out["HWF_slope"].attrs["units"] == "heatwave days per year" and out["HWF_intercept"].attrs["units"] == "heatwave days"
    assert out["HWC_slope_low"].attrs["units"] == "degC per year" and "90 %" in out["HWC_slope_low"].attrs["long_name"]
    only = metric.compute_metric_trends(ds, variables=["HWO"])
    assert sorted(only.keys()) == sorted(f"HWO_{s}" for s in NAMES)
