"""Heatwave onset and end (HWO, HWE) without a GPU: the oracle of tests/onset_oracle.py against an independent restatement and
against the reference's HWF / HWD through the contract's invariants, the packed accumulator update of k_scan's ONSET variant
(hdp_b200/csrc/seams.h) for every lane pattern, the flag of the C ABI and the metric layer's variables.  The kernels themselves are
checked by tests/test_gpu_onset.py."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from onset_oracle import NO_DAY, cold_onset_batch, compound_onset_batch, onset_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def index_heatwaves_py(hot, min_duration, max_break, max_subs):
    """The reference's index_heatwaves (hdp/metric.py:11-60) restated over the hot runs: branches A - D per run, in time order."""
    hot = np.asarray(hot, bool)
    edges = np.flatnonzero(np.diff(np.concatenate([[0], hot.astype(np.int8), [0]])))
    hw = np.zeros(hot.size, np.int64)
    idx, sub, in_hw, prev_e = 0, 0, False, None
    for s, e in zip(edges[::2], edges[1::2]):
        if prev_e is not None and s - prev_e > max_break:
            in_hw = False
        prev_e = e
        if e - s >= min_duration and not in_hw:
            idx, in_hw, label = idx + 1, True, idx + 1
        elif in_hw and sub < max_subs:
            sub, label = sub + 1, idx
        elif in_hw:
            label, sub = 0, 0
            if e - s >= min_duration:
                idx += 1
                label = idx
            else:
                in_hw = False
        else:
            label = 0
        hw[s:e] = label
    return hw


def onset_restated(x, thr, dm, defs, north, south, is_south):
    """uint16 [2, P, D, Y, C] with NumPy only: hot days, the restated ids, first / last positive id of each slice via argmax."""
    T, C = x.shape
    P = thr.shape[2]
    out = np.empty((2, P, len(defs), len(north), C), np.uint16)
    for c in range(C):
        seasons = south if is_south[c] else north
        for p in range(P):
            with np.errstate(invalid="ignore"):
                hot = x[:, c].astype(np.float64) > thr[c, dm, p]
            for d, df in enumerate(defs):
                hw = index_heatwaves_py(hot, *df)
                for y, (a, b) in enumerate(seasons):
                    lo, hi, _ = slice(int(a), int(b)).indices(T)
                    pos = hw[lo:max(lo, hi)] > 0
                    if not pos.any():
                        out[:, p, d, y, c] = NO_DAY
                    else:
                        out[:, p, d, y, c] = np.argmax(pos), pos.size - 1 - np.argmax(pos[::-1])
    return out


def ar1(seed, T, C, P, n_doy=365):
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
    x = z.astype(np.float32)
    x[rng.integers(0, T, 5), rng.integers(0, C, 5)] = np.nan
    thr = np.linspace(0.3, 1.2, P)[None, None, :] + 0.2 * rng.standard_normal((C, n_doy, 1))
    dm = np.arange(T) % n_doy
    return x, thr, dm


DEFS = [[3, 0, 0], [3, 1, 1], [1, 0, 0], [4, 2, 2], [2, 3, 5]]
# seasons that cross the series' ends, negative and out-of-range entries, an empty and a reversed one, a one-day one, overlaps
NORTH = [[100, 250], [-400, -100], [700, 5000], [300, 300], [500, 400], [365, 366], [200, 600]]
SOUTH = [[-5000, 80], [280, 430], [0, 1095], [-1, 2000], [640, 730], [1000, -50], [50, 51]]


def test_oracle_matches_an_independent_restatement():
    x, thr, dm = ar1(1, 3 * 365, 11, 3)
    is_south = (np.arange(11) % 2).astype(np.uint8)
    args = (dm, DEFS, NORTH, SOUTH, is_south)
    got = onset_batch(x, thr, *args)
    assert np.array_equal(got, onset_restated(x, thr, *args))
    assert (got != NO_DAY).any() and (got == NO_DAY).any()


@pytest.mark.parametrize("cold", [False, True])
def test_oracle_invariants_against_the_reference_metrics(cold):
    x, thr, dm = ar1(2, 4 * 365, 13, 4)
    is_south = (np.arange(13) % 3 == 0).astype(np.uint8)
    args = (dm, DEFS, NORTH, SOUTH, is_south)
    on = (cold_onset_batch if cold else onset_batch)(x, thr, *args).astype(np.int64)
    s = -1.0 if cold else 1.0
    met = oracle.metrics_batch((s * x).astype(np.float32), s * thr, *args)          # [P, D, C, 4, Y]
    hwf, hwd = met[..., 0, :].transpose(0, 1, 3, 2), met[..., 2, :].transpose(0, 1, 3, 2)   # [P, D, Y, C]
    o, e = on
    none = hwf == 0
    assert np.array_equal(o == NO_DAY, none) and np.array_equal(e == NO_DAY, none)
    assert none.any() and (~none).any()
    assert (o[~none] <= e[~none]).all()
    assert (e[~none] - o[~none] + 1 >= hwf[~none]).all() and (hwf >= hwd).all()
    # a value is a day of the clamped slice
    T = x.shape[0]
    length = np.array([[len(range(T)[a:b]) for a, b in tab] for tab in (NORTH, SOUTH)])     # [2, Y]
    lens = length[is_south.astype(int)].T[None, None]                                      # [1, 1, Y, C]
    assert (np.broadcast_to(lens, e.shape)[~none] > e[~none]).all()


def test_clipping_at_the_season_ends():
    # one run over days 90 .. 119, one definition labelling it: a season starting inside it gets HWO 0, one ending inside it HWE
    # hi - lo - 1
    T = 200
    x = np.zeros((T, 1), np.float32)
    x[90:120] = 1.0
    thr = np.full((1, 1, 1), 0.5)
    seasons = [[100, 150], [50, 110], [95, 105], [0, 90], [119, 120], [120, 200]]
    got = onset_batch(x, thr, np.zeros(T, np.int64), [[3, 0, 0]], seasons, seasons, None)[:, 0, 0, :, 0]
    assert got.T.tolist() == [[0, 19], [40, 59], [0, 9], [NO_DAY, NO_DAY], [0, 0], [NO_DAY, NO_DAY]]


def test_compound_of_one_measure_is_the_single_result():
    x, thr, dm = ar1(4, 2 * 365, 7, 2)
    is_south = (np.arange(7) % 2).astype(np.uint8)
    args = (dm, DEFS[:3], NORTH[:3], SOUTH[:3], is_south)
    for cold in (False, True):
        single = (cold_onset_batch if cold else onset_batch)(x, thr, *args)
        assert np.array_equal(compound_onset_batch(x, thr, x, thr, *args, cold=cold), single)


# ------------------------------------------------------------------------------------------------ the packed update
@pytest.fixture(scope="module")
def onset_host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("onset") / "libscan_onset_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-I", os.path.join(ROOT, "hdp_b200", "csrc"),
                    os.path.join(ROOT, "tests", "scan_onset_host.cpp"), "-o", so], check=True)
    L = ctypes.CDLL(so)
    L.scan_onset_mismatches.restype = ctypes.c_int64
    L.scan_onset_value_mismatches.restype = ctypes.c_int64
    return L


@pytest.mark.parametrize("bits", [8, 16])
def test_packed_update_every_lane_pattern(onset_host, bits):
    bad = (ctypes.c_uint32 * 6)()
    n = onset_host.scan_onset_mismatches(bits, bad)
    assert n == 0, "%d cases differ, first %s" % (n, list(bad))


def test_stored_value_and_sentinel(onset_host):
    assert onset_host.scan_onset_value_mismatches() == 0


# ------------------------------------------------------------------------------------------------ the C ABI (host logic)
def test_flag_value_matches_the_header():
    from hdp_b200 import _core, _lib
    header = open(os.path.join(ROOT, "include", "hdp_b200.h")).read()
    assert int(re.search(r"#define HDP_B200_ONSET (0x[0-9a-fA-F]+)", header).group(1), 16) == _core.ONSET == 0x200
    assert _core.ONSET & _core.COLD == 0 and _core.ONSET > 2
    assert _core.ONSET_NAMES == ("HWO", "HWE") and _core.COLD_ONSET_NAMES == ("CSO", "CSE") and _core.NO_DAY == 0xFFFF
    assert _lib.lib().hdp_b200_abi_version() == 6


def test_entry_points_without_a_u16_output_reject_the_flag():
    # an empty run (C = 0) gets as far as the argument checks and returns before it touches a device
    from hdp_b200 import _lib
    L = _lib.lib()
    defs = np.array([[3, 0, 0]], np.int32)
    seas = np.zeros((1, 2), np.int32)
    ws = np.zeros(1 << 20, np.uint8)
    out = np.zeros(64, np.uint16)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)              # noqa: E731
    tab = (p(defs), 1, p(seas), p(seas), 1, None)
    for unit, rc in ((0x200, 0), (0x300, 0), (0x202, 0), (0x203, -1), (0x400, -1)):
        assert L.hdp_b200_metrics(None, 0, 0, 1, 1, None, 1, 1, None, *tab, p(out), p(ws), ws.size, None, unit) == rc, unit
    for unit in (0x200, 0x300):
        assert L.hdp_b200_intensity(None, 0, 0, 1, 1, None, 1, 1, None, *tab, None, None, p(ws), ws.size, None, unit) == -1
        assert L.hdp_b200_intensity(None, 0, 0, 1, 1, None, 1, 1, None, *tab, None, p(out), p(ws), ws.size, None, unit) == 0
        assert L.hdp_b200_compound(None, 1, 1, None, 1, 1, 0, 0, None, None, 1, 1, None, *tab, None, None, p(ws), ws.size, None,
                                   unit) == -1
        assert L.hdp_b200_compound(None, 1, 1, None, 1, 1, 0, 0, None, None, 1, 1, None, *tab, p(out), None, p(ws), ws.size, None,
                                   unit) == 0
        # the host pipeline checks before it looks for a device; only the intensity and compound calls may omit h_out
        x = np.zeros((4, 1), np.float32)
        assert L.hdp_b200_intensity_host(p(x), 0, 4, 1, 1, None, None, 1, 1, p(np.zeros(4, np.int32)), *tab, None, None, unit) == -1
        assert L.hdp_b200_compound_host(p(x), 1, 1, p(x), 1, 1, 0, 4, None, None, None, None, 1, 1, p(np.zeros(4, np.int32)), *tab,
                                        None, p(np.zeros(1, np.float32)), unit) == -1
    # the threshold entry points reject the bit through their unit check
    ti, wr, q = np.zeros((1, 1), np.int32), np.zeros((1, 1), np.int32), np.array([0.9])
    for unit, rc in ((0, 0), (0x200, -1), (0x201, -1)):
        assert L.hdp_b200_thresholds(None, 0, 1, 1, 1, p(ti), p(wr), 1, 1, 1, p(q), 1, None, p(ws), ws.size, None, unit) == rc


def test_python_layer_needs_metrics_out_with_onset():
    from hdp_b200 import _core
    with pytest.raises(ValueError, match="metrics_out"):
        _core._check_onset(None, True, True)
    _core._check_onset(None, False, True)
    _core._check_onset(None, True, False)


# ------------------------------------------------------------------------------------------------ the metric layer
def six_planes(P, D, Y, C):
    """uint16 [6, P, D, Y, C]: planes 0 - 3 = 1 .. 4, HWO = 10 y + c, HWE = 20 + y except NO_DAY where (y + c) % 3 == 0."""
    out = np.broadcast_to(np.arange(1, 7, dtype=np.uint16)[:, None, None, None, None], (6, P, D, Y, C)).copy()
    y, c = np.meshgrid(np.arange(Y), np.arange(C), indexing="ij")
    none = (y + c) % 3 == 0
    out[4] = np.where(none, NO_DAY, 10 * y + c)[None, None]
    out[5] = np.where(none, NO_DAY, 20 + y)[None, None]
    return out


@pytest.fixture
def fake_onset(monkeypatch):
    """_core's host metric calls replaced by recorders that return six_planes (or four without onset) and intensity plane i = i + 0.5."""
    from hdp_b200 import _core
    calls = []

    def metrics(x, thr, defs, north, cold, onset):
        calls.append(dict(north=np.asarray(north), cold=cold, onset=onset))
        full = six_planes(thr.shape[2], len(defs), len(north), x.shape[1])
        return full if onset else full[:4].copy()

    def metrics_host(x, thr, dm, defs, north, south, is_south, out=None, units=None, *, cold=False, onset=False):
        return metrics(x, thr, defs, north, cold, onset)

    def intensity_host(x, thr, dm, defs, north, south, is_south, out=None, metrics_out=None, units=None, *, cold=False, onset=False):
        metrics_out[...] = metrics(x, thr, defs, north, cold, onset)
        return np.broadcast_to((np.arange(3, dtype=np.float32) + 0.5)[:, None, None, None, None], (3,) + metrics_out.shape[1:]).copy()

    def compound_metrics_host(xa, ta, xb, tb, dm, defs, north, south, is_south, out=None, units=None, *, cold=False, onset=False):
        return metrics(xa, ta, defs, north, cold, onset)

    def compound_intensity_host(xa, ta, xb, tb, dm, defs, north, south, is_south, out=None, metrics_out=None, units=None, *, cold=False,
                                onset=False):
        metrics_out[...] = metrics(xa, ta, defs, north, cold, onset)
        return np.broadcast_to((np.arange(3, dtype=np.float32) + 0.5)[None, :, None, None, None, None], (2, 3) + metrics_out.shape[1:]).copy()
    for name, fn in (("metrics_host", metrics_host), ("intensity_host", intensity_host), ("compound_metrics_host", compound_metrics_host),
                     ("compound_intensity_host", compound_intensity_host)):
        monkeypatch.setattr(_core, name, fn)
    return calls


def _measure_and_threshold(name="tmax"):
    from hdp_b200 import utils, xr
    m = utils.generate_test_warming_dataarray("2000-01-01", "2003-12-31", grid_shape=(2, 3)).astype(np.float32)
    m = xr.DataArray(xr.values_of(m), dims=list(m.dims), coords=dict(xr.coords_of(m)), name=name, attrs=dict(m.attrs))
    lat, lon = xr.coord_values(m, "lat"), xr.coord_values(m, "lon")
    thr = xr.DataArray(np.zeros((2, 3, 365, 2)), dims=["lon", "lat", "doy", "percentile"],
                       coords={"lon": lon, "lat": lat, "doy": np.arange(1, 366), "percentile": np.array([0.9, 0.95])}, name="t",
                       attrs={})
    return m, thr


@pytest.mark.parametrize("cold", [False, True])
@pytest.mark.parametrize("intensity", [False, True])
def test_metric_layer_onset_variables(fake_onset, cold, intensity):
    from hdp_b200 import metric, xr
    m, thr = _measure_and_threshold()
    defs = [[3, 0, 0], [3, 1, 1]]
    ds = metric.compute_individual_metrics(m, thr, defs, check_variables=False, intensity=intensity, cold=cold, onset=True)
    plain = metric.compute_individual_metrics(m, thr, defs, check_variables=False, intensity=intensity, cold=cold)
    assert [c["onset"] for c in fake_onset] == [True, False]
    o_name, e_name = ("CSO", "CSE") if cold else ("HWO", "HWE")
    f_name = "CSF" if cold else "HWF"
    assert sorted(ds.keys()) == sorted(list(plain.keys()) + [o_name, e_name])
    for n in plain.keys():                                          # the other variables are untouched
        assert np.array_equal(xr.values_of(ds[n]), xr.values_of(plain[n])) and ds[n].attrs.keys() == plain[n].attrs.keys()
    Y, C = 4, 6
    raw = six_planes(2, 2, Y, C)
    for name, plane in ((o_name, 4), (e_name, 5)):
        a = ds[name]
        assert tuple(a.dims) == tuple(ds[f_name].dims) and a.shape == ds[f_name].shape
        for d in a.dims:
            assert repr(xr.coord_values(a, d)) == repr(xr.coord_values(ds[f_name], d))
        v = np.asarray(xr.values_of(a))
        assert v.dtype == np.float32
        want = np.where(raw[plane] == NO_DAY, np.nan, raw[plane].astype(np.float32)).transpose(0, 1, 3, 2).reshape(v.shape)
        assert np.array_equal(v, want, equal_nan=True) and np.isnan(v).any() and not np.isnan(v).all()
        attrs = (metric.COLD_ONSET_ATTRS if cold else metric.ONSET_ATTRS)[name]
        assert all(a.attrs[k] == val for k, val in attrs.items()) and a.attrs["units"] == "days"
        starts = "north Nov 1, south May 1" if cold else "north May 1, south Nov 1"
        assert starts in a.attrs["description"]
        assert ("cold spell" in a.attrs["description"]) == cold
    assert ds[o_name].attrs["long_name"] == ("Cold Spell Onset" if cold else "Heatwave Onset")
    assert ds[e_name].attrs["long_name"] == ("Cold Spell End" if cold else "Heatwave End")
    assert np.nanmean(np.asarray(xr.values_of(ds[o_name]))) < 0xFFFF                   # a mean over years never sees the sentinel


def test_group_metrics_onset_names(fake_onset):
    from hdp_b200 import metric
    m, thr = _measure_and_threshold()
    m.attrs["baseline_variable"] = thr.attrs["baseline_variable"] = "t"
    ds = metric.compute_group_metrics({"t": m}, {"t_threshold": thr}, [[3, 0, 0]], check_variables=False, onset=True)
    assert sorted(ds.keys()) == sorted(f"t.t_threshold.{n}" for n in ("HWF", "HWN", "HWD", "HWA", "HWO", "HWE"))
    assert [c["onset"] for c in fake_onset] == [True]


@pytest.mark.parametrize("cold", [False, True])
def test_compound_metric_layer_onset(fake_onset, cold):
    from hdp_b200 import metric, xr
    ma, thr = _measure_and_threshold("tmax")
    mb, _ = _measure_and_threshold("tmin")
    defs = [[3, 0, 0], [3, 1, 1]]
    ds = metric.compute_compound_metrics(ma, thr, mb, thr, defs, check_variables=False, intensity=True, cold=cold, onset=True)
    o_name, e_name = ("CSO", "CSE") if cold else ("HWO", "HWE")
    f_name, c_name = ("CSF", "CSC") if cold else ("HWF", "HWC")
    assert [c["onset"] for c in fake_onset] == [True]
    assert tuple(ds[c_name].dims)[0] == "measure"
    for name in (o_name, e_name):
        a = ds[name]
        assert tuple(a.dims) == tuple(ds[f_name].dims) and "measure" not in a.dims      # one value per compound season, no measure dim
        assert a.attrs["long_name"] == metric.COMPOUND_LONG_NAMES[name] and a.attrs["long_name"].startswith("Compound ")
        assert "tmax" in a.attrs["description"] and "tmin" in a.attrs["description"] and a.attrs["units"] == "days"
    v = np.asarray(xr.values_of(ds[o_name]))
    raw = six_planes(2, 2, 4, 6)[4]
    assert np.array_equal(v, np.where(raw == NO_DAY, np.nan, raw.astype(np.float32)).transpose(0, 1, 3, 2).reshape(v.shape), equal_nan=True)
    plain = metric.compute_compound_metrics(ma, thr, mb, thr, defs, check_variables=False, cold=cold)
    assert o_name not in plain and e_name not in plain
