"""GPU parity of the heatwave intensity metrics (HWC, HWI, HWP; hdp_b200_intensity, csrc/intensity.cu) against the CPU oracle,
float32 bits equal; the integer metrics of the same pass against hdp_b200_metrics bit for bit; the host pipeline against the
device call; the opt-in of compute_group_metrics; one full-size cmip6_1deg measure."""
import re

import numpy as np
import pytest

import intensity_oracle
import oracle

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def core():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from hdp_b200 import _core
    yield _core
    _core.release_workspaces()
    torch.cuda.empty_cache()


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def ref_layout(heat):
    """float32 [3, P, D, Y, C] -> the oracle's [P, D, C, 3, Y]."""
    return heat.cpu().numpy().transpose(1, 2, 4, 0, 3) if isinstance(heat, torch.Tensor) else heat.transpose(1, 2, 4, 0, 3)


def check(core, x, thr, dm, defs, north, south, is_south, x_celsius=None, units=None, x_dev=None):
    """intensity_array (with metrics_out) against the oracle and against metrics_array; returns the device outputs."""
    P, D, Y, C = thr.shape[2], len(defs), len(north), x.shape[1]
    x_dev = dev(x) if x_dev is None else x_dev
    met = torch.empty((4, P, D, Y, C), dtype=torch.uint16, device="cuda")
    heat = core.intensity_array(x_dev, dev(thr), dm, defs, north, south, is_south, metrics_out=met, units=units)
    want = intensity_oracle.intensity_batch(np.ascontiguousarray(x if x_celsius is None else x_celsius), thr, dm, defs, north, south, is_south)
    assert np.array_equal(bits(ref_layout(heat)), bits(want))
    met_ref = core.metrics_array(x_dev, dev(thr), dm, defs, north, south, is_south, units=units)
    assert torch.equal(met.view(torch.int16), met_ref.view(torch.int16))
    hwf = met.cpu().numpy()[0]
    h = heat.cpu().numpy()
    assert np.array_equal(h[0] > 0, hwf > 0) and np.array_equal(h[2] > 0, hwf > 0)
    return heat, met


def _field(rng, ax, C, warm=2.0):
    doy = ax.dayofyr
    z = rng.standard_normal((len(ax), C))
    for t in range(1, len(ax)):
        z[t] = 0.6 * z[t - 1] + 0.8 * z[t]
    return (15 + 10 * np.sin(2 * np.pi * (doy[:, None] - 110) / 365) + 3 * z + warm).astype(np.float32)


def _thr(rng, C, n_doy, P):
    return (15 + 10 * np.sin(2 * np.pi * (np.arange(n_doy)[None, :, None] - 110) / 365) + np.linspace(1, 6, P)[None, None, :]
            + rng.standard_normal((C, n_doy, 1)))


@pytest.mark.parametrize("P,D,kind", [(1, 1, "readme"), (10, 6, "readme"), (32, 32, "random"), (10, 6, "random"), (1, 32, "random"),
                                      (32, 1, "readme")])
def test_definitions_and_percentiles(core, P, D, kind):
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(P * 100 + D)
    ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    C = 77                                                          # not a multiple of 32; both hemispheres in every warp
    x = _field(rng, ax, C)
    thr = _thr(rng, C, 365, P)
    if kind == "readme":
        defs = (workloads.README_DEFS * 6)[:D]
    else:
        defs = np.stack([rng.integers(0, 8, D), rng.integers(0, 4, D), rng.integers(0, 4, D)], axis=1).tolist()
    st = tb.hemisphere_ranges(ax)
    check(core, x, thr, tb.doy_map(ax.dayofyr), defs, st.north, st.south, (np.arange(C) % 3 == 1).astype(np.uint8))


def test_nan_and_infinite_inputs(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(8)
    ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "standard")
    C = 45
    x = _field(rng, ax, C)
    T = len(ax)
    x[rng.integers(0, T, 80), rng.integers(0, C, 80)] = np.nan
    x[rng.integers(0, T, 20), rng.integers(0, C, 20)] = np.inf
    x[rng.integers(0, T, 20), rng.integers(0, C, 20)] = -np.inf
    x[:, 3] = np.nan
    x[100:200, 4] = np.inf                                          # a season-long run of +inf
    thr = _thr(rng, C, 366, 4)                                      # n_doy = 366
    thr[rng.integers(0, C, 60), rng.integers(0, 366, 60), rng.integers(0, 4, 60)] = np.nan
    thr[5] = np.nan
    thr[6] = -np.inf
    st = tb.hemisphere_ranges(ax)
    heat, _ = check(core, x, thr, tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [1, 0, 2]], st.north, st.south,
                    (np.arange(C) % 2).astype(np.uint8))
    h = heat.cpu().numpy()
    assert (h[..., 3] == 0).all() and (h[..., 5] == 0).all() and np.isinf(h[..., 6]).all()
    assert np.isinf(h[:, :, :, 0, 4]).all()


@pytest.mark.parametrize("units", ["degK", "degF"])
def test_input_units(core, units):
    from hdp_b200 import _tables as tb, measure as hm, xr
    rng = np.random.default_rng(77)
    ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "noleap")
    C = 71
    cel = _field(rng, ax, C)
    raw = ((cel + 273.15) if units == "degK" else (cel * 1.8 + 32)).astype(np.float32)
    conv = hm.kelvin_to_celsius if units == "degK" else hm.fahrenheit_to_celsius
    x_c = xr.values_of(conv(xr.DataArray(raw, dims=["time", "cell"], coords={}, name="t", attrs={"units": units})))
    thr = _thr(rng, C, 365, 3)
    st = tb.hemisphere_ranges(ax)
    check(core, raw, thr, tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [4, 1, 1]], st.north, st.south,
          (np.arange(C) % 2).astype(np.uint8), x_celsius=x_c, units=units)


def test_time_contiguous_layout_and_single_doy(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(3)
    ax = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "noleap")
    C = 50
    x = _field(rng, ax, C)
    st = tb.hemisphere_ranges(ax)
    defs = [[3, 0, 0], [3, 1, 1]]
    south = (np.arange(C) % 2).astype(np.uint8)
    thr = _thr(rng, C, 365, 3)
    check(core, x, thr, tb.doy_map(ax.dayofyr), defs, st.north, st.south, south, x_dev=dev(x.T.copy()).t())
    zeros = np.zeros(len(ax), np.int64)                             # n_doy = 1: the no_season / fixed_thresholds variants
    thr_ns = core.thresholds_no_season_array(dev(x), np.array([0.5, 0.9, 0.99])).cpu().numpy()
    check(core, x, thr_ns, zeros, defs, st.north, st.south, south)
    check(core, x, core.fixed_thresholds(C, 24.5).cpu().numpy(), zeros, defs, st.north, st.south, south)


def _mask_x(masks, rng):
    """Hot where the mask is set, against a 0.5 threshold, with varied exceedances."""
    return np.where(masks, 0.5 + rng.uniform(0.01, 5.0, masks.shape), rng.uniform(-3.0, 0.5, masks.shape)).astype(np.float32)


def test_long_runs_negative_and_empty_seasons(core):
    rng = np.random.default_rng(12)
    T, C = 2000, 33
    masks = np.ones((T, C), bool)
    masks[700, :] = False
    masks[1500:1503, 1::2] = False
    x = _mask_x(masks, rng)
    thr = np.full((C, 1, 1), 0.5)
    dm = np.zeros(T, np.int64)
    seasons = [[100, 250], [465, 615], [830, 980], [1195, 1345], [1560, 1710]]
    check(core, x, thr, dm, [[3, 0, 0], [3, 1, 1], [5, 2, 0]], seasons, seasons, None)
    north = [[-1900, -1700], [400, 400], [600, 800], [-5, 3000], [2500, 2600]]      # negative, empty, past the end
    south = [[0, 1], [1, 2], [1990, 2000], [50, 50], [-100, -50]]
    check(core, x, thr, dm, [[3, 0, 0], [1, 1, 1]], north, south, (np.arange(C) % 2).astype(np.uint8))
    heat = core.intensity_array(dev(x), dev(thr), dm, [[3, 0, 0]], np.zeros((0, 2)), np.zeros((0, 2)))   # Y = 0
    assert tuple(heat.shape) == (3, 1, 1, 0, C)


def test_overlapping_season_table_is_unsupported(core):
    from hdp_b200 import _lib
    rng = np.random.default_rng(11)
    T, C = 300, 40
    masks = rng.random((T, C)) < 0.45
    x = _mask_x(masks, rng)
    thr = np.full((C, 1, 1), 0.5)
    north = [[0, 5], [0, 10], [20, 30], [42, 50], [100, 100], [-50, -1], [250, 400]]     # the table of test_overlapping_and_odd_seasons
    south = [[10, 60], [60, 61], [61, 200], [150, 260], [0, 300], [299, 300], [5, 5]]
    with pytest.raises(_lib.HdpB200Error) as e:
        core.intensity_array(dev(x), dev(thr), np.zeros(T, np.int64), [[1, 1, 1]], north, south, rng.integers(0, 2, C))
    assert e.value.code == -2 and "overlapping" in str(e.value)
    with pytest.raises(_lib.HdpB200Error) as e:
        core.intensity_host(x, thr, np.zeros(T, np.int64), [[1, 1, 1]], north, south, rng.integers(0, 2, C))
    assert e.value.code == -2


@pytest.mark.parametrize("chunk", [None, "32", "96"])
def test_host_pipeline(core, monkeypatch, chunk):
    # intensity_host against the device call: many chunks, pageable and pinned memory, both host layouts, resident thresholds
    from hdp_b200 import _tables as tb
    if chunk:
        monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", chunk)
    rng = np.random.default_rng(23)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1966-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    wt = tb.window_tables(base_ax.dayofyr, 7)
    C = 299
    xb = _field(rng, base_ax, C, warm=0.0)
    xr_ = _field(rng, run_ax, C)
    q = np.arange(0.9, 1.0, 0.01)
    thr_d = core.thresholds_array(dev(xb), wt, q)
    thr_h = thr_d.cpu().numpy()
    st = tb.hemisphere_ranges(run_ax)
    is_south = (rng.random(C) < 0.5).astype(np.uint8)
    defs = [[3, 0, 0], [3, 1, 1], [4, 0, 0], [4, 1, 1], [5, 0, 0], [5, 1, 1]]
    args = (tb.doy_map(run_ax.dayofyr), defs, st.north, st.south, is_south)
    met_d = torch.empty((4, q.size, len(defs), st.n_years, C), dtype=torch.uint16, device="cuda")
    heat_d = core.intensity_array(dev(xr_), thr_d, *args, metrics_out=met_d).cpu().numpy()
    met_d = met_d.cpu().numpy()
    assert np.array_equal(bits(ref_layout(heat_d)), bits(intensity_oracle.intensity_batch(xr_, thr_h, *args)))
    met_h = np.empty_like(met_d)
    assert np.array_equal(bits(core.intensity_host(xr_, thr_h, *args, metrics_out=met_h)), bits(heat_d))
    assert np.array_equal(met_h, met_d)
    assert np.array_equal(bits(core.intensity_host(np.ascontiguousarray(xr_.T).T, thr_h, *args)), bits(heat_d))
    assert np.array_equal(bits(core.intensity_host(xr_, thr_d, *args)), bits(heat_d))               # device-resident thresholds
    thr_k = core.thresholds_host(xb, wt, q, keep=True)                                                # remembered resident copy
    assert core.resident_thresholds(thr_k) is not None
    assert np.array_equal(bits(core.intensity_host(xr_, thr_k, *args)), bits(heat_d))
    # pinned host buffers
    x_pin = torch.from_numpy(xr_).pin_memory()
    out_pin = torch.empty(heat_d.shape, dtype=torch.float32).pin_memory()
    met_pin = torch.empty(met_d.shape, dtype=torch.int16).pin_memory()
    core.intensity_host(x_pin.numpy(), thr_h, *args, out=out_pin.numpy(), metrics_out=met_pin.numpy().view(np.uint16))
    assert np.array_equal(bits(out_pin.numpy()), bits(heat_d)) and np.array_equal(met_pin.numpy().view(np.uint16), met_d)
    core.host_release()


def test_host_pipeline_pageable_many_ring_blocks(core):
    # pageable arrays large enough that every copy runs through several 32 MB blocks of the staging rings
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(77)
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2007-12-31", "noleap")
    C = 40001
    xr_ = (15 + 10 * np.sin(2 * np.pi * (run_ax.dayofyr[:, None] - 110) / 365) + 2
           + 3 * rng.standard_normal((len(run_ax), C), dtype=np.float32)).astype(np.float32)
    thr = _thr(rng, C, 365, 4)
    st = tb.hemisphere_ranges(run_ax)
    defs = [[3, 0, 0], [3, 1, 1], [4, 1, 1]]
    args = (tb.doy_map(run_ax.dayofyr), defs, st.north, st.south, (rng.random(C) < 0.5).astype(np.uint8))
    met_d = torch.empty((4, 4, 3, st.n_years, C), dtype=torch.uint16, device="cuda")
    heat_d = core.intensity_array(dev(xr_), dev(thr), *args, metrics_out=met_d).cpu().numpy()
    met_h = np.empty((4, 4, 3, st.n_years, C), np.uint16)
    assert np.array_equal(bits(core.intensity_host(xr_, thr, *args, metrics_out=met_h)), bits(heat_d))
    assert np.array_equal(met_h, met_d.cpu().numpy())
    sel = np.arange(0, C, 997)
    want = intensity_oracle.intensity_batch(np.ascontiguousarray(xr_[:, sel]), thr[sel], args[0], defs, st.north, st.south, args[4][sel])
    assert np.array_equal(bits(ref_layout(heat_d)[:, :, sel]), bits(want))
    core.host_release()


def _no_stamps(attrs):
    """attrs with the minute time stamps of the history entries removed."""
    return {k: re.sub(r"\(\d{4}-\d\d-\d\d \d\d:\d\d\) ", "", v) if k == "history" else v for k, v in attrs.items()}


def test_group_metrics_opt_in(core):
    from hdp_b200 import _tables as tb, measure, metric, threshold, utils, xr
    grid = (2, 3)
    base = utils.generate_test_control_dataarray(grid_shape=grid, add_noise=True)
    test = utils.generate_test_warming_dataarray(grid_shape=grid, add_noise=True)
    rh = utils.generate_test_rh_dataarray(grid_shape=grid)
    base_measures = measure.format_standard_measures([base], rh=rh)
    test_measures = measure.format_standard_measures([test], rh=rh)
    percentiles = np.arange(0.9, 1.0, 0.01)
    defs = [[3, 0, 0], [3, 1, 1], [4, 0, 0], [4, 1, 1], [5, 0, 0], [5, 1, 1]]
    thresholds = threshold.compute_thresholds(base_measures, percentiles)
    plain = metric.compute_group_metrics(test_measures, thresholds, defs)
    plain_default = metric.compute_group_metrics(test_measures, thresholds, defs, intensity=False)
    full = metric.compute_group_metrics(test_measures, thresholds, defs, intensity=True)
    assert list(plain_default.keys()) == list(plain.keys()) and len(plain.keys()) == 8
    assert sorted(full.keys()) == sorted(list(plain.keys()) + [f"{m}.{m}_threshold.{n}" for m in test_measures.keys()
                                                               for n in ("HWC", "HWI", "HWP")])
    for name in plain.keys():
        assert np.array_equal(xr.values_of(full[name]), xr.values_of(plain[name]))
        assert xr.values_of(full[name]).dtype == np.int64 and _no_stamps(full[name].attrs) == _no_stamps(plain[name].attrs)
    long_names = {"HWC": "Heatwave Cumulative Intensity", "HWI": "Heatwave Mean Intensity", "HWP": "Heatwave Peak Intensity"}
    for mname in test_measures.keys():
        hwf = full[f"{mname}.{mname}_threshold.HWF"]
        r = xr.values_of(test_measures[mname]).reshape(6, -1).T
        t_axis = utils.time_axis_of(test_measures[mname])
        st = tb.hemisphere_ranges(t_axis)
        south = tb.is_south(np.tile(np.linspace(-90, 90, 3), 2))
        thr = xr.values_of(thresholds[f"{mname}_threshold"]).reshape(6, 365, 10)
        want = intensity_oracle.intensity_batch(np.ascontiguousarray(r), thr, tb.doy_map(t_axis.dayofyr), defs, st.north, st.south, south)
        for i, short in enumerate(("HWC", "HWI", "HWP")):
            da = full[f"{mname}.{mname}_threshold.{short}"]
            assert tuple(da.dims) == tuple(hwf.dims) and da.shape == hwf.shape and da.dtype == np.float32
            for d in da.dims:
                assert np.array_equal(np.asarray(xr.coord_values(da, d)), np.asarray(xr.coord_values(hwf, d)))
            assert da.attrs["units"] == test_measures[mname].attrs["units"]
            assert da.attrs["long_name"] == long_names[short] and "exceedance" in da.attrs["description"]
            assert _no_stamps(da.attrs)["history"] == _no_stamps(hwf.attrs)["history"]
            assert np.array_equal(bits(xr.values_of(da).reshape(10, 6, 6, -1)), bits(want[:, :, :, i, :]))


def test_cmip6_1deg_full_size(core):
    # one full-size measure (64 800 cells x 31 390 days) through the host pipeline with both outputs; a cell sample against
    # the oracle, the integer metrics against metrics_host
    from hdp_b200 import _tables as tb, synth, workloads
    wl = workloads.get("cmip6_1deg")
    lat, _ = synth.grid_latitudes(wl.n_lat, wl.n_lon)
    base = synth.gridded_field(lat, wl.base_axis().dayofyr, seed=4321, device="cuda")
    thr = core.thresholds_array(base, wl.window_tables(), wl.percentiles)
    del base
    warm = synth.gridded_field(lat, wl.run_axis().dayofyr, seed=4322, trend=4.0, device="cuda").cpu().numpy()
    st, dm = wl.seasons(), tb.doy_map(wl.run_axis().dayofyr)
    south = (lat < 0).astype(np.uint8)
    args = (dm, wl.defs, st.north, st.south, south)
    P, D, Y, C = len(wl.percentiles), len(wl.defs), st.n_years, lat.size
    met = np.empty((4, P, D, Y, C), np.uint16)
    heat = core.intensity_host(warm, thr, *args, metrics_out=met)
    assert np.array_equal(met, core.metrics_host(warm, thr, *args))
    assert np.isfinite(heat).all() and (heat >= 0).all()
    assert np.array_equal(heat[0] > 0, met[0] > 0)
    sel = np.unique(np.concatenate([[0, C - 1], np.random.default_rng(0).integers(0, C, 64)]))
    want = intensity_oracle.intensity_batch(np.ascontiguousarray(warm[:, sel]), thr[torch.as_tensor(sel, device="cuda")].cpu().numpy(),
                                  dm, wl.defs, st.north, st.south, south[sel])
    assert np.array_equal(bits(ref_layout(heat)[:, :, sel]), bits(want))
    core.host_release()
