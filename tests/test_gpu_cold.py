"""GPU parity of the cold-spell pass (HDP_B200_COLD: k_hot_words' cold instances, then the unchanged k_scan and k_intensity with the
deficit) bit for bit: against the oracle on negated inputs - cold(x, thr) is warm(-x, -thr) exactly - and against the library's own
heatwave call on (-x, -thr); the f32 rounding boundary of the threshold tile; units, sample layouts, thresholds without a day of
year, the host pipeline and the metric layer (compute_individual_metrics / compute_group_metrics with cold=True)."""
import re

import numpy as np
import pytest

import oracle
from intensity_oracle import intensity_batch
from test_gpu_instances import view_of
from test_instance_table import metrics_choice

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


@pytest.fixture
def lib(core):
    from hdp_b200 import _lib
    L = _lib.lib()
    yield L
    L.hdp_b200_metrics_run_filter(1)


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def ref_layout(out_u16):
    """uint16 [4, P, D, Y, C] -> the oracle's int64 [P, D, C, 4, Y]."""
    return np.asarray(out_u16.cpu().numpy() if isinstance(out_u16, torch.Tensor) else out_u16).astype(np.int64).transpose(1, 2, 4, 0, 3)


def heat_layout(out_f32):
    """float32 [3, P, D, Y, C] -> the oracle's [P, D, C, 3, Y]."""
    return np.asarray(out_f32.cpu().numpy() if isinstance(out_f32, torch.Tensor) else out_f32).transpose(1, 2, 4, 0, 3)


def same_f32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def cold_check(core, x, thr, dm, defs, north, south, is_south, x_dev=None, units=None, x_celsius=None, intensity=True):
    """metrics_array(cold=True) against the oracle on (-x, -thr) and against the heatwave call on (-x, -thr); with ``intensity``
    also intensity_array(cold=True, metrics_out=...).  x_celsius: what the kernels convert x to (``units``).  Returns both."""
    nx = -np.ascontiguousarray(x if x_celsius is None else x_celsius, np.float32)
    nt = -np.asarray(thr, np.float64)
    x_dev = dev(x) if x_dev is None else x_dev
    thd = dev(thr)
    args = (dm, defs, north, south, is_south)
    met = core.metrics_array(x_dev, thd, *args, units=units, cold=True)
    assert np.array_equal(ref_layout(met), oracle.metrics_batch(nx, nt, *args))
    assert torch.equal(met, core.metrics_array(dev(nx), dev(nt), *args))
    heat = None
    if intensity:
        met2 = torch.zeros_like(met)
        heat = core.intensity_array(x_dev, thd, *args, metrics_out=met2, units=units, cold=True)
        assert torch.equal(met2, met)
        assert same_f32(heat_layout(heat), intensity_batch(nx, nt, *args))
        assert torch.equal(heat, core.intensity_array(dev(nx), dev(nt), *args))
        h, f = heat.cpu().numpy(), met.cpu().numpy()[0]
        assert np.array_equal(h[0] > 0, f > 0) and np.array_equal(h[2] > 0, f > 0)
    return met, heat


def _field(rng, ax, C, shift=-2.0):
    z = rng.standard_normal((len(ax), C))
    for t in range(1, len(ax)):
        z[t] = 0.6 * z[t - 1] + 0.8 * z[t]
    return (15 + 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365) + 3 * z + shift).astype(np.float32)


def _thr_low(rng, C, n_doy, P):
    """Low-percentile-like thresholds: the seasonal cycle a few degrees down."""
    return (15 + 10 * np.sin(2 * np.pi * (np.arange(n_doy)[None, :, None] - 110) / 365) - np.linspace(1, 6, P)[None, None, :]
            + rng.standard_normal((C, n_doy, 1)))


def _cold_seasons(ax):
    """Each hemisphere's cold season: the other hemisphere's heatwave season."""
    from hdp_b200 import _tables as tb
    st = tb.hemisphere_ranges(ax)
    return st.south, st.north


# ------------------------------------------------------------------------------------------------ definitions, percentiles
@pytest.mark.parametrize("P,D,kind", [(1, 1, "readme"), (10, 6, "readme"), (32, 32, "random"), (10, 6, "random"), (1, 32, "random"),
                                      (32, 1, "readme")])
@pytest.mark.parametrize("run_filter", [1, 0])
def test_definitions_and_percentiles(core, lib, P, D, kind, run_filter):
    from hdp_b200 import _tables as tb, workloads
    lib.hdp_b200_metrics_run_filter(run_filter)
    rng = np.random.default_rng(P * 100 + D)
    ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    C = 77                                                          # not a multiple of 32; both hemispheres in every warp
    x = _field(rng, ax, C)
    thr = _thr_low(rng, C, 365, P)
    if kind == "readme":
        defs = (workloads.README_DEFS * 6)[:D]
    else:
        defs = np.stack([rng.integers(0, 8, D), rng.integers(0, 4, D), rng.integers(0, 4, D)], axis=1).tolist()
    north, south = _cold_seasons(ax)
    met, _ = cold_check(core, x, thr, tb.doy_map(ax.dayofyr), defs, north, south, (np.arange(C) % 3 == 1).astype(np.uint8))
    assert met.cpu().numpy()[0].max() > 0                           # there are cold spells


def _ar1_cold(rng, T, C, P):
    """AR(1) samples with per (cell, percentile) thresholds at mixed cold-day densities; cell 0 is one cold run over the whole
    series, cell 1 never cold."""
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
    x = z.astype(np.float32)
    dens = rng.uniform(0.02, 0.9, (C, P))
    q = np.stack([[np.quantile(x[:, c], dens[c, p]) for p in range(P)] for c in range(C)]).astype(np.float64)
    x[:, 0] = -10.0
    x[:, 1] = 10.0
    return x, np.repeat(q[:, None, :], 365, axis=1)


@pytest.mark.parametrize("run_filter", [1, 0])
def test_long_and_overlapping_seasons(core, lib, run_filter):
    # seasons over 255 days (16-bit accumulator lanes), and overlapping tables (several k_scan passes; metrics only)
    from hdp_b200 import _tables as tb
    lib.hdp_b200_metrics_run_filter(run_filter)
    rng = np.random.default_rng(255)
    T, C, P = 1500, 97, 3
    x, thr = _ar1_cold(rng, T, C, P)
    dm = tb.doy_map(tb.TimeAxis.daily((2001, 1, 1), T, "noleap").dayofyr)
    is_south = rng.integers(0, 2, C).astype(np.uint8)
    defs = [[3, 0, 0], [3, 1, 1], [1, 2, 0], [5, 1, 2], [2, 0, 1]]
    north, south = [[0, 300], [300, 700], [900, 1400]], [[50, 356], [400, 800], [1000, 1500]]
    assert metrics_choice(defs, north, south, T)[1][0] == 16
    cold_check(core, x, thr, dm, defs, north, south, is_south)
    north, south = [[0, 300], [100, 500], [450, 900], [-50, -1]], [[10, 270], [270, 600], [200, 300], [5, 5]]
    rc, info = metrics_choice(defs, north, south, T)
    assert rc == 0 and info[6] > 1
    cold_check(core, x, thr, dm, defs, north, south, is_south, intensity=False)


# ------------------------------------------------------------------------------------------------ the f32 rounding boundary
@pytest.mark.parametrize("P", [3, 17])
def test_rounding_boundary(core, P):
    # thresholds just above, at and just below the samples (in float64), inside their float32 ulp, +-inf, NaN, beyond +-FLT_MAX;
    # samples with NaN, +-inf, +-FLT_MAX, signed zeros and subnormals.  Definition [1, 0, 0] and one season over the whole
    # series: CSF is the number of days with (double)x < thr, HWF the number with (double)x > thr.
    rng = np.random.default_rng(P)
    T, C = 365, 64
    fmax = float(np.finfo(np.float32).max)
    x = (rng.standard_normal((T, C)) * 10).astype(np.float32)
    specials = np.array([np.nan, np.inf, -np.inf, fmax, -fmax, 0.0, -0.0, 1e-45, -1e-45, 1.17549435e-38], np.float32)
    mask = rng.random((T, C)) < 0.15
    x[mask] = rng.choice(specials, int(mask.sum()))
    xd = np.repeat(x.T.astype(np.float64)[:, :, None], P, axis=2)                  # [C, T, P]: the sample of day t
    with np.errstate(invalid="ignore", over="ignore"):
        ulp = np.spacing(np.abs(x.T)).astype(np.float64)[:, :, None]
        cand = [xd, np.nextafter(xd, np.inf), np.nextafter(xd, -np.inf), xd + rng.uniform(-1, 1, xd.shape) * ulp,
                np.full_like(xd, np.inf), np.full_like(xd, -np.inf), np.full_like(xd, np.nan),
                np.full_like(xd, 1e39), np.full_like(xd, -1e39), np.full_like(xd, np.nextafter(fmax, np.inf)),
                np.full_like(xd, -np.nextafter(fmax, np.inf)), np.full_like(xd, fmax), np.full_like(xd, -fmax),
                rng.normal(0, 10, xd.shape)]
    kind = rng.integers(0, len(cand), xd.shape)
    kind[:, :, 0] = rng.choice([0, 1, 2], (C, T))                   # percentile 0: the three one-ulp cases only
    thr = np.choose(kind, cand)
    dm = np.arange(T)
    seasons = [[0, T]]
    args = (dm, [[1, 0, 0]], seasons, seasons, None)
    cold = core.metrics_array(dev(x), dev(thr), *args, cold=True).cpu().numpy()
    warm = core.metrics_array(dev(x), dev(thr), *args).cpu().numpy()
    with np.errstate(invalid="ignore"):
        assert np.array_equal(cold[0, :, 0, 0, :], (xd < thr).sum(axis=1).T)
        assert np.array_equal(warm[0, :, 0, 0, :], (xd > thr).sum(axis=1).T)
    assert np.array_equal(ref_layout(cold), oracle.metrics_batch(-x, -thr, *args))
    heat = core.intensity_array(dev(x), dev(thr), *args, cold=True)
    assert same_f32(heat_layout(heat), intensity_batch(-x, -thr, *args))


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
    x[:, 4] = -np.inf                                               # every day a -inf sample: every season-long spell is inf
    thr = _thr_low(rng, C, 366, 4)                                  # n_doy = 366
    thr[rng.integers(0, C, 60), rng.integers(0, 366, 60), rng.integers(0, 4, 60)] = np.nan
    thr[5] = np.nan
    thr[6] = np.inf                                                 # every finite sample is below +inf
    thr[7] = -np.inf                                                # nothing is below -inf
    north, south = _cold_seasons(ax)
    met, heat = cold_check(core, x, thr, tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [1, 0, 2]], north, south,
                           (np.arange(C) % 2).astype(np.uint8))
    h, f = heat.cpu().numpy(), met.cpu().numpy()
    assert (f[..., 3] == 0).all() and (f[..., 5] == 0).all() and (f[..., 7] == 0).all() and (h[..., 7] == 0).all()
    for c in (4, 6):                                                # a -inf sample or a +inf threshold: an infinite deficit
        spell = f[0, ..., c] > 0
        assert spell.any() and np.isinf(h[:, spell, c]).all()


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
    thr = _thr_low(rng, C, 365, 3)
    north, south = _cold_seasons(ax)
    cold_check(core, raw, thr, tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [4, 1, 1]], north, south,
               (np.arange(C) % 2).astype(np.uint8), units=units, x_celsius=x_c)


# ------------------------------------------------------------------------------------------------ sample layouts
@pytest.mark.parametrize("kind", ["cell_offset", "time_range", "strided", "single_cell"])
def test_sample_layouts(core, kind):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(78)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C = 1 if kind == "single_cell" else 45
    x = _field(rng, ax, C)
    thr = _thr_low(rng, C, 365, 2)
    north, south = _cold_seasons(ax)
    is_south = (np.arange(C) % 2).astype(np.uint8)
    dm = tb.doy_map(ax.dayofyr)
    defs = [[3, 0, 0], [3, 1, 1], [5, 2, 1]]
    v = view_of("cell_offset" if kind == "single_cell" else kind, x)
    met, heat = cold_check(core, x, thr, dm, defs, north, south, is_south, x_dev=v)
    assert torch.equal(met, core.metrics_array(v.contiguous(), dev(thr), dm, defs, north, south, is_south, cold=True))
    if kind == "single_cell":                                       # and a single day: one-day seasons of a one-day run
        day = v[40:41]
        one = (dm[40:41], defs, [[0, 1]], [[0, 1]], is_south)
        assert np.array_equal(ref_layout(core.metrics_array(day, dev(thr), *one, cold=True)),
                              oracle.metrics_batch(-x[40:41], -thr, *one))


# ------------------------------------------------------------------------------------------------ thresholds without a day of year
def test_doy_free_thresholds_over_a_long_run(core):
    # the no-season and fixed-value variants at low percentiles over a CMIP-length run, through all four entry points
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(31390)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1990-12-31", "noleap")
    run_ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C = 97
    season = lambda ax, shift: shift + 15 + 8 * np.sin(2 * np.pi * ax.dayofyr[:, None] / 365)     # noqa: E731
    xb = (season(base_ax, 0) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (season(run_ax, -1) + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    north, south = _cold_seasons(run_ax)
    zeros = np.zeros(len(run_ax), np.int64)
    is_south = (np.arange(C) % 2).astype(np.uint8)
    defs = workloads.README_DEFS
    args = (zeros, defs, north, south, is_south)
    thr_ns = core.thresholds_no_season_array(dev(xb), np.array([0.01, 0.05, 0.1]))
    for thr in (thr_ns, core.fixed_thresholds(C, 7.5)):
        th = thr.cpu().numpy()
        want, want_heat = oracle.metrics_batch(-xr, -th, *args), intensity_batch(-xr, -th, *args)
        assert np.array_equal(ref_layout(core.metrics_array(dev(xr), thr, *args, cold=True)), want)
        met = torch.zeros((4, th.shape[2], len(defs), len(north), C), dtype=torch.uint16, device="cuda")
        assert same_f32(heat_layout(core.intensity_array(dev(xr), thr, *args, metrics_out=met, cold=True)), want_heat)
        assert np.array_equal(ref_layout(met), want)
        assert np.array_equal(ref_layout(core.metrics_host(xr, th, *args, cold=True)), want)
        met_h = np.zeros((4, th.shape[2], len(defs), len(north), C), np.uint16)
        assert same_f32(heat_layout(core.intensity_host(xr, th, *args, metrics_out=met_h, cold=True)), want_heat)
        assert np.array_equal(ref_layout(met_h), want)
        assert want[:, :, :, 0].max() > 0
    core.host_release()


# ------------------------------------------------------------------------------------------------ host pipeline
@pytest.mark.parametrize("chunk", [None, "32"])
def test_host_pipeline(core, monkeypatch, chunk):
    from hdp_b200 import _tables as tb
    if chunk:
        monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", chunk)
    rng = np.random.default_rng(23)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1966-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    wt = tb.window_tables(base_ax.dayofyr, 7)
    C = 299
    xb = _field(rng, base_ax, C, shift=0.0)
    xr_ = _field(rng, run_ax, C)
    q = np.arange(0.01, 0.105, 0.01)
    thr_d = core.thresholds_array(dev(xb), wt, q)
    thr_h = thr_d.cpu().numpy()
    north, south = _cold_seasons(run_ax)
    defs = [[3, 0, 0], [3, 1, 1], [4, 0, 0], [4, 1, 1], [5, 0, 0], [5, 1, 1]]
    args = (tb.doy_map(run_ax.dayofyr), defs, north, south, (rng.random(C) < 0.5).astype(np.uint8))
    met_d, heat_d = cold_check(core, xr_, thr_h, *args)
    met_d, heat_d = met_d.cpu().numpy(), heat_d.cpu().numpy()
    assert np.array_equal(core.metrics_host(xr_, thr_h, *args, cold=True), met_d)
    assert np.array_equal(core.metrics_host(xr_, thr_d, *args, cold=True), met_d)                    # device-resident thresholds
    met_h = np.empty_like(met_d)
    assert same_f32(core.intensity_host(xr_, thr_h, *args, metrics_out=met_h, cold=True), heat_d)
    assert np.array_equal(met_h, met_d)
    assert same_f32(core.intensity_host(np.ascontiguousarray(xr_.T).T, thr_h, *args, cold=True), heat_d)
    assert same_f32(core.intensity_host(xr_, thr_d, *args, cold=True), heat_d)
    thr_k = core.thresholds_host(xb, wt, q, keep=True)                                                # remembered resident copy
    assert core.resident_thresholds(thr_k) is not None
    assert same_f32(core.intensity_host(xr_, thr_k, *args, cold=True), heat_d)
    assert np.array_equal(core.metrics_host(xr_, thr_k, *args, cold=True), met_d)
    assert not np.array_equal(core.metrics_host(xr_, thr_h, *args), met_d)                          # the heatwave pass differs
    core.host_release()


# ------------------------------------------------------------------------------------------------ the metric layer
def _no_stamps(attrs):
    return {k: re.sub(r"\(\d{4}-\d\d-\d\d \d\d:\d\d\) ", "", v) if k == "history" else v for k, v in attrs.items()}


@pytest.mark.parametrize("intensity", [False, True])
def test_individual_and_group_metrics(core, intensity):
    from hdp_b200 import _tables as tb, measure, metric, threshold, utils, xr
    grid = (2, 3)
    test = utils.generate_test_warming_dataarray(grid_shape=grid, add_noise=True)
    rh = utils.generate_test_rh_dataarray(grid_shape=grid)
    test_measures = measure.format_standard_measures([test], rh=rh)
    percentiles = np.arange(0.01, 0.105, 0.01)
    defs = [[3, 0, 0], [3, 1, 1], [4, 0, 0], [4, 1, 1], [5, 0, 0], [5, 1, 1]]
    thresholds = threshold.compute_thresholds(test_measures, percentiles)       # (the warmed run has no days below its baseline's)
    warm = metric.compute_group_metrics(test_measures, thresholds, defs, intensity=intensity)
    cold = metric.compute_group_metrics(test_measures, thresholds, defs, intensity=intensity, cold=True)
    short = ("CSF", "CSN", "CSD", "CSA") + (("CSC", "CSI", "CSP") if intensity else ())
    assert sorted(cold.keys()) == sorted(f"{m}.{m}_threshold.{n}" for m in test_measures.keys() for n in short)
    for mname in test_measures.keys():
        tname = f"{mname}_threshold"
        ds = metric.compute_individual_metrics(test_measures[mname], thresholds[tname], defs, intensity=intensity, cold=True)
        assert sorted(ds.keys()) == sorted(short)
        r = xr.values_of(test_measures[mname]).reshape(6, -1).T
        t_axis = utils.time_axis_of(test_measures[mname])
        st = tb.hemisphere_ranges(t_axis)
        south = tb.is_south(np.tile(np.linspace(-90, 90, 3), 2))
        thr = np.ascontiguousarray(xr.values_of(thresholds[tname]).reshape(6, 365, 10))
        args = (tb.doy_map(t_axis.dayofyr), defs, st.south, st.north, south)                      # the swapped tables
        met = core.metrics_host(r, thr, *args, cold=True)
        assert np.array_equal(ref_layout(met), oracle.metrics_batch(-np.ascontiguousarray(r), -thr, *args))
        heat = core.intensity_host(r, thr, *args, cold=True) if intensity else None
        for i, n in enumerate(short):
            da, hw = cold[f"{mname}.{tname}.{n}"], warm[f"{mname}.{tname}.{'HWF' if i < 4 else 'HWC'}"]
            assert tuple(da.dims) == tuple(hw.dims) and da.shape == hw.shape and xr.values_of(da).dtype == xr.values_of(hw).dtype
            for d in da.dims:
                assert repr(xr.coord_values(da, d)) == repr(xr.coord_values(hw, d))
            assert _no_stamps(da.attrs)["history"] == _no_stamps(hw.attrs)["history"]
            attrs = {**metric.COLD_METRIC_ATTRS, **metric.COLD_INTENSITY_ATTRS}[n]
            assert all(da.attrs[k] == v for k, v in attrs.items())
            want = met[i] if i < 4 else heat[i - 4]                                                  # [P, D, Y, C]
            got = xr.values_of(da).reshape(10, 6, 6, -1)                                             # [P, D, C, Y]
            if i < 4:
                assert np.array_equal(got, want.transpose(0, 1, 3, 2).astype(np.int64))
            else:
                assert da.attrs["units"] == test_measures[mname].attrs["units"]
                assert same_f32(got, want.transpose(0, 1, 3, 2))
            assert np.array_equal(xr.values_of(da), xr.values_of(ds[n]))
        assert met[0].max() > 0
