"""GPU parity of the compound pass (hdp_b200_compound: k_hot_pair, then the unchanged k_scan and k_intensity on its words) bit for bit:
against the masked-input oracle (tests/test_compound_host.py: compound metrics at percentile p = single-measure metrics of
where(M_p, x_a, NaN)), and against the library's own single-measure calls (identities); every k_hot_pair instance, the f32 rounding
boundary of each measure's tile, layouts, thresholds without a day of year, the host pipeline and compute_compound_metrics."""
import numpy as np
import pytest

from test_compound_host import compound_mask, compound_oracle
from test_gpu_instances import view_of

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


def host(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def same_f32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def check(core, xa, ta, xb, tb, dm, defs, north, south, is_south, xa_dev=None, xb_dev=None, units=None, xa_c=None, xb_c=None, cold=False):
    """compound_metrics_array and compound_intensity_array (with metrics_out) against the masked oracle; xa_c / xb_c: the samples in
    Celsius when ``units`` converts them.  Returns (metrics, intensity) as host arrays."""
    xa_dev = dev(xa) if xa_dev is None else xa_dev
    xb_dev = dev(xb) if xb_dev is None else xb_dev
    args = (dm, defs, north, south, is_south)
    met = core.compound_metrics_array(xa_dev, dev(ta), xb_dev, dev(tb), *args, units=units, cold=cold)
    met2 = torch.zeros_like(met)
    heat = core.compound_intensity_array(xa_dev, dev(ta), xb_dev, dev(tb), *args, metrics_out=met2, units=units, cold=cold)
    assert torch.equal(met, met2)
    want, want_h = compound_oracle(xa if xa_c is None else xa_c, ta, xb if xb_c is None else xb_c, tb, *args, cold=cold)
    m, h = host(met), host(heat)
    assert np.array_equal(m.astype(np.int64).transpose(1, 2, 4, 0, 3), want)
    assert same_f32(h.transpose(0, 2, 3, 5, 1, 4), want_h)
    return m, h


def _pair_fields(rng, ax, C, rho=0.7):
    """tmax-like and tmin-like fields whose noise is correlated (rho)."""
    T = len(ax)
    z = rng.standard_normal((T, C))
    w = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.6 * z[t - 1] + 0.8 * z[t]
        w[t] = 0.6 * w[t - 1] + 0.8 * w[t]
    cyc = 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)
    xa = (25 + cyc + 3 * z).astype(np.float32)
    xb = (14 + cyc + 3 * (rho * z + np.sqrt(1 - rho * rho) * w)).astype(np.float32)
    return xa, xb


def _thr(rng, C, n_doy, P, base, cold=False):
    cyc = 10 * np.sin(2 * np.pi * (np.arange(n_doy)[None, :, None] - 110) / 365)
    off = np.linspace(1, 4, P)[None, None, :]
    return base + cyc + (-off if cold else off) + 0.5 * rng.standard_normal((C, n_doy, 1))


def _seasons(ax, cold=False):
    from hdp_b200 import _tables as tb
    st = tb.hemisphere_ranges(ax)
    return (st.south, st.north) if cold else (st.north, st.south)


# ------------------------------------------------------------------------------------------------ every k_hot_pair instance
@pytest.mark.parametrize("cold", [False, True])
@pytest.mark.parametrize("units", [None, "degK", "degF"])
@pytest.mark.parametrize("P", [4, 8, 10, 16, 20, 32])
def test_every_instance(core, P, units, cold):
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(P * 7 + (units is not None) * 3 + cold)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C = 45
    xa, xb = _pair_fields(rng, ax, C)
    ta, tb_ = _thr(rng, C, 365, P, 25, cold), _thr(rng, C, 365, P, 14, cold)
    ra, rb = xa, xb
    if units == "degK":
        ra, rb = (xa + np.float32(273.15)).astype(np.float32), (xb + np.float32(273.15)).astype(np.float32)
    elif units == "degF":
        ra, rb = (xa * np.float32(1.8) + np.float32(32)).astype(np.float32), (xb * np.float32(1.8) + np.float32(32)).astype(np.float32)
    to_c = {None: lambda v: v, "degK": lambda v: (v - np.float32(273.15)).astype(np.float32),
            "degF": lambda v: ((v - np.float32(32)) / np.float32(1.8)).astype(np.float32)}[units]
    north, south = _seasons(ax, cold)
    m, _ = check(core, ra, ta, rb, tb_, tb.doy_map(ax.dayofyr), workloads.README_DEFS, north, south, (np.arange(C) % 3 == 1).astype(np.uint8),
                 units=units, xa_c=to_c(ra), xb_c=to_c(rb), cold=cold)
    assert m[0].max() > 0


# ------------------------------------------------------------------------------------------------ definitions, run filter
@pytest.mark.parametrize("D,kind", [(1, "readme"), (6, "readme"), (32, "random"), (13, "random")])
@pytest.mark.parametrize("run_filter", [1, 0])
def test_definitions(core, lib, D, kind, run_filter):
    from hdp_b200 import _tables as tb, workloads
    lib.hdp_b200_metrics_run_filter(run_filter)
    rng = np.random.default_rng(D * 11 + run_filter)
    ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    C = 77                                                          # not a multiple of 32; both hemispheres in every warp
    xa, xb = _pair_fields(rng, ax, C)
    P = 3
    ta, tb_ = _thr(rng, C, 365, P, 25), _thr(rng, C, 365, P, 14)
    defs = (workloads.README_DEFS * 6)[:D] if kind == "readme" else \
        np.stack([rng.integers(0, 8, D), rng.integers(0, 4, D), rng.integers(0, 4, D)], axis=1).tolist()
    north, south = _seasons(ax)
    m, _ = check(core, xa, ta, xb, tb_, tb.doy_map(ax.dayofyr), defs, north, south, (np.arange(C) % 3 == 1).astype(np.uint8))
    assert m[0].max() > 0


# ------------------------------------------------------------------------------------------------ identities
def test_identities(core):
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(5)
    ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "standard")
    C = 70
    xa, xb = _pair_fields(rng, ax, C)
    ta, tb_ = _thr(rng, C, 366, 5, 25), _thr(rng, C, 366, 5, 14)
    dm = tb.doy_map(ax.dayofyr)
    north, south = _seasons(ax)
    args = (dm, workloads.README_DEFS, north, south, (np.arange(C) % 2).astype(np.uint8))
    A, TA, B, TB = dev(xa), dev(ta), dev(xb), dev(tb_)
    # compound(A, A) == single(A)
    single = core.metrics_array(A, TA, *args)
    single_h = core.intensity_array(A, TA, *args)
    assert torch.equal(core.compound_metrics_array(A, TA, A, TA, *args), single)
    h = core.compound_intensity_array(A, TA, A, TA, *args)
    assert torch.equal(h[0], single_h) and torch.equal(h[1], single_h)
    # thr_b = -inf: A alone; thr_b = +inf: nothing
    assert torch.equal(core.compound_metrics_array(A, TA, B, torch.full_like(TB, -np.inf), *args), single)
    assert torch.equal(core.compound_intensity_array(A, TA, B, torch.full_like(TB, -np.inf), *args)[0], single_h)
    assert (core.compound_metrics_array(A, TA, B, torch.full_like(TB, np.inf), *args) == 0).all()
    assert (core.compound_intensity_array(A, TA, B, torch.full_like(TB, np.inf), *args) == 0).all()
    # cold(x_a, t_a, x_b, t_b) == warm(-x_a, -t_a, -x_b, -t_b)
    cold_args = (dm, workloads.README_DEFS, south, north, (np.arange(C) % 2).astype(np.uint8))
    assert torch.equal(core.compound_metrics_array(A, TA, B, TB, *cold_args, cold=True),
                       core.compound_metrics_array(-A, -TA, -B, -TB, *cold_args))
    assert torch.equal(core.compound_intensity_array(A, TA, B, TB, *cold_args, cold=True),
                       core.compound_intensity_array(-A, -TA, -B, -TB, *cold_args))
    # the compound mask is the AND of the two single masks, and the oracle's mask
    mask = core.compound_hot_days_array(A, TA, B, TB, dm)
    assert torch.equal(mask, core.hot_days_array(A, TA, dm) & core.hot_days_array(B, TB, dm))
    assert np.array_equal(host(mask).astype(bool), compound_mask(xa, ta, xb, tb_, dm))
    assert host(mask).any()
    mask_c = core.compound_hot_days_array(A, TA, B, TB, dm, cold=True)
    assert np.array_equal(host(mask_c).astype(bool), compound_mask(xa, ta, xb, tb_, dm, cold=True))
    assert torch.equal(mask_c, core.compound_hot_days_array(-A, -TA, -B, -TB, dm))


# ------------------------------------------------------------------------------------------------ the f32 rounding boundary
def _boundary_thresholds(rng, x, P):
    T, C = x.shape
    fmax = float(np.finfo(np.float32).max)
    xd = np.repeat(x.T.astype(np.float64)[:, :, None], P, axis=2)                  # [C, T, P]
    with np.errstate(invalid="ignore", over="ignore"):
        ulp = np.spacing(np.abs(x.T)).astype(np.float64)[:, :, None]
        cand = [xd, np.nextafter(xd, np.inf), np.nextafter(xd, -np.inf), xd + rng.uniform(-1, 1, xd.shape) * ulp,
                np.full_like(xd, np.inf), np.full_like(xd, -np.inf), np.full_like(xd, np.nan),
                np.full_like(xd, 1e39), np.full_like(xd, -1e39), np.full_like(xd, np.nextafter(fmax, np.inf)),
                np.full_like(xd, -np.nextafter(fmax, np.inf)), np.full_like(xd, fmax), np.full_like(xd, -fmax)]
    kind = rng.integers(0, len(cand), xd.shape)
    kind[:, :, 0] = rng.choice([0, 1, 2], (C, T))                   # percentile 0: the three one-ulp cases only
    return np.choose(kind, cand)


def _boundary_samples(rng, T, C):
    fmax = float(np.finfo(np.float32).max)
    x = (rng.standard_normal((T, C)) * 10).astype(np.float32)
    specials = np.array([np.nan, np.inf, -np.inf, fmax, -fmax, 0.0, -0.0, 1e-45, -1e-45], np.float32)
    mask = rng.random((T, C)) < 0.15
    x[mask] = rng.choice(specials, int(mask.sum()))
    return x


@pytest.mark.parametrize("cold", [False, True])
@pytest.mark.parametrize("side", ["a", "b"])
def test_rounding_boundary_of_each_measure(core, side, cold):
    # one measure at its rounding boundary, the other always (never, for the second check) past its threshold: the compound
    # days are then exactly the boundary measure's days.  Definition [1, 0, 0], one season over the whole series.
    rng = np.random.default_rng(3 + (side == "b") * 2 + cold)
    T, C, P = 365, 64, 3
    x = _boundary_samples(rng, T, C)
    thr = _boundary_thresholds(rng, x, P)
    other = np.zeros((T, C), np.float32)
    open_thr = np.full((C, T, P), np.inf if cold else -np.inf)
    dm = np.arange(T)
    seasons = [[0, T]]
    args = (dm, [[1, 0, 0]], seasons, seasons, None)
    xa, ta, xb, tb_ = (x, thr, other, open_thr) if side == "a" else (other, open_thr, x, thr)
    m, _ = check(core, xa, ta, xb, tb_, *args, cold=cold)
    xd = np.repeat(x.T.astype(np.float64)[:, :, None], P, axis=2)
    with np.errstate(invalid="ignore"):
        assert np.array_equal(m[0, :, 0, 0, :], ((xd < thr) if cold else (xd > thr)).sum(axis=1).T)
    single = core.metrics_array(dev(x), dev(thr), *args, cold=cold)
    assert np.array_equal(m, host(single))
    closed = np.full((C, T, P), -np.inf if cold else np.inf)
    xa, ta, xb, tb_ = (x, thr, other, closed) if side == "a" else (other, closed, x, thr)
    assert (host(core.compound_metrics_array(dev(xa), dev(ta), dev(xb), dev(tb_), *args, cold=cold)) == 0).all()


def test_nan_and_infinite_samples(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(8)
    ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "standard")
    C, T = 45, len(ax)
    xa, xb = _pair_fields(rng, ax, C)
    for x in (xa, xb):
        x[rng.integers(0, T, 80), rng.integers(0, C, 80)] = np.nan
        x[rng.integers(0, T, 20), rng.integers(0, C, 20)] = np.inf
        x[rng.integers(0, T, 20), rng.integers(0, C, 20)] = -np.inf
    xa[:, 3] = np.nan
    xb[:, 4] = np.nan
    xa[:, 5] = np.inf                                               # every day: an infinite exceedance of A
    xb[:, 6] = np.inf
    ta, tb_ = _thr(rng, C, 366, 4, 25), _thr(rng, C, 366, 4, 14)
    ta[rng.integers(0, C, 60), rng.integers(0, 366, 60), rng.integers(0, 4, 60)] = np.nan
    tb_[7] = np.nan
    north, south = _seasons(ax)
    m, h = check(core, xa, ta, xb, tb_, tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [1, 0, 2]], north, south,
                 (np.arange(C) % 2).astype(np.uint8))
    assert (m[..., 3] == 0).all() and (m[..., 4] == 0).all() and (m[..., 7] == 0).all()
    for c, blk in ((5, 0), (6, 1)):
        hw = m[0, ..., c] > 0
        assert hw.any() and np.isinf(h[blk][:, hw, c]).all() and np.isfinite(h[1 - blk][0, hw, c]).all()


# ------------------------------------------------------------------------------------------------ layouts
@pytest.mark.parametrize("ka,kb", [("contig", "time_range"), ("time_range", "contig"), ("strided", "cell_offset"),
                                   ("cell_offset", "strided"), ("time_range", "time_range")])
def test_sample_layouts(core, ka, kb):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(78)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C = 45
    xa, xb = _pair_fields(rng, ax, C)
    ta, tb_ = _thr(rng, C, 365, 2, 25), _thr(rng, C, 365, 2, 14)
    north, south = _seasons(ax)
    va = dev(xa) if ka == "contig" else view_of(ka, xa)
    vb = dev(xb) if kb == "contig" else view_of(kb, xb)
    args = (tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [5, 2, 1]], north, south, (np.arange(C) % 2).astype(np.uint8))
    m, h = check(core, xa, ta, xb, tb_, *args, xa_dev=va, xb_dev=vb)
    assert np.array_equal(host(core.compound_metrics_array(dev(xa), dev(ta), dev(xb), dev(tb_), *args)), m)
    mask = core.compound_hot_days_array(va, dev(ta), vb, dev(tb_), args[0])
    assert np.array_equal(host(mask).astype(bool), compound_mask(xa, ta, xb, tb_, args[0]))


# ------------------------------------------------------------------------------------------------ thresholds without a day of year
def test_doy_free_thresholds_over_a_long_run(core):
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(31390)
    ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C = 37
    xa, xb = _pair_fields(rng, ax, C)
    ta = np.stack([np.full((C, 1), 31.0), np.full((C, 1), 33.0)], axis=2)
    tb_ = np.stack([np.full((C, 1), 19.0), np.full((C, 1), 21.0)], axis=2)
    north, south = _seasons(ax)
    m, _ = check(core, xa, ta, xb, tb_, np.zeros(len(ax), np.int64), workloads.README_DEFS, north, south,
                 (np.arange(C) % 2).astype(np.uint8))
    assert m[0].max() > 0


# ------------------------------------------------------------------------------------------------ host pipeline
@pytest.mark.parametrize("chunk", [None, "32"])
def test_host_pipeline(core, monkeypatch, chunk):
    from hdp_b200 import _tables as tb, workloads
    if chunk:
        monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", chunk)
    rng = np.random.default_rng(23)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1966-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2008-12-31", "noleap")
    wt = tb.window_tables(base_ax.dayofyr, 7)
    C = 299
    ba, bb = _pair_fields(rng, base_ax, C)
    xa, xb = _pair_fields(rng, run_ax, C)
    q = np.arange(0.9, 0.995, 0.01)
    ta_d, tb_d = core.thresholds_array(dev(ba), wt, q), core.thresholds_array(dev(bb), wt, q)
    ta_h, tb_h = ta_d.cpu().numpy(), tb_d.cpu().numpy()
    north, south = _seasons(run_ax)
    args = (tb.doy_map(run_ax.dayofyr), workloads.README_DEFS, north, south, (rng.random(C) < 0.5).astype(np.uint8))
    met_d, heat_d = check(core, xa, ta_h, xb, tb_h, *args)
    assert met_d[0].max() > 0
    tb_k = core.thresholds_host(bb, wt, q, keep=True)                                               # remembered resident copy
    assert core.resident_thresholds(tb_k) is not None
    pinned = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()             # noqa: E731
    for A, TA, B, TB in ((xa, ta_h, xb, tb_h), (xa, ta_d, xb, tb_h), (xa, ta_h, xb, tb_d), (xa, ta_d, xb, tb_k),
                         (pinned(xa), ta_h, np.ascontiguousarray(xb.T).T, tb_h), (np.ascontiguousarray(xa.T).T, ta_h, pinned(xb), tb_k)):
        assert np.array_equal(core.compound_metrics_host(A, TA, B, TB, *args), met_d)
        met_h = np.empty_like(met_d)
        assert same_f32(core.compound_intensity_host(A, TA, B, TB, *args, metrics_out=met_h), heat_d)
        assert np.array_equal(met_h, met_d)
    out = pinned(np.zeros_like(heat_d))
    core.compound_intensity_host(xa, ta_h, xb, tb_h, *args, out=out)
    assert same_f32(out, heat_d)
    core.host_release()


# ------------------------------------------------------------------------------------------------ the metric layer
def test_compute_compound_metrics(core):
    # the temperature and its heat-index measure of format_standard_measures: one grid, one time axis, two measures
    from hdp_b200 import _tables as tb, measure, metric, threshold, utils, xr
    grid = (2, 3)
    test = utils.generate_test_warming_dataarray(grid_shape=grid, add_noise=True)
    rh = utils.generate_test_rh_dataarray(grid_shape=grid)
    measures = measure.format_standard_measures([test], rh=rh)
    na, nb = list(measures.keys())[:2]
    percentiles = np.array([0.9, 0.95])
    thresholds = threshold.compute_thresholds(measures, percentiles)
    defs = [[3, 0, 0], [3, 1, 1], [4, 1, 1]]
    ma, mb = measures[na], measures[nb]
    ta, tb_ = thresholds[f"{na}_threshold"], thresholds[f"{nb}_threshold"]
    t_axis = utils.time_axis_of(ma)
    st = tb.hemisphere_ranges(t_axis)
    south = tb.is_south(np.tile(np.linspace(-90, 90, 3), 2))
    ra, rb = (xr.values_of(m).reshape(6, -1).T for m in (ma, mb))
    tha, thb = (np.ascontiguousarray(xr.values_of(t).reshape(6, 365, 2)) for t in (ta, tb_))
    for cold in (False, True):
        ds = metric.compute_compound_metrics(ma, ta, mb, tb_, defs, intensity=True, cold=cold)
        names = ("CSF", "CSN", "CSD", "CSA", "CSC", "CSI", "CSP") if cold else ("HWF", "HWN", "HWD", "HWA", "HWC", "HWI", "HWP")
        assert sorted(ds.keys()) == sorted(names)
        assert ds.attrs["compound_measures"] == f"{na} & {nb}"
        args = (tb.doy_map(t_axis.dayofyr), defs, *((st.south, st.north) if cold else (st.north, st.south)), south)
        met = np.empty((4, 2, len(defs), st.n_years, 6), np.uint16)
        heat = core.compound_intensity_host(ra, tha, rb, thb, *args, metrics_out=met, cold=cold)
        for i, n in enumerate(names):
            da = ds[n]
            assert da.attrs["long_name"].startswith("Compound ")
            if i < 4:
                assert tuple(da.dims) == ("percentile", "definition", "lon", "lat", "time")
                assert np.array_equal(xr.values_of(da).reshape(2, len(defs), 6, -1), met[i].transpose(0, 1, 3, 2).astype(np.int64))
            else:
                assert tuple(da.dims) == ("measure", "percentile", "definition", "lon", "lat", "time")
                assert list(xr.coord_values(da, "measure")) == [na, nb]
                assert same_f32(xr.values_of(da).reshape(2, 2, len(defs), 6, -1), heat[:, i - 4].transpose(0, 1, 2, 4, 3))
        if not cold:
            assert met[0].max() > 0
    core.host_release()


# ------------------------------------------------------------------------------------------------ one full-size call
def test_cmip6_full_size(core):
    # cmip6_1deg (64 800 cells, 31 390 days, P 10, the README definitions) on the device; a sample of cells against the oracle
    from hdp_b200 import _tables as tb, workloads
    w = workloads.get("cmip6_1deg")
    ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C, T, P = w.cells, len(ax), len(w.percentiles)
    g = torch.Generator(device="cuda").manual_seed(6)
    doy = torch.as_tensor(ax.dayofyr, device="cuda", dtype=torch.float32)[:, None]
    cyc = 10 * torch.sin(2 * np.pi * (doy - 110) / 365)
    z = torch.randn((T, C), device="cuda", generator=g)
    xa = (25 + cyc + 3 * z).float()
    xb = (14 + cyc + 3 * (0.7 * z + 0.714 * torch.randn((T, C), device="cuda", generator=g))).float()
    del z
    off = torch.linspace(3, 6, P, device="cuda", dtype=torch.float64)
    cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
    ta = (25 + cyc_d[None, :, None] + off[None, None, :]).expand(C, 365, P).contiguous()
    tb_ = (14 + cyc_d[None, :, None] + off[None, None, :]).expand(C, 365, P).contiguous()
    north, south = _seasons(ax)
    is_south = (np.arange(C) // w.n_lon) < w.n_lat // 2
    args = (tb.doy_map(ax.dayofyr), w.defs, north, south, is_south.astype(np.uint8))
    met = torch.empty((4, P, len(w.defs), len(north), C), dtype=torch.uint16, device="cuda")
    heat = core.compound_intensity_array(xa, ta, xb, tb_, *args, metrics_out=met)
    torch.cuda.synchronize()
    cells = np.random.default_rng(0).choice(C, 48, replace=False)
    cells.sort()
    sel = torch.as_tensor(cells, device="cuda")
    want, want_h = compound_oracle(host(xa[:, sel]), host(ta[sel]), host(xb[:, sel]), host(tb_[sel]), args[0], args[1], north, south,
                                   args[4][cells])
    met_sel = host(met.view(torch.int16)[..., sel]).view(np.uint16)                              # (no uint16 gather on the device)
    assert np.array_equal(met_sel.astype(np.int64).transpose(1, 2, 4, 0, 3), want)
    assert same_f32(host(heat[..., sel]).transpose(0, 2, 3, 5, 1, 4), want_h)
    assert want[..., 0, :].max() > 0
