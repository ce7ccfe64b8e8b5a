"""Trend statistics (hdp_b200_trend, k_trend) on the device, every plane bit for bit against tests/trend_oracle.py (mk_p to 1e-13
relative: it goes through the device's erfc): both dtypes, Y from 1 to 512, C not a multiple of 32, heavy ties, the u16 sentinel, f32
NaN and +-inf, signed zeros, both median parities and both CI clamps, the real metric and intensity outputs, the metric layer and
one full-size cmip6_1deg measure."""
from statistics import NormalDist

import numpy as np
import pytest

from test_gpu_onset import ar1_case
from test_trend_host import random_series
from trend_oracle import NAMES, trend_batch

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def core():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from hdp_b200 import _core
    return _core


def zq_of(alpha):
    return NormalDist().inv_cdf(alpha / 2)


def same(got, want):
    """every plane but mk_p bit for bit (NaN where NaN), mk_p to 1e-13 relative"""
    got = got.cpu().numpy() if isinstance(got, torch.Tensor) else got
    got, want = got.reshape(8, -1), want.reshape(8, -1)
    for q, name in enumerate(NAMES):
        if name == "mk_p":
            assert np.array_equal(np.isnan(got[q]), np.isnan(want[q]))
            ok = ~np.isnan(want[q])
            assert np.allclose(got[q][ok], want[q][ok], rtol=1e-13, atol=0), name
        else:
            nan = np.isnan(want[q])
            assert np.array_equal(np.isnan(got[q]), nan), name
            assert np.array_equal(got[q][~nan].view(np.uint64), want[q][~nan].view(np.uint64)), name


def run(core, x, missing=None, alpha=0.05):
    got = core.trend_array(torch.as_tensor(np.ascontiguousarray(x)).cuda(), missing=missing, alpha=alpha)
    assert got.shape == (8, *x.shape[:-2], x.shape[-1]) and got.dtype == torch.float64
    same(got, trend_batch(x.reshape(-1, *x.shape[-2:]), zq_of(alpha), missing))
    return got.cpu().numpy()


@pytest.mark.parametrize("kind", ["poisson", "high", "float"])
@pytest.mark.parametrize("Y", [1, 2, 3, 86, 251, 512])
def test_random_series(core, kind, Y):
    rng = np.random.default_rng(Y + 100 * len(kind))
    C = 45 if Y <= 86 else 35
    x = np.concatenate([random_series(rng, kind, Y, C) for _ in range(2 if Y <= 86 else 1)])
    miss = 0xFFFF if kind == "poisson" else None
    got = run(core, x, miss)
    assert (got[7] >= 2).any() or Y < 2
    if kind == "high":                                              # values near 65 534 without a sentinel: 0xFFFF is a value
        x2 = x.copy()
        x2[:, ::3] = 0xFFFF
        got = run(core, x2)
        assert (got[7] == Y).all()


def test_leading_dims_and_alpha(core):
    rng = np.random.default_rng(3)
    x = rng.poisson(2.0, (2, 3, 40, 33)).astype(np.uint16)
    for alpha in (0.01, 0.05, 0.3):
        run(core, x, alpha=alpha)


def test_signed_zeros_and_infinities(core):
    x = np.zeros((1, 12, 37), np.float32)
    rng = np.random.default_rng(9)
    x[0] = np.where(rng.random((12, 37)) < 0.5, -0.0, 0.0)
    x[0, :, 5:] += rng.integers(-1, 2, (12, 32)).astype(np.float32)
    x[0, 3, 7:20] = np.inf
    x[0, 4, 10:30] = -np.inf
    x[0, 5, 12:33] = np.nan
    x[0, :, 36] = np.float32(3e38) * np.where(np.arange(12) % 2, 1, -1)  # differences beyond float32, exact in float64
    run(core, x)


def test_median_parities_and_ci_clamps(core):
    # n = 2 (N = 1: both CI ranks clamp to the one slope), n = 3 (N = 3, odd), n = 4 (N = 6, even), all equal (var with ties only),
    # and a large alpha, where Rl and Ru meet the median ranks
    cols = [[0, 5], [1, 2, 4], [0, 1, 3, 4], [2, 2, 2, 2, 2], [9, 1, 8, 2, 7, 3, 6, 4, 5]]
    x = np.full((1, 9, 33), 0xFFFF, np.uint16)
    for c, v in enumerate(cols):
        x[0, :len(v), c] = v
        x[0, -len(v):, c + len(cols)] = v
    for alpha in (0.05, 0.999):
        got = run(core, x, 0xFFFF, alpha)
    assert got[0, 0, 0] == got[2, 0, 0] == got[3, 0, 0] == 5.0


def test_unsupported_and_invalid(core):
    from hdp_b200 import _lib
    x = torch.zeros((1, 513, 4), dtype=torch.float32, device="cuda")
    with pytest.raises(_lib.HdpB200Error) as e:
        core.trend_array(x)
    assert e.value.code == -2
    L = _lib.lib()
    out = torch.empty((8, 1, 4), dtype=torch.float64, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    y = torch.zeros((1, 5, 4), dtype=torch.float32, device="cuda")
    assert L.hdp_b200_trend(y.data_ptr(), 2, 1, 5, 4, -1, 0.5, out.data_ptr(), s) == -1          # zq must be < 0
    assert L.hdp_b200_trend(y.data_ptr(), 3, 1, 5, 4, -1, -1.96, out.data_ptr(), s) == -1         # unknown dtype
    assert L.hdp_b200_trend(y.data_ptr(), 1, 1, 5, 4, 70000, -1.96, out.data_ptr(), s) == -1      # sentinel outside uint16
    assert L.hdp_b200_trend(y.data_ptr(), 2, 0, 5, 4, -1, -1.96, out.data_ptr(), s) == 0          # nothing to do


def warming_outputs(core):
    """intensity_array with onset=True on an AR(1) field with a warming trend over 40 seasons of 100 days: u16 [6, P, D, Y, C] and f32
    [3, P, D, Y, C]."""
    rng = np.random.default_rng(11)
    Y, L, C, P = 40, 100, 45, 2
    x, thr = ar1_case(rng, Y * L, C, P)
    x = (x + 0.02 * (np.arange(Y * L) // L)[:, None]).astype(np.float32)
    seasons = np.stack([np.arange(Y) * L + 10, np.arange(Y) * L + 90], 1)
    defs = [[3, 0, 0], [2, 1, 1]]
    dm = np.arange(Y * L) % 365
    met = torch.empty((6, P, len(defs), Y, C), dtype=torch.uint16, device="cuda")
    heat = core.intensity_array(torch.as_tensor(x).cuda(), torch.as_tensor(thr).cuda(), dm, defs, seasons, seasons,
                                metrics_out=met, onset=True)
    return met, heat


def test_metric_and_intensity_outputs(core):
    met, heat = warming_outputs(core)
    m = met.cpu().numpy()
    assert (m[4] == core.NO_DAY).any() and (m[4] != core.NO_DAY).any()
    run(core, m[:4])
    got = run(core, m[4:], core.NO_DAY)
    assert (got[7] < m.shape[3]).any()
    h = heat.cpu().numpy()
    got = run(core, h)
    assert (got[0] > 0).mean() > 0.5                                # the warming shows
    # the device tensors as they are (views of the output, no copies)
    same(core.trend_array(met[:4]), trend_batch(m[:4].reshape(-1, *m.shape[-2:]), zq_of(0.05)))


def _measure_and_threshold(name, seed):
    from hdp_b200 import utils, xr
    m = utils.generate_test_warming_dataarray("1990-01-01", "2009-12-31", grid_shape=(2, 3), add_noise=True).astype(np.float32)
    m = xr.DataArray(xr.values_of(m) + np.float32(seed), dims=list(m.dims), coords=dict(xr.coords_of(m)), name=name,
                     attrs={**m.attrs, "units": "degC"})
    lat, lon = xr.coord_values(m, "lat"), xr.coord_values(m, "lon")
    base = float(np.nanmean(xr.values_of(m)))
    thr = xr.DataArray(np.full((2, 3, 365, 2), base) + np.array([0.5, 1.0]), dims=["lon", "lat", "doy", "percentile"],
                       coords={"lon": lon, "lat": lat, "doy": np.arange(1, 366), "percentile": np.array([0.9, 0.95])}, name="t",
                       attrs={})
    return m, thr


def _check_trends(ds, trends, alpha=0.05):
    from hdp_b200 import xr
    lead_dims = ("measure", "percentile", "definition")
    names = [v for v in ds if "time" in ds[v].dims]
    assert sorted(trends.keys()) == sorted(f"{v}_{s}" for v in names for s in NAMES)
    for v in names:
        da = ds[v]
        dims = tuple(da.dims)
        lead = [d for d in dims if d in lead_dims]
        cells = [d for d in dims if d not in lead_dims and d != "time"]
        vals = np.asarray(xr.values_of(da)).transpose([dims.index(d) for d in (*lead, "time", *cells)])
        Y = vals.shape[len(lead)]
        x = vals.astype(np.uint16 if np.issubdtype(vals.dtype, np.integer) else np.float32).reshape(-1, Y, int(np.prod(vals.shape[len(lead) + 1:])))
        want = trend_batch(x, zq_of(alpha))
        got = np.stack([np.asarray(xr.values_of(trends[f"{v}_{s}"])) for s in NAMES])
        assert tuple(trends[f"{v}_slope"].dims) == (*lead, *cells)
        same(got, want)


def test_metric_layer(core):
    from hdp_b200 import metric
    ma, thr = _measure_and_threshold("tmax", 0)
    mb, _ = _measure_and_threshold("tmin", -1)
    defs = [[3, 0, 0], [3, 1, 1]]
    ds = metric.compute_individual_metrics(ma, thr, defs, check_variables=False, intensity=True, onset=True)
    tr = metric.compute_metric_trends(ds)
    _check_trends(ds, tr)
    assert tr["HWF_slope"].attrs["units"] == "heatwave days per year" and tr["HWC_intercept"].attrs["units"] == "degC"
    assert tr.attrs["alpha"] == 0.05 and "trend_method" in tr.attrs
    ma.attrs["baseline_variable"] = thr.attrs["baseline_variable"] = "t"
    grp = metric.compute_group_metrics({"t": ma}, {"t_threshold": thr}, defs, check_variables=False, onset=True)
    _check_trends(grp, metric.compute_metric_trends(grp, alpha=0.1), 0.1)
    cds = metric.compute_compound_metrics(ma, thr, mb, thr, defs, check_variables=False, intensity=True, onset=True)
    ctr = metric.compute_metric_trends(cds)
    _check_trends(cds, ctr)
    assert tuple(ctr["HWC_slope"].dims)[0] == "measure"
    core.host_release()


def test_cmip6_full_size_measure(core):
    # one full-size cmip6_1deg measure with onset: [6, P, D, Y, C] u16, two calls (planes 0 - 3 without a sentinel, 4 - 5 with 0xFFFF),
    # a sample of cells against the oracle
    from hdp_b200 import _tables as tb, workloads
    w = workloads.get("cmip6_1deg")
    ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C, T, P = w.cells, len(ax), len(w.percentiles)
    g = torch.Generator(device="cuda").manual_seed(7)
    doy = torch.as_tensor(ax.dayofyr, device="cuda", dtype=torch.float32)[:, None]
    year = torch.as_tensor(ax.year - ax.year[0], device="cuda", dtype=torch.float32)[:, None]
    x = (25 + 10 * torch.sin(2 * np.pi * (doy - 110) / 365) + 3 * torch.randn((T, C), device="cuda", generator=g) + 0.03 * year).float()
    off = torch.linspace(2, 5, P, device="cuda", dtype=torch.float64)
    cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
    thr = (25 + cyc_d[None, :, None] + off[None, None, :]).expand(C, 365, P).contiguous()
    st = tb.hemisphere_ranges(ax)
    is_south = ((np.arange(C) // w.n_lon) < w.n_lat // 2).astype(np.uint8)
    met = core.metrics_array(x, thr, tb.doy_map(ax.dayofyr), w.defs, st.north, st.south, is_south, onset=True)
    del x
    a = core.trend_array(met[:4])
    b = core.trend_array(met[4:], missing=core.NO_DAY)
    assert a.shape == (8, 4, P, len(w.defs), C) and b.shape == (8, 2, P, len(w.defs), C)
    cells = np.sort(np.random.default_rng(0).choice(C, 16, replace=False))
    sel = torch.as_tensor(cells, device="cuda")
    m = met.view(torch.int16)[..., sel].cpu().numpy().view(np.uint16)                  # (no uint16 gather on the device)
    Y = m.shape[3]
    same(a[..., sel].cpu().numpy(), trend_batch(m[:4].reshape(-1, Y, cells.size), zq_of(0.05)))
    same(b[..., sel].cpu().numpy(), trend_batch(m[4:].reshape(-1, Y, cells.size), zq_of(0.05), core.NO_DAY))
    assert float(torch.nanmean(a[0, 0]).item()) > 0                  # HWF rises with the warming
