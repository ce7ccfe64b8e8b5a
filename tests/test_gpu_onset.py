"""Heatwave onset and end (HWO, HWE: HDP_B200_ONSET) on the device, every plane bit for bit against tests/onset_oracle.py (the
reference's indicate_hot_days and index_heatwaves, then the first and last positive id of each season slice) and planes 0 - 3 also
against the call without the flag: every k_scan instantiation with the run filter on and off, season edges, lane widths, cold spells,
compound days, the intensity calls, the host pipeline, thresholds without a day-of-year axis, the metric layer and one full-size call."""
import ctypes

import numpy as np
import pytest

import oracle
from onset_oracle import NO_DAY, cold_onset_batch, compound_onset_batch, onset_batch
from test_compound_host import compound_oracle
from test_instance_table import SCAN_T, metrics_choice, scan_case, scan_instances

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def core():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from hdp_b200 import _core
    return _core


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


def ref_layout(out_u16):
    """uint16 [4, P, D, Y, C] -> the reference's int64 [P, D, C, 4, Y]."""
    return host(out_u16)[:4].astype(np.int64).transpose(1, 2, 4, 0, 3)


def check(core, x, thr, args, cold=False, want=None):
    """metrics_array with onset=True on (x, thr): planes 0 - 3 against the flagless call and the reference's metrics, planes 4 and 5
    against the onset oracle (``want``, computed unless given).  Returns the six planes (host)."""
    xd, thd = dev(x), dev(thr)
    got = core.metrics_array(xd, thd, *args, cold=cold, onset=True)
    assert got.shape[0] == 6
    assert torch.equal(got[:4], core.metrics_array(xd, thd, *args, cold=cold))
    s = -1.0 if cold else 1.0
    assert np.array_equal(ref_layout(got), oracle.metrics_batch((s * x).astype(np.float32), s * thr, *args))
    if want is None:
        want = (cold_onset_batch if cold else onset_batch)(x, thr, *args)
    assert np.array_equal(host(got[4:]), want)
    return host(got)


def ar1_case(rng, T, C, P):
    """AR(1) samples, persistent enough for long runs; per (cell, percentile) thresholds at mixed hot-day densities, constant over
    the day-of-year axis (365 rows); cell 0 hot all the time, cell 1 never."""
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
    x = z.astype(np.float32)
    dens = rng.uniform(0.02, 0.9, (C, P))
    q = np.stack([[np.quantile(x[:, c], 1 - dens[c, p]) for p in range(P)] for c in range(C)]).astype(np.float64)
    x[:, 0] = 10.0
    x[:, 1] = -10.0
    return x, np.repeat(q[:, None, :], 365, axis=1)


# ------------------------------------------------------------------------------------------------ every k_scan instantiation
@pytest.mark.parametrize("inst", scan_instances(), ids=lambda i: "b{}_ng{}_ks{}_f{}{}".format(*i))
def test_scan_instantiation(core, lib, inst):
    from hdp_b200 import _tables as tb
    defs, north, south = scan_case(*inst)
    rng = np.random.default_rng(sum(inst))
    C, P = 97, 2
    x, thr = ar1_case(rng, SCAN_T, C, P)
    dm = tb.doy_map(tb.TimeAxis.daily((2001, 1, 1), SCAN_T, "noleap").dayofyr)
    is_south = rng.integers(0, 2, C).astype(np.uint8)          # both hemispheres in every warp
    args = (dm, defs.tolist(), north, south, is_south)
    want = onset_batch(x, thr, *args)
    assert (want != NO_DAY).any() and (want == NO_DAY).any()
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        rc, info = metrics_choice(defs, north, south)
        assert rc == 0 and tuple(info[:3]) == inst[:3] and (info[4], info[5]) == ((inst[3], inst[4]) if on else (0, 0))
        check(core, x, thr, args, want=want)


# ------------------------------------------------------------------------------------------------ season edges
def designed_case(C=45, T=900):
    """Runs placed on the season edges: cell c has hot runs [s, s + n) at a few days per cell, plus AR(1) noise in the later cells."""
    rng = np.random.default_rng(5)
    x = np.full((T, C), -1.0, np.float32)
    runs = [(95, 10), (99, 1), (100, 1), (100, 3), (148, 5), (149, 1), (240, 20), (249, 1), (250, 4), (0, 4), (T - 3, 3), (365, 1),
            (364, 3), (398, 5), (500, 40), (598, 3)]
    for c in range(C):
        for s, n in runs[c % len(runs):c % len(runs) + 3]:
            x[s:s + n, c] = 1.0
    noisy = rng.standard_normal((T, C)) > 0.6
    x[:, C // 2:] = np.where(noisy[:, C // 2:], 1.0, x[:, C // 2:])
    return x, np.zeros((C, 1, 1))


# season entries: starts and ends inside runs, a one-day season, empty / reversed / negative / out-of-range entries and overlapping
# seasons (several passes of k_scan)
EDGE_NORTH = [[100, 150], [149, 150], [-800, -650], [250, 250], [400, 398], [600, 5000], [-5000, 2], [364, 366], [96, 400]]
EDGE_SOUTH = [[99, 100], [100, 101], [0, 900], [-1, 900], [240, 250], [897, 2000], [250, 252], [500, 505], [505, 500]]


def test_season_edges(core, lib):
    x, thr = designed_case()
    T, C = x.shape
    is_south = (np.arange(C) % 3 == 1).astype(np.uint8)
    defs = [[1, 0, 0], [3, 0, 0], [2, 1, 1], [3, 2, 2], [5, 3, 0]]
    args = (np.zeros(T, np.int64), defs, EDGE_NORTH, EDGE_SOUTH, is_south)
    assert metrics_choice(defs, EDGE_NORTH, EDGE_SOUTH, T)[1][6] > 1          # overlapping seasons: several passes
    want = onset_batch(x, thr, *args)
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        got = check(core, x, thr, args, want=want)
    # one-day blocks: the run [99, 100) in the season [99, 100), and a run crossing into [100, 101)
    assert (got[4:, :, :, 1][..., is_south == 1] != NO_DAY).any()
    assert (got[4, :, :, 0][..., is_south == 0] == 0).any()                    # a run that began before the season
    assert (got[5, :, :, 0][..., is_south == 0] == 150 - 100 - 1).any()        # one that continues past its end


@pytest.mark.parametrize("days,bits", [(255, 8), (256, 16), (65535, 16)])
def test_last_day_of_the_longest_seasons(core, lib, days, bits):
    # a heatwave on the last day of a 255-day season (8-bit lanes: the largest offset they hold), of a 256-day season (16-bit lanes)
    # and of a 65 535-day season (the largest the u16 output holds); and one that runs past it
    T = 180 * 365 if days > 300 else 700
    C = 37
    x = np.full((T, C), -1.0, np.float32)
    a = 10
    b = a + days
    x[b - 4:b, 0::2] = 1.0                                       # ends on the season's last day
    x[b - 2:b + 5, 1::2] = 1.0                                   # continues past it
    x[a:a + 3, 0::3] = 1.0                                       # and one on its first days
    thr = np.zeros((C, 1, 1))
    defs = [[1, 0, 0], [3, 0, 0], [2, 1, 1], [8000, 0, 0]]
    north = south = [[a, b]]
    is_south = (np.arange(C) % 2).astype(np.uint8)
    assert metrics_choice(defs, north, south, T)[1][0] == bits
    args = (np.zeros(T, np.int64), defs, north, south, is_south)
    got = check(core, x, thr, args)
    assert got[5, 0, 0, 0, 0] == days - 1 and got[5, 0, 0, 0, 1] == days - 1 and got[4, 0, 0, 0, 3] == 0
    assert (got[4:, 0, 3] == NO_DAY).all()


@pytest.mark.parametrize("D", [1, 32])
def test_definition_counts(core, lib, D):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(D)
    ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "noleap")
    C, P = 77, 3                                                 # not a multiple of 32
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    defs = [[3, 1, 1]] if D == 1 else [[int(rng.integers(1, 6)), int(rng.integers(0, 4)), int(rng.integers(0, 4))] for _ in range(D)]
    args = (tb.doy_map(ax.dayofyr), defs, st.north, st.south, (np.arange(C) % 2).astype(np.uint8))
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        check(core, x, thr, args)


# ------------------------------------------------------------------------------------------------ cold spells, compound days
def test_cold_is_warm_on_negated_inputs(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(8)
    ax = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "noleap")
    C, P = 70, 2
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    args = (tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [2, 2, 3]], st.south, st.north, (np.arange(C) % 2).astype(np.uint8))
    got = check(core, x, thr, args, cold=True)
    warm = core.metrics_array(dev(-x), dev(-thr), *args, onset=True)
    assert np.array_equal(got, host(warm))


def _pair(rng, T, C, P):
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.6 * z[t - 1] + 0.8 * z[t]
    xa = (20 + 3 * z).astype(np.float32)
    xb = (12 + 3 * (0.7 * z + 0.7 * rng.standard_normal((T, C)))).astype(np.float32)
    ta = 20 + np.linspace(0.5, 3, P)[None, None, :] + 0.3 * rng.standard_normal((C, 365, 1))
    tb_ = 12 + np.linspace(0.5, 3, P)[None, None, :] + 0.3 * rng.standard_normal((C, 365, 1))
    return xa, ta, xb, tb_


@pytest.mark.parametrize("cold", [False, True])
def test_compound(core, cold):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(12)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C, P = 41, 3
    xa, ta, xb, tb_ = _pair(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    north, south = (st.south, st.north) if cold else (st.north, st.south)
    args = (tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [1, 0, 0]], north, south, (np.arange(C) % 2).astype(np.uint8))
    d = [dev(a) for a in (xa, ta, xb, tb_)]
    got = core.compound_metrics_array(*d, *args, cold=cold, onset=True)
    assert torch.equal(got[:4], core.compound_metrics_array(*d, *args, cold=cold))
    want_met, _ = compound_oracle(xa, ta, xb, tb_, *args, intensity=False, cold=cold)
    assert np.array_equal(ref_layout(got), want_met)
    assert np.array_equal(host(got[4:]), compound_onset_batch(xa, ta, xb, tb_, *args, cold=cold))
    assert (host(got[4:]) != NO_DAY).any()
    # compound(A, A) = single(A), all six planes
    same = core.compound_metrics_array(d[0], d[1], d[0], d[1], *args, cold=cold, onset=True)
    assert torch.equal(same, core.metrics_array(d[0], d[1], *args, cold=cold, onset=True))
    # the intensity call with metrics_out: the same planes, the same intensity as without the flag
    met = torch.zeros_like(got)
    heat = core.compound_intensity_array(*d, *args, metrics_out=met, cold=cold, onset=True)
    assert torch.equal(met, got) and torch.equal(heat, core.compound_intensity_array(*d, *args, cold=cold))


def test_intensity_with_metrics_out(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(13)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C, P = 50, 2
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    args = (tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1]], st.north, st.south, (np.arange(C) % 2).astype(np.uint8))
    xd, thd = dev(x), dev(thr)
    for cold in (False, True):
        met = torch.zeros((6, P, 2, len(st.north), C), dtype=torch.uint16, device="cuda")
        heat = core.intensity_array(xd, thd, *args, metrics_out=met, cold=cold, onset=True)
        assert torch.equal(met, core.metrics_array(xd, thd, *args, cold=cold, onset=True))
        assert torch.equal(heat, core.intensity_array(xd, thd, *args, cold=cold))
    with pytest.raises(TypeError, match=r"\[6, P, D, Y, C\]"):
        core.intensity_array(xd, thd, *args, metrics_out=met[:4].contiguous(), onset=True)


# ------------------------------------------------------------------------------------------------ host pipeline, long runs
@pytest.mark.parametrize("chunk", [None, "64"])
def test_host_pipeline(core, monkeypatch, chunk):
    from hdp_b200 import _tables as tb
    if chunk:
        monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", chunk)
    rng = np.random.default_rng(23)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1966-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2006-12-31", "noleap")
    wt = tb.window_tables(base_ax.dayofyr, 7)
    C = 299
    cyc = lambda ax: 15 + 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)            # noqa: E731
    xb = (cyc(base_ax) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (cyc(run_ax) + 1 + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    xa, ta, xb2, tb_ = _pair(rng, len(run_ax), C, 3)
    q = np.array([0.9, 0.95, 0.99])
    thr_d = core.thresholds_array(dev(xb), wt, q)
    thr_h = thr_d.cpu().numpy()
    thr_k = core.thresholds_host(xb, wt, q, keep=True)                                            # remembered resident copy
    assert core.resident_thresholds(thr_k) is not None
    st = tb.hemisphere_ranges(run_ax)
    args = (tb.doy_map(run_ax.dayofyr), [[3, 0, 0], [3, 1, 1], [4, 2, 1]], st.north, st.south, (rng.random(C) < 0.5).astype(np.uint8))
    want = check(core, xr, thr_h, args)
    pinned = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()             # noqa: E731
    for X, TH in ((xr, thr_h), (pinned(xr), thr_h), (xr, pinned(thr_h)), (xr, thr_d), (np.ascontiguousarray(xr.T).T, thr_k)):
        assert np.array_equal(core.metrics_host(X, TH, *args, onset=True), want)
        met_h = np.zeros_like(want)
        core.intensity_host(X, TH, *args, metrics_out=met_h, onset=True)
        assert np.array_equal(met_h, want)
    out = pinned(np.zeros_like(want))
    core.metrics_host(xr, thr_h, *args, out=out, onset=True)
    assert np.array_equal(out, want)
    want_c = host(core.compound_metrics_array(*(dev(a) for a in (xa, ta, xb2, tb_)), *args, onset=True))
    assert np.array_equal(core.compound_metrics_host(xa, ta, xb2, tb_, *args, onset=True), want_c)
    met_c = pinned(np.zeros_like(want_c))
    core.compound_intensity_host(xa, ta, xb2, tb_, *args, metrics_out=met_c, onset=True)
    assert np.array_equal(met_c, want_c)
    core.host_release()


def test_doy_free_thresholds_over_a_long_run(core):
    # n_doy = 1 over a CMIP-length run (31 390 days): words of 32 days, seasons of the whole run's calendar
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(31390)
    run_ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C = 37
    xr = (16 + 8 * np.sin(2 * np.pi * run_ax.dayofyr[:, None] / 365) + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    st = tb.hemisphere_ranges(run_ax)
    args = (np.zeros(len(run_ax), np.int64), workloads.README_DEFS, st.north, st.south, (np.arange(C) % 2).astype(np.uint8))
    got = check(core, xr, np.full((C, 1, 2), 0.0) + np.array([21.0, 24.5]), args)
    assert (got[4:] != NO_DAY).any()


# ------------------------------------------------------------------------------------------------ the metric layer
def test_metric_functions(core):
    from hdp_b200 import _tables as tb, measure, metric, threshold, utils, xr
    grid = (2, 3)
    test = utils.generate_test_warming_dataarray(grid_shape=grid, add_noise=True)
    rh = utils.generate_test_rh_dataarray(grid_shape=grid)
    measures = measure.format_standard_measures([test], rh=rh)
    na, nb = list(measures.keys())[:2]
    thresholds = threshold.compute_thresholds(measures, np.array([0.9, 0.95]))
    defs = [[3, 0, 0], [3, 1, 1], [4, 1, 1]]
    ma, mb = measures[na], measures[nb]
    ta, tb_ = thresholds[f"{na}_threshold"], thresholds[f"{nb}_threshold"]
    t_axis = utils.time_axis_of(ma)
    st = tb.hemisphere_ranges(t_axis)
    south = tb.is_south(np.tile(np.linspace(-90, 90, 3), 2))
    ra, rb = (np.ascontiguousarray(xr.values_of(m).reshape(6, -1).T) for m in (ma, mb))
    tha, thb = (np.ascontiguousarray(xr.values_of(t).reshape(6, 365, 2)) for t in (ta, tb_))
    dm = tb.doy_map(t_axis.dayofyr)

    def as_days(plane):                                          # [P, D, Y, C] u16 -> the variable's float32 [P, D, lon, lat, Y]
        return np.where(plane == NO_DAY, np.nan, plane.astype(np.float32)).transpose(0, 1, 3, 2)
    for cold in (False, True):
        args = (dm, defs, *((st.south, st.north) if cold else (st.north, st.south)), south)
        names = ("CSO", "CSE") if cold else ("HWO", "HWE")
        ds = metric.compute_individual_metrics(ma, ta, defs, cold=cold, onset=True)
        want = (cold_onset_batch if cold else onset_batch)(ra, tha, *args)
        plain = metric.compute_individual_metrics(ma, ta, defs, cold=cold)
        for n in plain.keys():
            assert np.array_equal(xr.values_of(ds[n]), xr.values_of(plain[n]))
        for i, n in enumerate(names):
            v = np.asarray(xr.values_of(ds[n])).reshape(2, len(defs), 6, -1)
            assert v.dtype == np.float32 and np.array_equal(v, as_days(want[i]), equal_nan=True)
            assert ds[n].attrs["units"] == "days"
        grp = metric.compute_group_metrics({na: ma}, {f"{na}_threshold": ta}, defs, cold=cold, onset=True)
        assert np.array_equal(xr.values_of(grp[f"{na}.{na}_threshold.{names[0]}"]), xr.values_of(ds[names[0]]), equal_nan=True)
        cds = metric.compute_compound_metrics(ma, ta, mb, tb_, defs, cold=cold, onset=True, intensity=True)
        want_c = compound_onset_batch(ra, tha, rb, thb, *args, cold=cold)
        for i, n in enumerate(names):
            v = np.asarray(xr.values_of(cds[n])).reshape(2, len(defs), 6, -1)
            assert np.array_equal(v, as_days(want_c[i]), equal_nan=True) and "measure" not in cds[n].dims
        if not cold:
            assert (want != NO_DAY).any()
    core.host_release()


# ------------------------------------------------------------------------------------------------ one full-size call
def test_cmip6_full_size(core):
    # cmip6_1deg (64 800 cells, 31 390 days, P 10, the README definitions) on the device; a sample of cells against the oracle
    from hdp_b200 import _tables as tb, workloads
    w = workloads.get("cmip6_1deg")
    ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C, T, P = w.cells, len(ax), len(w.percentiles)
    g = torch.Generator(device="cuda").manual_seed(7)
    doy = torch.as_tensor(ax.dayofyr, device="cuda", dtype=torch.float32)[:, None]
    x = (25 + 10 * torch.sin(2 * np.pi * (doy - 110) / 365) + 3 * torch.randn((T, C), device="cuda", generator=g)).float()
    off = torch.linspace(2, 5, P, device="cuda", dtype=torch.float64)
    cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
    thr = (25 + cyc_d[None, :, None] + off[None, None, :]).expand(C, 365, P).contiguous()
    st = tb.hemisphere_ranges(ax)
    is_south = ((np.arange(C) // w.n_lon) < w.n_lat // 2).astype(np.uint8)
    args = (tb.doy_map(ax.dayofyr), w.defs, st.north, st.south, is_south)
    met = core.metrics_array(x, thr, *args, onset=True)
    assert torch.equal(met[:4], core.metrics_array(x, thr, *args))
    torch.cuda.synchronize()
    cells = np.sort(np.random.default_rng(0).choice(C, 24, replace=False))
    sel = torch.as_tensor(cells, device="cuda")
    xs, ts = host(x[:, sel]), host(thr[sel])
    got = host(met.view(torch.int16)[..., sel]).view(np.uint16)                                  # (no uint16 gather on the device)
    assert np.array_equal(got[:4].astype(np.int64).transpose(1, 2, 4, 0, 3), oracle.metrics_batch(xs, ts, *args[:4], is_south[cells]))
    assert np.array_equal(got[4:], onset_batch(xs, ts, *args[:4], is_south[cells]))
    assert (got[4:] != NO_DAY).any()


# ------------------------------------------------------------------------------------------------ where the flag is refused
def test_flag_refused_where_it_has_no_output(core):
    from hdp_b200 import _lib
    L = _lib.lib()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)              # noqa: E731
    T, C = 64, 33
    x, thr = torch.zeros((T, C), device="cuda"), torch.zeros((C, 1, 1), dtype=torch.float64, device="cuda")
    dm = np.zeros(T, np.int32)
    defs, seas = np.array([[3, 0, 0]], np.int32), np.array([[0, T]], np.int32)
    ws = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    heat = torch.empty((3, 1, 1, 1, C), device="cuda")
    mask = torch.empty((1, T, C), dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    tab = (p(dm), p(defs), 1, p(seas), p(seas), 1, None)
    assert L.hdp_b200_intensity(x.data_ptr(), C, T, C, 1, thr.data_ptr(), 1, 1, *tab, heat.data_ptr(), None, ws.data_ptr(), ws.numel(), s,
                                0x200) == -1
    assert L.hdp_b200_compound(x.data_ptr(), C, 1, x.data_ptr(), C, 1, C, T, thr.data_ptr(), thr.data_ptr(), 1, 1, *tab, None,
                               torch.empty((2, 3, 1, 1, 1, C), device="cuda").data_ptr(), ws.data_ptr(), ws.numel(), s, 0x200) == -1
    assert L.hdp_b200_compound_hot_days(x.data_ptr(), C, 1, x.data_ptr(), C, 1, C, T, thr.data_ptr(), thr.data_ptr(), 1, 1, p(dm),
                                        mask.data_ptr(), ws.data_ptr(), ws.numel(), s, 0x200) == -1
    from hdp_b200 import _tables as tb
    wt = tb.window_tables(tb.TimeAxis.date_range("1961-01-01", "1962-12-31", "noleap").dayofyr, 2)
    ti, wr, q = np.ascontiguousarray(wt.time_index, np.int32), np.ascontiguousarray(wt.win_rows, np.int32), np.array([0.9])
    xb = torch.zeros((730, C), device="cuda")
    out = torch.empty((C, wt.n_doy, 1), dtype=torch.float64, device="cuda")
    assert L.hdp_b200_thresholds(xb.data_ptr(), C, 730, C, 1, p(ti), p(wr), wt.n_doy, wt.n_y, wt.width, p(q), 1, out.data_ptr(),
                                 ws.data_ptr(), ws.numel(), s, 0x200) == -1
    torch.cuda.synchronize()
