"""Every compiled k_thr_net instance and k_scan instantiation, the u16 output's boundaries, thresholds without a day-of-year axis
over a long run, and every sample layout the array API accepts - all against the oracle.

The cases come from the tables of tests/test_instance_table.py, which checks without a GPU that each one reaches its instance."""
import numpy as np
import pytest

import oracle
from conftest import bits_equal
from intensity_oracle import intensity_batch
from test_instance_table import NET_CALENDARS, NET_CASES, metrics_choice, net_axis, scan_case, scan_instances, SCAN_T

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
    L.hdp_b200_thresholds_force_generic(0)
    L.hdp_b200_metrics_run_filter(1)


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def ref_layout(out_u16):
    """uint16 [4, P, D, Y, C] -> the reference's int64 [P, D, C, 4, Y]."""
    return np.asarray(out_u16.cpu().numpy() if isinstance(out_u16, torch.Tensor) else out_u16).astype(np.int64).transpose(1, 2, 4, 0, 3)


def heat_layout(out_f32):
    """float32 [3, P, D, Y, C] -> the oracle's [P, D, C, 3, Y]."""
    return np.asarray(out_f32.cpu().numpy() if isinstance(out_f32, torch.Tensor) else out_f32).transpose(1, 2, 4, 0, 3)


def same_f32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def launched(core, fn):
    """Runs fn() and returns the names of the kernels it launched."""
    core.timing_enable(True)
    core.timing_read()
    try:
        fn()
    finally:
        names = [n for n, _ in core.timing_read()]
        core.timing_enable(False)
    return names


# ------------------------------------------------------------------------------------------------ A. every k_thr_net instance
def net_columns(rng, T, C):
    """The column recipe of test_gpu_parity.py::test_thresholds_network_kernel: ties, constants, trends, samples equal to the
    kernel's pad value, NaN / +-inf (handed over to k_thr_seg) and a NaN in the last sample, which every -1 pad reads."""
    x = (15 + 3 * rng.standard_normal((T, C))).astype(np.float32)
    x[:, 0] = np.round(x[:, 0])
    x[:, 1] = 2.5
    x[:, 2] = np.arange(T, dtype=np.float32) * np.float32(1e-3)
    x[:, 3] = -np.arange(T, dtype=np.float32)
    x[T // 2, 4] = 3e38
    x[:, 5] = -3.402823466e+38
    x[:, 6] = np.where(rng.random(T) < 0.3, 99.0, x[:, 6])
    x[rng.integers(0, T, 3), 11] = np.nan
    x[rng.integers(0, T, 3), 12] = np.inf
    x[rng.integers(0, T, 3), 13] = -np.inf
    x[T - 1, 14] = np.nan
    x[0, C - 1] = np.inf
    return x


@pytest.mark.parametrize("calendar", NET_CALENDARS)
@pytest.mark.parametrize("inst", sorted(NET_CASES), ids=lambda i: "ny{}_k{}_m{}".format(*i))
def test_net_instance(core, lib, inst, calendar):
    from hdp_b200 import _tables as tb
    years, radius, q, tm_warps = NET_CASES[inst]
    ax = net_axis(calendar, years)
    wt = tb.window_tables(ax.dayofyr, radius)
    T, C = len(ax), 45                                          # a full tile and a ragged one
    x = net_columns(np.random.default_rng(sum(inst) + len(calendar)), T, C)
    want = oracle.thresholds_batch(x, wt.window_samples(), np.array(q))
    for mode in ((0, 6) if tm_warps else (0,)):                 # with tensor memory (the default) and without it
        lib.hdp_b200_thresholds_force_generic(mode)
        got = []
        assert "k_thr_net" in launched(core, lambda: got.append(core.thresholds_array(dev(x), wt, q)))
        assert bits_equal(got[0].cpu().numpy(), want), mode


# ------------------------------------------------------------------------------------------------ B. every k_scan instantiation
def ar1_case(rng, T, C, P):
    """AR(1) samples, persistent enough for long runs at every density; per (cell, percentile) thresholds at mixed hot-day
    densities, constant over the day-of-year axis (365 rows)."""
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
    x = z.astype(np.float32)
    dens = rng.uniform(0.02, 0.9, (C, P))
    q = np.stack([[np.quantile(x[:, c], 1 - dens[c, p]) for p in range(P)] for c in range(C)]).astype(np.float64)
    x[:, 0] = 10.0                                              # one run over the whole series
    x[:, 1] = -10.0
    return x, np.repeat(q[:, None, :], 365, axis=1)


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
    want = oracle.metrics_batch(x, thr, *args)
    want_heat = intensity_batch(x, thr, *args)
    xd, thd = dev(x), dev(thr)
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        rc, info = metrics_choice(defs, north, south)
        assert rc == 0 and tuple(info[:3]) == inst[:3] and (info[4], info[5]) == ((inst[3], inst[4]) if on else (0, 0))
        met = core.metrics_array(xd, thd, *args)
        assert np.array_equal(ref_layout(met), want), on
        met2 = torch.zeros_like(met)
        heat = core.intensity_array(xd, thd, *args, metrics_out=met2)
        assert torch.equal(met2, met)
        assert same_f32(heat_layout(heat), want_heat)


# ------------------------------------------------------------------------------------------------ u16 boundaries
def hot_case(T, C):
    """Every day hot: one run over the whole series, so every season's values are known exactly."""
    from hdp_b200 import _tables as tb
    x = np.ones((T, C), np.float32)
    thr = np.full((C, 365, 1), 0.5)
    dm = tb.doy_map(tb.TimeAxis.daily((1850, 1, 1), T, "noleap").dayofyr)
    return x, thr, dm


@pytest.mark.parametrize("days,bits", [(255, 8), (256, 16)])
def test_full_lane_and_lane_width_switch(core, lib, days, bits):
    # four definitions per register, two of them labelling the run and two never (min_duration beyond the series): a full 8-bit
    # lane of 255 must not carry into its neighbour, and one more day switches to 16-bit lanes
    T, C = 700, 37
    x, thr, dm = hot_case(T, C)
    defs = [[1, 0, 0], [8000, 0, 0], [3, 1, 1], [8000, 0, 0]]
    north, south = [[10, 10 + days], [300, 300 + days]], [[5, 5 + days], [400, 400 + days]]
    is_south = (np.arange(C) % 3 == 0).astype(np.uint8)
    assert metrics_choice(defs, north, south, T)[1][0] == bits
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        out = ref_layout(core.metrics_array(dev(x), dev(thr), dm, defs, north, south, is_south))
        assert np.array_equal(out, oracle.metrics_batch(x, thr, dm, defs, north, south, is_south))
        for d, hot in enumerate((True, False, True, False)):
            want = np.array([days, 1, days, days] if hot else [0, 0, 0, 0])
            assert (out[0, d] == want[:, None]).all(), (d, out[0, d, 0])


def test_longest_season_the_u16_output_holds(core, lib):
    # a 65 535-day season: HWF = HWD = HWA = 65535, HWN = 1; one day more does not fit: code -2 from the metrics, while the
    # intensity pass (float32) still takes it
    from hdp_b200 import _lib
    T, C = 180 * 365, 33
    x, thr, dm = hot_case(T, C)
    defs = [[3, 0, 0], [1, 1, 1]]
    is_south = (np.arange(C) % 2).astype(np.uint8)
    north, south = [[0, 65535]], [[100, 65635]]
    args = (dm, defs, north, south, is_south)
    out = ref_layout(core.metrics_array(dev(x), dev(thr), *args))
    assert (out == np.array([65535, 1, 65535, 65535])[:, None]).all()
    assert np.array_equal(out, oracle.metrics_batch(x, thr, *args))
    north = [[0, 65536]]
    args = (dm, defs, north, south, is_south)
    with pytest.raises(_lib.HdpB200Error) as e:
        core.metrics_array(dev(x), dev(thr), *args)
    assert e.value.code == -2
    heat = core.intensity_array(dev(x), dev(thr), *args)
    assert same_f32(heat_layout(heat), intensity_batch(x, thr, *args))


# ------------------------------------------------------------------------------------------------ thresholds without a day of year
def test_doy_free_thresholds_over_a_long_run(core):
    # the no-season and fixed-value variants (threshold tables of one row, doy_map = 0) over a CMIP-length run: its words must
    # still be 32 days long, else the word tables outgrow k_scan's and k_intensity's shared memory
    from hdp_b200 import _tables as tb, workloads
    rng = np.random.default_rng(31390)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1990-12-31", "noleap")
    run_ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
    C = 97
    season = lambda ax, warm: warm + 15 + 8 * np.sin(2 * np.pi * ax.dayofyr[:, None] / 365)     # noqa: E731
    xb = (season(base_ax, 0) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (season(run_ax, 1) + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    st = tb.hemisphere_ranges(run_ax)
    zeros = np.zeros(len(run_ax), np.int64)
    is_south = (np.arange(C) % 2).astype(np.uint8)
    args = (zeros, workloads.README_DEFS, st.north, st.south, is_south)
    thr_ns = core.thresholds_no_season_array(dev(xb), np.array([0.5, 0.9, 0.99]))
    for thr in (thr_ns, core.fixed_thresholds(C, 24.5)):
        th = thr.cpu().numpy()
        want, want_heat = oracle.metrics_batch(xr, th, *args), intensity_batch(xr, th, *args)
        assert np.array_equal(ref_layout(core.metrics_array(dev(xr), thr, *args)), want)
        met = torch.zeros((4, th.shape[2], len(workloads.README_DEFS), len(st.north), C), dtype=torch.uint16, device="cuda")
        assert same_f32(heat_layout(core.intensity_array(dev(xr), thr, *args, metrics_out=met)), want_heat)
        assert np.array_equal(ref_layout(met), want)
        assert np.array_equal(ref_layout(core.metrics_host(xr, th, *args)), want)
        met_h = np.zeros((4, th.shape[2], len(workloads.README_DEFS), len(st.north), C), np.uint16)
        assert same_f32(heat_layout(core.intensity_host(xr, th, *args, metrics_out=met_h)), want_heat)
        assert np.array_equal(ref_layout(met_h), want)
        hot = core.hot_days_array(dev(xr), thr, zeros).cpu().numpy()
        assert np.array_equal(hot, xr.astype(np.float64)[None] > th[:, 0, :].T[:, None, :])


# ------------------------------------------------------------------------------------------------ C. sample layouts
@pytest.fixture(params=["default", "cand", "seg_all", "seg_heavy", "ranked", "generic"])
def thr_path(request, lib):
    """Every threshold path (as in test_gpu_parity.py): k_thr_net where the tables allow, the segment kernels without it, k_thr_seg
    with and without its candidate filter, k_thr_ranked and the generic gather + sort."""
    lib.hdp_b200_thresholds_force_generic({"default": 0, "generic": 1, "ranked": 2, "seg_all": 3, "seg_heavy": 4, "cand": 5}[request.param])
    yield request.param
    lib.hdp_b200_thresholds_force_generic(0)


def view_of(kind, x):
    """A [T, C] float32 CUDA view with x's values in one of the layouts the array API accepts."""
    T, C = x.shape
    if kind == "cell_offset":                                   # cells 5 .. 5 + C of a wider array: ld_c = 1, ld_t > C, not 32-aligned
        big = torch.full((T, C + 40), float("nan"), device="cuda")
        big[:, 5:5 + C] = dev(x)
        v = big[:, 5:5 + C]
        assert v.stride() == (C + 40, 1)
    elif kind == "time_range":                                  # days 7 .. 7 + T of a time-contiguous array: ld_t = 1, ld_c > T
        big = torch.full((C, T + 30), float("nan"), device="cuda")
        big[:, 7:7 + T] = dev(x.T)
        v = big[:, 7:7 + T].t()
        assert v.stride() == (1, T + 30)
    else:                                                       # every other day and every third cell (k_gather_strided)
        big = torch.full((2 * T, 3 * C), float("nan"), device="cuda")
        big[::2, ::3] = dev(x)
        v = big[::2, ::3]
        assert v.stride() == (6 * C, 3)
    return v


def kelvin(x):
    """Kelvin samples and the Celsius values the kernels convert them to (the float32 arithmetic of hdp.measure)."""
    from hdp_b200 import measure as hm, xr
    xk = (x.astype(np.float64) + 273.15).astype(np.float32)
    da = xr.DataArray(xk, dims=["time", "cell"], coords={}, name="t", attrs={"units": "degK"})
    return xk, np.ascontiguousarray(xr.values_of(hm.kelvin_to_celsius(da)))


@pytest.mark.parametrize("kind", ["cell_offset", "time_range", "strided", "single_cell"])
def test_sample_layouts(core, lib, thr_path, kind):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(77)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1968-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C = 1 if kind == "single_cell" else 45
    season = lambda ax: 15 + 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)   # noqa: E731
    xb = (season(base_ax) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (season(run_ax) + 2 + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    xb[rng.integers(0, len(base_ax), 2), C - 1] = np.nan
    wt = tb.window_tables(base_ax.dayofyr, 7)
    q = np.array([0.9, 0.95])
    vkind = "cell_offset" if kind == "single_cell" else kind

    want = oracle.thresholds_batch(xb, wt.window_samples(), q)
    got = core.thresholds_array(view_of(vkind, xb), wt, q).cpu().numpy()
    assert bits_equal(got, want)
    if thr_path != "default":                                   # units on the paths that convert a (densified) copy first
        xk, xc = kelvin(xb)
        v = view_of(vkind, xk)
        got_k = core.thresholds_array(v, wt, q, units="degK").cpu().numpy()
        assert bits_equal(got_k, core.thresholds_array(v.contiguous(), wt, q, units="degK").cpu().numpy())
        assert bits_equal(got_k, oracle.thresholds_batch(xc, wt.window_samples(), q))
    if thr_path != "default":                                   # the metric pass does not depend on the threshold path
        return

    st = tb.hemisphere_ranges(run_ax)
    is_south = (np.arange(C) % 2).astype(np.uint8)
    args = (tb.doy_map(run_ax.dayofyr), [[3, 0, 0], [3, 1, 1], [5, 2, 1]], st.north, st.south, is_south)
    thr = np.nan_to_num(want, nan=1e9)
    v, thd = view_of(vkind, xr), dev(thr)
    want_met, want_heat = oracle.metrics_batch(xr, thr, *args), intensity_batch(xr, thr, *args)
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        met = core.metrics_array(v, thd, *args)
        assert torch.equal(met, core.metrics_array(v.contiguous(), thd, *args))
        assert np.array_equal(ref_layout(met), want_met)
    met2 = torch.zeros_like(met)
    heat = core.intensity_array(v, thd, *args, metrics_out=met2)
    assert torch.equal(heat, core.intensity_array(v.contiguous(), thd, *args))
    assert torch.equal(met2, met) and same_f32(heat_layout(heat), want_heat)
    hot = core.hot_days_array(v, thd, args[0])
    assert torch.equal(hot, core.hot_days_array(v.contiguous(), thd, args[0]))
    want_hot = np.stack([np.stack([oracle.indicate_hot_days(xr[:, c], thr[c, :, p], args[0]) for c in range(C)], axis=1)
                         for p in range(len(q))])
    assert np.array_equal(hot.cpu().numpy().astype(bool), want_hot)
    if kind == "single_cell":                                   # and a single day: one-day seasons of a one-day run
        day = v[40:41]
        one = (args[0][40:41], args[1], [[0, 1]], [[0, 1]], is_south)
        assert np.array_equal(ref_layout(core.metrics_array(day, thd, *one)), oracle.metrics_batch(xr[40:41], thr, *one))
        assert torch.equal(core.hot_days_array(day, thd, one[0]), core.hot_days_array(day.contiguous(), thd, one[0]))


@pytest.mark.parametrize("rank", range(3))
def test_run_sharded_rank_of_three(core, monkeypatch, rank):
    # the production slicing of shard.run_sharded (base_tc[:, c0:c1] / run_tc[:, c0:c1]: pitched views) with the CUDA kernels, as
    # rank `rank` of a world of 3 sees it, without a process group: the rank's shard against the oracle
    import torch.distributed as dist
    from hdp_b200 import _tables as tb, shard
    monkeypatch.setattr(dist, "is_available", lambda: True)
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 3)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: rank)
    rng = np.random.default_rng(3)
    base_ax = tb.TimeAxis.date_range("1961-01-01", "1970-12-31", "noleap")
    run_ax = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "noleap")
    C = 100                                                     # not a multiple of 3 x 32
    season = lambda ax: 15 + 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)   # noqa: E731
    xb = (season(base_ax) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (season(run_ax) + 2 + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    wt = tb.window_tables(base_ax.dayofyr, 7)
    q = np.array([0.9, 0.95, 0.99])
    st, dm = tb.hemisphere_ranges(run_ax), tb.doy_map(run_ax.dayofyr)
    south = (np.arange(C) % 3 == 0).astype(np.uint8)
    defs = [[3, 0, 0], [3, 1, 1], [4, 1, 1]]
    thr, met = shard.run_sharded(dev(xb), dev(xr), wt, q, dm, defs, st.north, st.south, dev(south), gather=False)
    c0, c1 = shard.cell_range(C, rank, 3)
    assert c1 > c0 and tuple(thr.shape) == (c1 - c0, 365, 3)
    want_thr = oracle.thresholds_batch(np.ascontiguousarray(xb[:, c0:c1]), wt.window_samples(), q)
    assert bits_equal(thr.cpu().numpy(), want_thr)
    want = oracle.metrics_batch(np.ascontiguousarray(xr[:, c0:c1]), want_thr, dm, defs, st.north, st.south, south[c0:c1])
    assert np.array_equal(ref_layout(met), want)
