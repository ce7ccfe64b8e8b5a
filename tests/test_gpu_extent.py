"""Heatwave spatial extent (hdp_b200_extent) on the device, bit for bit against tests/extent_oracle.py (the reference's
indicate_hot_days and index_heatwaves, then the weights of the cells on the days with an id > 0 of each season slice), and the
optional u16 output against hdp_b200_metrics: every k_scan instantiation with the run filter on and off, lane widths, both hemispheres
in a warp, padding lanes, season edges, definition and region counts, cold spells, accumulation over cell ranges, the host pipeline,
thresholds without a day-of-year axis, the metric layer and one full-size call."""
import ctypes

import numpy as np
import pytest

from extent_oracle import cold_extent_batch, extent_batch
from test_gpu_onset import ar1_case, designed_case, dev, host
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


def cells(rng, C, R):
    """Random u32 weights (some 0) and regions in -1 .. R (R and -1: in no region)."""
    w = rng.integers(0, 1 << 20, C).astype(np.uint32)
    w[rng.integers(0, C, 3)] = 0
    r = rng.integers(-1, R + 1, C).astype(np.int32)
    return w, r


def check(core, x, thr, args, w=None, r=None, R=1, cold=False, want=None):
    """extent_array on (x, thr) against the oracle (``want`` unless given) and its metrics_out against metrics_array; returns the
    extent (host)."""
    xd, thd = dev(x), dev(thr)
    met = torch.zeros((4, thr.shape[2], len(args[1]), len(args[2]), x.shape[1]), dtype=torch.uint16, device="cuda")
    got = core.extent_array(xd, thd, *args, weights=w, regions=r, n_regions=R, metrics_out=met, cold=cold)
    assert torch.equal(met, core.metrics_array(xd, thd, *args, cold=cold))
    assert torch.equal(got, core.extent_array(xd, thd, *args, weights=w, regions=r, n_regions=R, cold=cold))     # without metrics_out
    if want is None:
        want = (cold_extent_batch if cold else extent_batch)(x, thr, *args, w, r, R)
    assert np.array_equal(host(got), want)
    return host(got)


# ------------------------------------------------------------------------------------------------ every k_scan instantiation
@pytest.mark.parametrize("inst", scan_instances(), ids=lambda i: "b{}_ng{}_ks{}_f{}{}".format(*i))
def test_scan_instantiation(core, lib, inst):
    from hdp_b200 import _tables as tb
    defs, north, south = scan_case(*inst)
    rng = np.random.default_rng(sum(inst))
    C, P, R = 97, 2, 3                                         # C not a multiple of 32: padding lanes
    x, thr = ar1_case(rng, SCAN_T, C, P)
    dm = tb.doy_map(tb.TimeAxis.daily((2001, 1, 1), SCAN_T, "noleap").dayofyr)
    is_south = rng.integers(0, 2, C).astype(np.uint8)          # both hemispheres in every warp
    args = (dm, defs.tolist(), north, south, is_south)
    w, r = cells(rng, C, R)
    want = extent_batch(x, thr, *args, w, r, R)
    assert want.any()
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        rc, info = metrics_choice(defs, north, south)
        assert rc == 0 and tuple(info[:3]) == inst[:3] and (info[4], info[5]) == ((inst[3], inst[4]) if on else (0, 0))
        check(core, x, thr, args, w, r, R, want=want)


# ------------------------------------------------------------------------------------------------ season edges
# disjoint per hemisphere: starts and ends inside runs, one-day seasons, empty / reversed / negative / out-of-range entries, a season
# that runs to the end of the series (designed_case has a run on its last three days)
EDGE_NORTH = [[-5000, 2], [96, 100], [100, 150], [150, 151], [250, 250], [364, 366], [400, 398], [500, 505], [597, 5000]]
EDGE_SOUTH = [[0, 90], [99, 100], [100, 101], [240, 250], [250, 252], [505, 500], [-403, -300], [700, 700], [897, 2000]]


def test_season_edges(core, lib):
    x, thr = designed_case()
    T, C = x.shape
    is_south = (np.arange(C) % 3 == 1).astype(np.uint8)
    defs = [[1, 0, 0], [3, 0, 0], [2, 1, 1], [3, 2, 2], [5, 3, 0]]
    args = (np.zeros(T, np.int64), defs, EDGE_NORTH, EDGE_SOUTH, is_south)
    rng = np.random.default_rng(4)
    w, r = cells(rng, C, 2)
    want = extent_batch(x, thr, *args, w, r, 2)
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        check(core, x, thr, args, w, r, 2, want=want)
    got = check(core, x, thr, args)                            # every cell counts once
    assert got[..., T - 1].any()                               # a run still open at the end of the series
    assert got[..., 99].any() and got[..., 100].any()          # one-day seasons


def test_refusals(core):
    from hdp_b200 import _lib
    L = _lib.lib()
    x, thr = designed_case(C=33, T=400)
    T, C = x.shape
    xd, thd = dev(x), dev(thr)
    dm = np.zeros(T, np.int64)
    with pytest.raises(_lib.HdpB200Error, match="-2"):        # overlapping seasons could count a day twice
        core.extent_array(xd, thd, dm, [[3, 0, 0]], [[0, 100], [50, 150]], [[0, 10], [20, 30]])
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)            # noqa: E731
    defs, seas = np.array([[3, 0, 0]], np.int32), np.array([[0, T]], np.int32)
    dmi = np.zeros(T, np.int32)
    ext = torch.zeros((1, 1, 1, T), dtype=torch.int64, device="cuda")
    ws = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    call = lambda unit, R=1: L.hdp_b200_extent(xd.data_ptr(), C, T, C, 1, thd.data_ptr(), 1, 1, p(dmi), p(defs), 1, p(seas), p(seas), 1,  # noqa: E731
                                               None, None, None, R, ext.data_ptr(), None, ws.data_ptr(), ws.numel(), s, unit)
    assert call(0x200) == -1 and call(0x300) == -1 and call(0, 0) == -1 and call(0, 257) == -2
    assert L.hdp_b200_extent(xd.data_ptr(), C, T, C, 1, thd.data_ptr(), 1, 1, p(dmi), p(defs), 1, p(seas), p(seas), 1, None, None, None, 1,
                             ext.data_ptr(), None, ws.data_ptr(), 100, s, 0) == -3
    torch.cuda.synchronize()
    assert not ext.any()                                       # nothing written by a refused call
    assert call(0) == 0 and ext.sum() > 0


@pytest.mark.parametrize("D,R", [(1, 1), (32, 3), (5, 256)])
def test_definition_and_region_counts(core, lib, D, R):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(D + R)
    ax = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "noleap")
    C, P = 301, 2
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    defs = [[3, 1, 1]] if D == 1 else [[int(rng.integers(1, 6)), int(rng.integers(0, 4)), int(rng.integers(0, 4))] for _ in range(D)]
    args = (tb.doy_map(ax.dayofyr), defs, st.north, st.south, (np.arange(C) % 2).astype(np.uint8))
    w, r = cells(rng, C, R)
    for on in (1, 0):
        lib.hdp_b200_metrics_run_filter(on)
        check(core, x, thr, args, w, r, R)
    # NULL weights and regions: a cell count of region 0
    got = check(core, x, thr, args)
    met = core.metrics_array(dev(x), dev(thr), *args)
    assert np.array_equal(got.sum(axis=-1)[0], host(met[0]).astype(np.int64).sum(axis=(2, 3)))


def test_cold_is_warm_on_negated_inputs(core):
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(8)
    ax = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "noleap")
    C, P = 70, 2
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    args = (tb.doy_map(ax.dayofyr), [[3, 0, 0], [3, 1, 1], [2, 2, 3]], st.south, st.north, (np.arange(C) % 2).astype(np.uint8))
    w, r = cells(rng, C, 2)
    got = check(core, x, thr, args, w, r, 2, cold=True)
    warm = core.extent_array(dev(-x), dev(-thr), *args, weights=w, regions=r, n_regions=2)
    assert np.array_equal(got, host(warm)) and got.any()


def test_accumulation_over_cell_ranges(core):
    # three uneven, not 32-aligned cell ranges added into one output equal the whole call
    from hdp_b200 import _tables as tb
    rng = np.random.default_rng(17)
    ax = tb.TimeAxis.date_range("2001-01-01", "2004-12-31", "noleap")
    C, P, R = 250, 3, 4
    x, thr = ar1_case(rng, len(ax), C, P)
    st = tb.hemisphere_ranges(ax)
    south = (rng.random(C) < 0.5).astype(np.uint8)
    defs = [[3, 0, 0], [3, 1, 1], [4, 2, 1]]
    dm = tb.doy_map(ax.dayofyr)
    w, r = cells(rng, C, R)
    xd, thd = dev(x), dev(thr)
    whole = core.extent_array(xd, thd, dm, defs, st.north, st.south, south, weights=w, regions=r, n_regions=R)
    acc = torch.zeros_like(whole)
    for a, b in ((0, 45), (45, 190), (190, C)):
        core.extent_array(xd[:, a:b], thd[a:b].contiguous(), dm, defs, st.north, st.south, south[a:b], weights=w[a:b], regions=r[a:b],
                          n_regions=R, out=acc)
    assert torch.equal(acc, whole) and whole.any()


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
    C, R = 299, 3
    cyc = lambda ax: 15 + 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)            # noqa: E731
    xb = (cyc(base_ax) + 3 * rng.standard_normal((len(base_ax), C))).astype(np.float32)
    xr = (cyc(run_ax) + 1 + 3 * rng.standard_normal((len(run_ax), C))).astype(np.float32)
    q = np.array([0.9, 0.95, 0.99])
    thr_d = core.thresholds_array(dev(xb), wt, q)
    thr_h = thr_d.cpu().numpy()
    thr_k = core.thresholds_host(xb, wt, q, keep=True)                                            # remembered resident copy
    assert core.resident_thresholds(thr_k) is not None
    st = tb.hemisphere_ranges(run_ax)
    args = (tb.doy_map(run_ax.dayofyr), [[3, 0, 0], [3, 1, 1], [4, 2, 1]], st.north, st.south, (rng.random(C) < 0.5).astype(np.uint8))
    w, r = cells(rng, C, R)
    want = check(core, xr, thr_h, args, w, r, R)
    want_met = host(core.metrics_array(dev(xr), dev(thr_h), *args))
    pinned = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()             # noqa: E731
    for X, TH in ((xr, thr_h), (pinned(xr), thr_h), (xr, pinned(thr_h)), (xr, thr_d), (np.ascontiguousarray(xr.T).T, thr_k)):
        assert np.array_equal(core.extent_host(X, TH, *args, weights=w, regions=r, n_regions=R), want)
        met_h = np.zeros_like(want_met)
        out = np.full_like(want, 7)                                                                # overwritten, not added to
        core.extent_host(X, TH, *args, weights=w, regions=r, n_regions=R, out=out, metrics_out=met_h)
        assert np.array_equal(out, want) and np.array_equal(met_h, want_met)
    out = pinned(np.zeros_like(want))
    core.extent_host(xr, thr_h, *args, weights=pinned(w), regions=pinned(r), n_regions=R, out=out)
    assert np.array_equal(out, want)
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
    w, r = cells(rng, C, 2)
    got = check(core, xr, np.full((C, 1, 2), 0.0) + np.array([21.0, 24.5]), args, w, r, 2)
    assert got.any()


# ------------------------------------------------------------------------------------------------ the metric layer
def test_compute_heatwave_extent(core):
    from hdp_b200 import _tables as tb, measure, metric, threshold, utils, xr
    from conftest import bits_equal
    grid = (2, 3)
    test = utils.generate_test_warming_dataarray(grid_shape=grid, add_noise=True)
    rh = utils.generate_test_rh_dataarray(grid_shape=grid)
    measures = measure.format_standard_measures([test], rh=rh)
    name = list(measures.keys())[0]
    m = measures[name]
    thresholds = threshold.compute_thresholds(measures, np.array([0.9, 0.95]))
    t = thresholds[f"{name}_threshold"]
    defs = [[3, 0, 0], [3, 1, 1], [4, 1, 1]]
    t_axis = utils.time_axis_of(m)
    st = tb.hemisphere_ranges(t_axis)
    lat = np.tile(np.asarray(xr.coord_values(m, "lat"), np.float64), 2)
    south = tb.is_south(lat)
    x = np.ascontiguousarray(xr.values_of(m).reshape(6, -1).T)
    th = np.ascontiguousarray(xr.values_of(t).reshape(6, 365, 2))
    dm = tb.doy_map(t_axis.dayofyr)
    for cold in (False, True):
        ds = metric.compute_heatwave_extent(m, t, defs, cold=cold)
        v = np.asarray(xr.values_of(ds["CSS" if cold else "HWS"]))
        wq = metric.quantize_weights(np.cos(np.deg2rad(lat)), np.zeros(6), 1)
        seas = (st.south, st.north) if cold else (st.north, st.south)
        raw = (cold_extent_batch if cold else extent_batch)(x, th, dm, defs, *seas, south, wq, None, 1)
        assert bits_equal(v, raw / float(wq.astype(np.int64).sum()))
        assert v.shape == (1, 2, 3, x.shape[0]) and (v >= 0).all() and (v <= 1).all()
        # regions: each region's share from its own cells
        reg = np.array([[0, 1, -1], [1, 0, 1]])
        dr = metric.compute_heatwave_extent(m, t, defs, cold=cold, weights=np.ones(grid), regions=reg, region_names=["a", "b"])
        vr = np.asarray(xr.values_of(dr["CSS" if cold else "HWS"]))
        rr = reg.reshape(-1)
        raw_r = (cold_extent_batch if cold else extent_batch)(x, th, dm, defs, *seas, south, np.full(6, 1 << 30), rr, 2)
        assert bits_equal(vr, raw_r / (np.bincount(rr[rr >= 0], minlength=2) * float(1 << 30))[:, None, None, None])
    assert v.any() or vr.any()
    core.host_release()


# ------------------------------------------------------------------------------------------------ one full-size call
def test_cmip6_full_size(core):
    # cmip6_1deg (64 800 cells, 31 390 days, P 10, the README definitions): the invariant against the call's own HWF on all cells,
    # and the oracle on a sample of cells as region 0 with every other cell in no region
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
    wts = np.random.default_rng(1).integers(0, 1 << 30, C).astype(np.uint32)
    met = torch.zeros((4, P, len(w.defs), len(st.north), C), dtype=torch.uint16, device="cuda")
    ext = core.extent_array(x, thr, *args, weights=wts, metrics_out=met)
    assert torch.equal(met, core.metrics_array(x, thr, *args))
    hwf = met[0].to(torch.int64).sum(dim=2)                                                        # [P, D, C]
    assert torch.equal(ext[0].sum(dim=-1), (hwf * torch.as_tensor(wts.astype(np.int64), device="cuda")).sum(dim=-1))
    sample = np.sort(np.random.default_rng(0).choice(C, 24, replace=False))
    reg = np.full(C, -1, np.int32)
    reg[sample] = 0
    sub = host(core.extent_array(x, thr, *args, weights=wts, regions=reg))
    sel = torch.as_tensor(sample, device="cuda")
    assert np.array_equal(sub, extent_batch(host(x[:, sel]), host(thr[sel]), *args[:4], is_south[sample], wts[sample], None, 1))
    assert sub.any()
