"""Heatwave spatial extent (HWS) without a GPU: the oracle of tests/extent_oracle.py against a per-day restatement and, through the
contract's invariant, against the reference's HWF; the weight quantization and region handling of the metric layer; the C ABI's
argument checks; and the Dataset that compute_heatwave_extent assembles (with a stand-in for the device call).  The kernels
themselves are checked by tests/test_gpu_extent.py."""
import ctypes
import os
import re

import numpy as np
import pytest

import oracle
from extent_oracle import cold_extent_batch, extent_batch
from test_onset_host import DEFS, _measure_and_threshold, ar1, index_heatwaves_py

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORTH = [[100, 250], [465, 615], [830, 980]]
SOUTH = [[-5000, 40], [280, 430], [1010, 3000]]


def extent_restated(x, thr, dm, defs, north, south, is_south, w, r, R):
    """int64 [R, P, D, T] day by day: day t counts for cell c when it lies in one of the cell's season slices and its restated id is
    > 0."""
    T, C = x.shape
    P = thr.shape[2]
    out = np.zeros((R, P, len(defs), T), np.int64)
    for c in range(C):
        if not 0 <= r[c] < R:
            continue
        in_season = np.zeros(T, bool)
        for a, b in (south if is_south[c] else north):
            in_season[slice(int(a), int(b))] = True
        for p in range(P):
            with np.errstate(invalid="ignore"):
                hot = x[:, c].astype(np.float64) > thr[c, dm, p]
            for d, df in enumerate(defs):
                hw = index_heatwaves_py(hot, *df)
                for t in range(T):
                    if in_season[t] and hw[t] > 0:
                        out[r[c], p, d, t] += w[c]
    return out


def _case(seed=3, T=1100, C=11, P=2):
    x, thr, dm = ar1(seed, T, C, P)
    rng = np.random.default_rng(seed)
    is_south = (np.arange(C) % 3 == 1).astype(np.uint8)
    w = rng.integers(0, 1000, C).astype(np.uint32)
    r = rng.integers(-1, 4, C).astype(np.int32)
    return x, thr, dm, is_south, w, r


def test_oracle_matches_a_per_day_restatement():
    x, thr, dm, is_south, w, r = _case()
    got = extent_batch(x, thr, dm, DEFS, NORTH, SOUTH, is_south, w, r, 3)
    assert np.array_equal(got, extent_restated(x, thr, dm, DEFS, NORTH, SOUTH, is_south, w, r, 3))
    assert got.any()


@pytest.mark.parametrize("cold", [False, True])
def test_invariant_against_the_reference_hwf(cold):
    # sum_t ext[r, p, d, t] = sum_{c in r} w_c sum_y HWF[p, d, y, c]
    x, thr, dm, is_south, w, r = _case(seed=9)
    s = -1.0 if cold else 1.0
    ext = (cold_extent_batch if cold else extent_batch)(x, thr, dm, DEFS, NORTH, SOUTH, is_south, w, r, 4)
    ref = oracle.metrics_batch((s * x).astype(np.float32), s * thr, dm, DEFS, NORTH, SOUTH, is_south)      # [P, D, C, 4, Y]
    hwf = ref[:, :, :, 0, :].sum(axis=-1)                                                                 # [P, D, C]
    for reg in range(4):
        sel = r == reg
        assert np.array_equal(ext[reg].sum(axis=-1), (hwf[:, :, sel] * w[sel].astype(np.int64)).sum(axis=-1))
    # NULL weights and regions: one region, a cell count
    ones = extent_batch(x, thr, dm, DEFS[:2], NORTH, SOUTH, is_south) if not cold else None
    if ones is not None:
        assert np.array_equal(ones[0].sum(axis=-1), hwf[:, :2].sum(axis=-1))


def test_days_outside_every_season_and_runs_across_season_starts():
    T, C = 400, 2
    x = np.full((T, C), -1.0, np.float32)
    x[95:110, :] = 1.0                                          # a heatwave that begins before the season [100, 150)
    x[148:160, :] = 1.0                                         # and one that runs past its end
    x[300:320, :] = 1.0                                         # outside every season
    ext = extent_batch(x, np.zeros((C, 1, 1)), np.zeros(T, np.int64), [[3, 0, 0]], [[100, 150]], [[100, 150]], None)
    want = np.zeros(T, np.int64)
    want[100:110] = 2
    want[148:150] = 2
    assert np.array_equal(ext[0, 0, 0], want)


# ------------------------------------------------------------------------------------------------ weights and regions
def test_weight_quantization():
    from hdp_b200 import metric
    w = np.cos(np.deg2rad(np.linspace(-89.5, 89.5, 180)))
    q = metric.quantize_weights(w, np.zeros(180, np.int32), 1)
    assert q.dtype == np.uint32 and q.max() == 1 << 30 and int(q.astype(np.int64).sum()) < 1 << 53
    assert np.allclose(q / q.max(), w / w.max(), atol=2.0 ** -30)
    # zero weights stay zero; all-zero weights give all zeros
    w0 = w.copy()
    w0[::7] = 0.0
    assert (metric.quantize_weights(w0, np.zeros(180, np.int32), 1)[::7] == 0).all()
    assert (metric.quantize_weights(np.zeros(5), np.zeros(5, np.int32), 1) == 0).all()
    for bad in (np.array([1.0, -0.5]), np.array([1.0, np.nan]), np.array([1.0, np.inf])):
        with pytest.raises(ValueError):
            metric.quantize_weights(bad, np.zeros(2, np.int32), 1)
    # many cells: the largest weight is scaled below 2^30 so that every region's total stays below 2^53
    n = (1 << 24) + 5
    big = np.ones(n)
    qb = metric.quantize_weights(big, np.zeros(n, np.int32), 1)
    assert qb.max() < 1 << 30 and int(qb.astype(np.int64).sum()) < 1 << 53
    # cells in no region do not count towards any total
    qr = metric.quantize_weights(big, np.full(n, -1, np.int32), 1)
    assert qr.max() == 1 << 30


def test_share_and_regions():
    from hdp_b200 import metric
    wq = np.array([3, 5, 0, 7, 9], np.uint32)
    reg = np.array([0, 0, 1, -1, 5], np.int32)                 # region 1 has weight 0, cells 3 and 4 are in no region (R = 3)
    ext = np.zeros((3, 1, 1, 4), np.int64)
    ext[0, 0, 0] = [0, 3, 5, 8]
    share = metric.extent_share(ext, wq, reg, 3)
    assert np.array_equal(share[0, 0, 0], np.array([0, 3, 5, 8]) / 8.0)
    assert np.isnan(share[1]).all() and np.isnan(share[2]).all()


def test_core_extent_cells():
    from hdp_b200 import _core
    w, r, R = _core._extent_cells([1, 2, 3], [0, 7, -3], 2, 3)
    assert w.dtype == np.uint32 and r.dtype == np.int32 and R == 2 and r.tolist() == [0, -1, -1]
    assert _core._extent_cells(None, None, 1, 3) == (None, None, 1)
    for kw in (dict(weights=[1, -2, 3]), dict(weights=[1.5, 2, 3]), dict(weights=[1, 2]), dict(regions=[0.5, 1, 2]),
               dict(n_regions=0), dict(n_regions=257)):
        args = dict(weights=None, regions=None, n_regions=1)
        args.update(kw)
        with pytest.raises(ValueError):
            _core._extent_cells(args["weights"], args["regions"], args["n_regions"], 3)


# ------------------------------------------------------------------------------------------------ the C ABI (host logic)
def test_header_constants():
    from hdp_b200 import _core, _lib
    header = open(os.path.join(ROOT, "include", "hdp_b200.h")).read()
    assert int(re.search(r"#define HDP_B200_MAX_REGIONS\s+(\d+)", header).group(1)) == _core.MAX_REGIONS == 256
    assert int(re.search(r"#define HDP_B200_KERNEL_EXTENT\s+(\d+)", header).group(1)) == 15
    assert _core.KERNEL_NAMES[15] == "k_extent_prefix"
    assert _lib.lib().hdp_b200_abi_version() == 6


def test_argument_checks_before_any_device_work():
    from hdp_b200 import _lib
    L = _lib.lib()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)              # noqa: E731
    defs = np.array([[3, 0, 0]], np.int32)
    seas = np.zeros((1, 2), np.int32)
    tab = (p(defs), 1, p(seas), p(seas), 1, None)
    ext = np.zeros(64, np.int64)
    ws = np.zeros(1 << 16, np.uint8)
    dev = lambda R, e, unit: L.hdp_b200_extent(None, 0, 0, 1, 1, None, 1, 1, None, *tab, None, None, R, e, None, p(ws), ws.size, None,  # noqa: E731
                                              unit)
    assert dev(1, p(ext), 0x200) == -1                         # onset and extent are not combined
    assert dev(1, p(ext), 0x300) == -1
    assert dev(0, p(ext), 0) == -1 and dev(257, p(ext), 0) == -2
    assert L.hdp_b200_extent_workspace_bytes(10, 100, 10, 1, 365, 2, 3, 1, 0, None) == 0
    assert L.hdp_b200_extent_workspace_bytes(10, 100, 10, 1, 365, 2, 3, 1, 257, None) == 0
    small = L.hdp_b200_extent_workspace_bytes(10, 100, 10, 1, 365, 2, 3, 1, 1, None)
    assert L.hdp_b200_extent_workspace_bytes(10, 100, 10, 1, 365, 2, 3, 1, 4, None) - small >= 3 * 2 * 3 * 101 * 8
    x = np.zeros((4, 1), np.float32)
    dm = np.zeros(4, np.int32)
    host = lambda R, e, unit: L.hdp_b200_extent_host(p(x), 1, 4, 1, 1, None, None, 1, 1, p(dm), *tab, None, None, R, e, None, unit)  # noqa: E731
    assert host(1, p(ext), 0x200) == -1 and host(1, None, 0) == -1 and host(300, p(ext), 0) == -2


# ------------------------------------------------------------------------------------------------ the metric layer
@pytest.fixture
def fake_extent(monkeypatch):
    """_core.extent_host replaced by the oracle, which records its arguments."""
    from hdp_b200 import _core
    calls = []

    def extent_host(x, thr, dm, defs, north, south, is_south, weights=None, regions=None, n_regions=1, out=None, metrics_out=None,
                    units=None, *, cold=False):
        calls.append(dict(north=np.asarray(north), weights=weights, regions=regions, R=n_regions, cold=cold, is_south=is_south))
        fn = cold_extent_batch if cold else extent_batch
        return fn(x, thr, dm, defs, north, south, is_south, weights, regions, n_regions)
    monkeypatch.setattr(_core, "extent_host", extent_host)
    return calls


@pytest.mark.parametrize("cold", [False, True])
def test_metric_layer_dataset(fake_extent, cold):
    from hdp_b200 import _tables as tb, metric, utils, xr
    m, thr = _measure_and_threshold()
    levels = np.moveaxis(np.percentile(xr.values_of(m), [40, 60], axis=-1), 0, -1)[:, :, None, :]   # hot and cold days in every cell
    thr = xr.DataArray(np.zeros((2, 3, 365, 2)) + levels, dims=list(thr.dims),
                       coords=dict(xr.coords_of(thr)), attrs={"history": "made\n"})
    m.attrs["history"] = "measured\n"
    defs = [[3, 0, 0], [3, 1, 1]]
    ds = metric.compute_heatwave_extent(m, thr, defs, cold=cold, check_variables=False)
    name = "CSS" if cold else "HWS"
    assert list(ds.keys()) == [name]
    a = ds[name]
    T = len(utils.time_axis_of(m).year)
    assert tuple(a.dims) == ("region", "percentile", "definition", "time") and a.shape == (1, 2, 2, T)
    assert list(xr.coord_values(a, "region")) == ["all"] and list(xr.coord_values(a, "definition")) == ["3-0-0", "3-1-1"]
    assert np.array_equal(np.asarray(xr.coord_values(a, "time")), np.asarray(xr.coord_values(m, "time")))
    v = np.asarray(xr.values_of(a))
    assert v.dtype == np.float64 and (v >= 0).all() and (v <= 1).all() and v.any()
    assert a.attrs["long_name"] == ("Cold Spell Spatial Extent" if cold else "Heatwave Spatial Extent")
    assert "(Measure) measured" in a.attrs["history"] and "(Threshold) made" in a.attrs["history"]
    assert ds.attrs["hdp_type"] == "metric"
    st = tb.hemisphere_ranges(utils.time_axis_of(m))
    call = fake_extent[-1]
    assert call["cold"] == cold and np.array_equal(call["north"], st.south if cold else st.north)
    # default weights: cos(lat), quantized; the share is ext / total, with the same quantized weights
    lat = np.tile(np.asarray(xr.coord_values(m, "lat"), np.float64), 2)
    assert np.array_equal(call["weights"], metric.quantize_weights(np.cos(np.deg2rad(lat)), np.zeros(6), 1))
    x = np.ascontiguousarray(xr.values_of(m).reshape(6, -1).T)       # dims (lon, lat, time)
    raw = (cold_extent_batch if cold else extent_batch)(x, (np.zeros((2, 3, 365, 2)) + levels).reshape(6, 365, 2),
                                                         tb.doy_map(utils.time_axis_of(m).dayofyr), defs,
                                                         *((st.south, st.north) if cold else (st.north, st.south)), call["is_south"],
                                                         call["weights"], None, 1)
    assert np.array_equal(v, raw / float(call["weights"].astype(np.int64).sum()))


def test_metric_layer_regions(fake_extent):
    from hdp_b200 import metric, xr
    m, thr = _measure_and_threshold()
    reg = np.array([[0, 1, -1], [1, 0, 9]])                    # [lon, lat] like the measure's cell dims; 9: outside the 2 regions
    ds = metric.compute_heatwave_extent(m, thr, [[3, 0, 0]], weights=np.ones((2, 3)), regions=reg, region_names=["a", "b"],
                                        check_variables=False)
    call = fake_extent[-1]
    assert call["R"] == 2 and call["regions"].tolist() == [0, 1, -1, 1, 0, -1] and (call["weights"] == 1 << 30).all()
    assert list(xr.coord_values(ds["HWS"], "region")) == ["a", "b"]
    metric.compute_heatwave_extent(m, thr, [[3, 0, 0]], regions=reg, region_names=["a"], check_variables=False)
    assert fake_extent[-1]["R"] == 1 and fake_extent[-1]["regions"].tolist() == [0, -1, -1, -1, 0, -1]     # one name: one region
    metric.compute_heatwave_extent(m, thr, [[3, 0, 0]], regions=reg, check_variables=False)
    assert fake_extent[-1]["R"] == 10                                                                        # no names: 0 .. max
    with pytest.raises(ValueError, match="cell dims"):
        metric.compute_heatwave_extent(m, thr, [[3, 0, 0]], regions=np.zeros(5, int), check_variables=False)
    with pytest.raises(ValueError, match="negative"):
        metric.compute_heatwave_extent(m, thr, [[3, 0, 0]], weights=-np.ones((2, 3)), check_variables=False)
    with pytest.raises(AssertionError):
        metric.compute_heatwave_extent(m, thr, [[3, 0, 0]])
