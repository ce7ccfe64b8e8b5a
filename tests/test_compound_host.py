"""Compound heatwaves without a GPU: the masked-input oracle construction the GPU tests check against (compound metrics at percentile
p = single-measure metrics of where(M_p, x_a, NaN)), the host-side plan of k_hot_pair, the workspace sizes of hdp_b200_compound and
the argument checks of metric.compute_compound_metrics.  The kernels themselves are checked by tests/test_gpu_compound.py."""
import numpy as np
import pytest

import oracle
from intensity_oracle import intensity_batch


def compound_mask(xa, ta, xb, tb, dm, cold=False):
    """bool [P, T, C]: both measures beyond their thresholds (float64 comparisons; NaN on any side: False)."""
    xa, xb = np.asarray(xa, np.float64), np.asarray(xb, np.float64)
    ta_t, tb_t = np.asarray(ta)[:, dm, :].transpose(2, 1, 0), np.asarray(tb)[:, dm, :].transpose(2, 1, 0)     # [P, T, C]
    with np.errstate(invalid="ignore"):
        if cold:
            return (xa[None] < ta_t) & (xb[None] < tb_t)
        return (xa[None] > ta_t) & (xb[None] > tb_t)


def compound_oracle(xa, ta, xb, tb, dm, defs, north, south, is_south, intensity=True, cold=False):
    """(int64 [P, D, C, 4, Y], float32 [2, P, D, C, 3, Y] or None) by the masked-input construction, one percentile at a time; the
    cold direction through the heatwave oracles on negated inputs."""
    M = compound_mask(xa, ta, xb, tb, dm, cold)
    s = -1.0 if cold else 1.0
    met, heat = [], []
    for p in range(M.shape[0]):
        ma = np.where(M[p], s * np.asarray(xa, np.float32), np.float32(np.nan)).astype(np.float32)
        mb = np.where(M[p], s * np.asarray(xb, np.float32), np.float32(np.nan)).astype(np.float32)
        tpa, tpb = s * np.asarray(ta)[:, :, p:p + 1], s * np.asarray(tb)[:, :, p:p + 1]
        met.append(oracle.metrics_batch(ma, tpa, dm, defs, north, south, is_south)[0])
        if intensity:
            heat.append(np.stack([intensity_batch(ma, tpa, dm, defs, north, south, is_south)[0],
                                  intensity_batch(mb, tpb, dm, defs, north, south, is_south)[0]]))
    return np.stack(met), (np.stack(heat, axis=1) if intensity else None)


def small_case(seed=3, T=3 * 365, C=9, n_doy=365, P=3):
    rng = np.random.default_rng(seed)
    dm = np.arange(T) % n_doy
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.6 * z[t - 1] + 0.8 * z[t]
    xa = (20 + 3 * z).astype(np.float32)
    xb = (12 + 3 * (0.7 * z + 0.7 * rng.standard_normal((T, C)))).astype(np.float32)
    ta = 20 + np.linspace(1, 4, P)[None, None, :] + 0.3 * rng.standard_normal((C, n_doy, 1))
    tb = 12 + np.linspace(1, 4, P)[None, None, :] + 0.3 * rng.standard_normal((C, n_doy, 1))
    north = np.array([[0, 365], [365, 730], [730, T]])
    south = np.array([[100, 400], [500, 800], [900, 1000]])
    return xa, ta, xb, tb, dm, [[3, 0, 0], [3, 1, 1], [1, 0, 0], [4, 2, 2]], north, south, (np.arange(C) % 2).astype(np.uint8)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------ the oracle construction
@pytest.mark.parametrize("cold", [False, True])
def test_oracle_same_measure_is_single(cold):
    xa, ta, _, _, dm, defs, north, south, is_south = small_case()
    met, heat = compound_oracle(xa, ta, xa, ta, dm, defs, north, south, is_south, cold=cold)
    s = -1.0 if cold else 1.0
    want = oracle.metrics_batch((s * xa).astype(np.float32), s * ta, dm, defs, north, south, is_south)
    assert np.array_equal(met, want) and want[:, :, :, 0].max() > 0
    want_h = intensity_batch((s * xa).astype(np.float32), s * ta, dm, defs, north, south, is_south)
    assert np.array_equal(bits(heat[0]), bits(want_h)) and np.array_equal(bits(heat[1]), bits(want_h))


def test_oracle_open_second_threshold_is_first_measure_alone():
    xa, ta, xb, _, dm, defs, north, south, is_south = small_case(5)
    met, heat = compound_oracle(xa, ta, xb, np.full_like(ta, -np.inf), dm, defs, north, south, is_south)
    assert np.array_equal(met, oracle.metrics_batch(xa, ta, dm, defs, north, south, is_south))
    assert np.array_equal(bits(heat[0]), bits(intensity_batch(xa, ta, dm, defs, north, south, is_south)))
    assert (heat[1][..., 0, :] > 0).sum() == (heat[0][..., 0, :] > 0).sum()          # B's exceedance over -inf is inf on those days
    assert np.isinf(heat[1][heat[0] > 0]).all()


def test_oracle_nan_second_measure_is_zero():
    xa, ta, xb, tb, dm, defs, north, south, is_south = small_case(7)
    met, heat = compound_oracle(xa, ta, np.full_like(xb, np.nan), tb, dm, defs, north, south, is_south)
    assert (met == 0).all() and (heat == 0).all()


def test_oracle_compound_is_below_each_measure():
    xa, ta, xb, tb, dm, defs, north, south, is_south = small_case(9)
    met, _ = compound_oracle(xa, ta, xb, tb, dm, defs, north, south, is_south, intensity=False)
    hwf = met[..., 0, :]
    assert hwf.max() > 0
    assert (hwf <= oracle.metrics_batch(xa, ta, dm, defs, north, south, is_south)[..., 0, :]).all()
    assert (hwf <= oracle.metrics_batch(xb, tb, dm, defs, north, south, is_south)[..., 0, :]).all()


# ------------------------------------------------------------------------------------------------ the C ABI (host logic)
@pytest.fixture(scope="module")
def L():
    from hdp_b200 import _lib
    return _lib.lib()


def plan(L, P):
    import ctypes
    info = (ctypes.c_int * 3)()
    rc = L.hdp_b200_compound_plan(P, info)
    return rc, tuple(info)


def test_plan_reaches_every_group_size_and_slices(L):
    seen = {}
    for P in range(1, 33):
        rc, (pg, slices, smem) = plan(L, P)
        assert rc == 0
        ppad = -(-P // pg) * pg
        gps = -(-(ppad // pg) // slices)
        assert smem == gps * 2 * 32 * pg * 33 * 4 <= 227 * 1024
        assert slices * gps * pg >= P
        seen.setdefault(pg, []).append((P, slices))
    assert sorted(seen) == [4, 8, 10, 16, 20]
    for P, pg in ((4, 4), (8, 8), (10, 10), (16, 16), (20, 20)):
        assert plan(L, P)[1][0] == pg
    assert plan(L, 10)[1] == (10, 1, 84480)                         # the README percentile set: two CTAs per SM
    assert plan(L, 20)[1] == (20, 1, 168960)
    assert plan(L, 32)[1] == (16, 2, 135168)                        # both tiles of 32 percentiles do not fit one CTA
    assert plan(L, 0)[0] == -1 and plan(L, 33)[0] == -2


def test_workspace_sizes(L):
    ws = lambda C, lca=1, lcb=1, T=31390, n_doy=365, P=10, Y=86: L.hdp_b200_compound_workspace_bytes(C, T, lca, lcb, n_doy, P, 6, Y, None)  # noqa: E731
    sizes = [ws(C) for C in (1, 64, 128, 4096, 64800)]
    assert all(s > 0 for s in sizes) and sizes == sorted(sizes) and len(set(sizes)) == len(sizes)
    C, T = 64, 31390 + 2                                             # C * T * 4 a multiple of the workspace alignment
    assert (C * T * 4) % 256 == 0
    base = ws(C, T=T)
    assert ws(C, T, 1, T=T) == base + C * T * 4 and ws(C, 1, T, T=T) == base + C * T * 4
    assert ws(C, T, T, T=T) == base + 2 * C * T * 4
    assert base >= L.hdp_b200_intensity_workspace_bytes(C, T, C, 1, 365, 10, 6, 86, None)
    for bad in (dict(C=-1), dict(C=8, T=-1), dict(C=8, n_doy=0), dict(C=8, P=0), dict(C=8, Y=-1)):
        assert ws(**bad) == 0
    # n_doy = 1: both thresholds are replicated to 32 rows
    assert ws(C, n_doy=1) == L.hdp_b200_intensity_workspace_bytes(C, 31390, C, 1, 1, 10, 6, 86, None) + 256 * -(-(C * 32 * 10 * 8) // 256)


def test_entry_points_check_their_arguments(L):
    import ctypes
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)                 # noqa: E731
    defs = np.array([[3, 0, 0]], np.int32)
    seas = np.zeros((1, 2), np.int32)
    ws = np.zeros(1 << 20, np.uint8)
    # an empty run (C = 0) gets as far as the argument checks and returns before it touches a device
    for unit in (0, 1, 2, 0x100, 0x102):
        assert L.hdp_b200_compound(None, 1, 1, None, 1, 1, 0, 0, None, None, 1, 1, None, p(defs), 1, p(seas), p(seas), 1, None, None, None,
                                   p(ws), ws.size, None, unit) == 0
    # neither output, or no second measure
    x = np.zeros((4, 1), np.float32)
    assert L.hdp_b200_compound(p(x), 1, 1, None, 1, 1, 1, 4, None, None, 1, 1, None, p(defs), 1, p(seas), p(seas), 1, None, None, None,
                               p(ws), ws.size, None, 0) == -1
    assert L.hdp_b200_compound_host(p(x), 1, 1, None, 1, 1, 1, 4, None, None, None, None, 1, 1, None, p(defs), 1, p(seas), p(seas), 1,
                                    None, None, None, 0) == -1


# ------------------------------------------------------------------------------------------------ the metric layer
def _pair(n_years=4, lat=(-10.0, 20.0, 35.0)):
    from hdp_b200 import utils, xr
    m = utils.generate_test_warming_dataarray("2000-01-01", f"{1999 + n_years}-12-31", grid_shape=(2, len(lat))).astype(np.float32)
    lon = xr.coord_values(m, "lon")

    def thr(name, percentiles=(0.9, 0.95), n_doy=365):
        return xr.DataArray(np.zeros((2, len(lat), n_doy, len(percentiles))), dims=["lon", "lat", "doy", "percentile"],
                            coords={"lon": lon, "lat": xr.coord_values(m, "lat"), "doy": np.arange(1, n_doy + 1),
                                    "percentile": np.array(percentiles)}, name=name, attrs={})
    return m, thr


def test_metric_layer_rejects_mismatched_inputs():
    from hdp_b200 import metric, utils, xr
    m, thr = _pair()
    defs = [[3, 0, 0]]
    with pytest.raises(ValueError, match="percentile"):
        metric.compute_compound_metrics(m, thr("a"), m, thr("b", (0.9, 0.99)), defs, check_variables=False)
    with pytest.raises(ValueError, match="percentile"):
        metric.compute_compound_metrics(m, thr("a"), m, thr("b", (0.9,)), defs, check_variables=False)
    with pytest.raises(ValueError, match="days of year"):
        metric.compute_compound_metrics(m, thr("a"), m, thr("b", n_doy=366), defs, check_variables=False)
    other = utils.generate_test_warming_dataarray("2001-01-01", "2004-12-31", grid_shape=(2, 3)).astype(np.float32)
    with pytest.raises(ValueError, match="time axis"):
        metric.compute_compound_metrics(m, thr("a"), other, thr("b"), defs, check_variables=False)
    shifted = xr.DataArray(xr.values_of(m), dims=list(m.dims), coords={**dict(xr.coords_of(m)), "lon": xr.coord_values(m, "lon") + 1.0},
                           name="tmin", attrs=dict(m.attrs))
    with pytest.raises(ValueError, match="lon"):
        metric.compute_compound_metrics(m, thr("a"), shifted, thr("b"), defs, check_variables=False)
    small = utils.generate_test_warming_dataarray("2000-01-01", "2003-12-31", grid_shape=(2, 2)).astype(np.float32)
    with pytest.raises(ValueError):
        metric.compute_compound_metrics(m, thr("a"), small, thr("b"), defs, check_variables=False)


@pytest.fixture
def fake_compound(monkeypatch):
    """_core.compound_metrics_host / compound_intensity_host replaced by recorders that fill every metric plane i with i + 1 and
    intensity block b, plane i with 10 b + i + 0.5: the metric layer can then be checked without a device."""
    from hdp_b200 import _core
    calls = []

    def metrics_host(xa, ta, xb, tb, dm, defs, north, south, is_south, out=None, units=None, *, cold=False):
        calls.append(dict(north=np.asarray(north), south=np.asarray(south), cold=cold, shapes=(xa.shape, xb.shape, ta.shape, tb.shape)))
        P, D, Y, C = ta.shape[2], len(defs), len(north), xa.shape[1]
        return np.broadcast_to(np.arange(1, 5, dtype=np.uint16)[:, None, None, None, None], (4, P, D, Y, C)).copy()

    def intensity_host(xa, ta, xb, tb, dm, defs, north, south, is_south, out=None, metrics_out=None, units=None, *, cold=False):
        met = metrics_host(xa, ta, xb, tb, dm, defs, north, south, is_south, cold=cold)
        metrics_out[...] = met
        v = (10 * np.arange(2)[:, None] + np.arange(3)[None, :] + 0.5).astype(np.float32)
        return np.broadcast_to(v[:, :, None, None, None, None], (2, 3) + met.shape[1:]).copy()
    monkeypatch.setattr(_core, "compound_metrics_host", metrics_host)
    monkeypatch.setattr(_core, "compound_intensity_host", intensity_host)
    return calls


@pytest.mark.parametrize("cold", [False, True])
def test_metric_layer_variables(fake_compound, cold):
    from hdp_b200 import _tables as tb, metric, utils, xr
    m, thr = _pair()
    mb = xr.DataArray(xr.values_of(m), dims=list(m.dims), coords=dict(xr.coords_of(m)), name="tmin", attrs=dict(m.attrs))
    ma = xr.DataArray(xr.values_of(m), dims=list(m.dims), coords=dict(xr.coords_of(m)), name="tmax", attrs=dict(m.attrs))
    defs = [[3, 0, 0], [3, 1, 1]]
    ds = metric.compute_compound_metrics(ma, thr("a"), mb, thr("b"), defs, check_variables=False, intensity=True, cold=cold)
    st = tb.hemisphere_ranges(utils.time_axis_of(m))
    c = fake_compound[-1]
    assert c["cold"] == cold
    north, south = (st.south, st.north) if cold else (st.north, st.south)
    assert np.array_equal(c["north"], north) and np.array_equal(c["south"], south)
    assert ds.attrs["compound_measures"] == "tmax & tmin"
    metric_names = ["CSF", "CSN", "CSD", "CSA"] if cold else ["HWF", "HWN", "HWD", "HWA"]
    int_names = ["CSC", "CSI", "CSP"] if cold else ["HWC", "HWI", "HWP"]
    assert sorted(ds.keys()) == sorted(metric_names + int_names)
    for i, n in enumerate(metric_names):
        a = ds[n]
        assert tuple(a.dims) == ("percentile", "definition", "lon", "lat", "time")
        assert (np.asarray(xr.values_of(a)) == i + 1).all()
        assert a.attrs["long_name"].startswith("Compound ") and "tmax" in a.attrs["description"] and "tmin" in a.attrs["description"]
    assert ds[metric_names[0]].attrs["long_name"] == ("Compound Cold Spell Frequency" if cold else "Compound Heatwave Frequency")
    for i, n in enumerate(int_names):
        a = ds[n]
        assert tuple(a.dims) == ("measure", "percentile", "definition", "lon", "lat", "time")
        assert list(xr.coord_values(a, "measure")) == ["tmax", "tmin"]
        v = np.asarray(xr.values_of(a))
        assert (v[0] == i + 0.5).all() and (v[1] == 10 + i + 0.5).all()
        assert a.attrs["long_name"].startswith("Compound ")
    assert list(xr.coord_values(ds[metric_names[0]], "percentile")) == [0.9, 0.95]
    ds2 = metric.compute_compound_metrics(ma, thr("a"), mb, thr("b"), defs, check_variables=False, cold=cold)
    assert sorted(ds2.keys()) == sorted(metric_names)
