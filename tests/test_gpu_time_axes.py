"""Both paths on time axes that are not whole continuous years (tests/time_axes.py), bit for bit against the oracles.

Path 1: baselines that start mid-year (rows in first-appearance order, -1 pads in many rows, NY = 30 and 32), that miss days (pads in
arbitrary rows, the wrap rows of the window short) and May - September subsets (153 / 154 rows), on every threshold path.
Path 2: run axes of the same kinds cut the series into many short hot-day words, blocks without words, k_scan's run filter looking
across short neighbouring words, seasons of about 520 days (16-bit accumulator lanes); then the limits of the word tables (k_scan,
k_intensity, k_unpack_mask), the workspace bound of a NULL day-of-year map, and day-of-year maps that reach past the threshold table."""
import ctypes

import numpy as np
import pytest

import intensity_oracle
import onset_oracle
import oracle
import time_axes as ta
from conftest import bits_equal
from test_compound_host import compound_mask, compound_oracle

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


def ref_layout(out_u16):
    """uint16 [4, P, D, Y, C] -> the reference's int64 [P, D, C, 4, Y]."""
    return np.asarray(out_u16.cpu().numpy() if isinstance(out_u16, torch.Tensor) else out_u16).astype(np.int64).transpose(1, 2, 4, 0, 3)


def heat_layout(heat):
    """float32 [3, P, D, Y, C] -> the oracle's [P, D, C, 3, Y]."""
    return np.asarray(heat.cpu().numpy() if isinstance(heat, torch.Tensor) else heat).transpose(1, 2, 4, 0, 3)


def same_f32(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


AXES = {
    "mid_noleap": lambda: ta.mid("noleap"),
    "mid_standard": lambda: ta.mid("standard"),
    "gappy_noleap": lambda: ta.gappy("noleap"),
    "gappy_standard": lambda: ta.gappy("standard"),
    "summer_noleap": lambda: ta.summer("noleap"),
    "summer_standard": lambda: ta.summer("standard"),
}
_cache = {}


def cached(key, fn):
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


# ------------------------------------------------------------------------------------------ path 1
@pytest.fixture(params=["default", "cand", "seg_all", "seg_heavy", "ranked", "generic", "net_smem"])
def thr_path(request, core):
    """Every threshold path: the default (k_thr_net where the tables and quantiles allow, else the segment kernels), the segment
    kernels without k_thr_net (k_thr_cand + k_thr_seg), k_thr_seg with and without its candidate filter, k_thr_ranked, the generic
    gather+sort fallback, and k_thr_net with every list in shared memory (no tensor-memory variant)."""
    from hdp_b200 import _lib
    code = {"default": 0, "generic": 1, "ranked": 2, "seg_all": 3, "seg_heavy": 4, "cand": 5, "net_smem": 6}[request.param]
    _lib.lib().hdp_b200_thresholds_force_generic(code)
    yield request.param
    _lib.lib().hdp_b200_thresholds_force_generic(0)


QSETS = {
    "high": np.arange(0.9, 1.0, 0.01),                       # the README sweep
    "low": np.arange(1, 11) / 100.0,                         # the cold-spell sweep
    "ends": np.array([0.0, 0.5, 1.0]),
}


def _baseline(name, C=203):
    ax = AXES[name]()
    rng = np.random.default_rng(len(name) * 13 + C)
    T = len(ax)
    doy = ax.dayofyr[:, None]
    x = (15 + 12 * np.sin(2 * np.pi * (doy - 110) / 365) + 3 * rng.standard_normal((T, C))).astype(np.float32)
    x[T - 1, 0] = np.nan                                     # the sample every -1 pad reads
    x[rng.integers(0, T, 3), 1] = np.inf
    x[rng.integers(0, T, 3), 2] = -np.inf
    x[:, 3] = np.round(x[:, 3])                              # heavy ties
    x[:, 4] = 2.5                                            # constant
    x[:, 5] = np.where(rng.random(T) < 0.3, 99.0, x[:, 5])   # ties inside the top
    x[rng.integers(0, T, 3), 6] = np.nan
    x[:, 7] = np.arange(T, dtype=np.float32) * np.float32(1e-3)      # a trend: the last rows hold every window's top
    return ax, x


def _net_launches(core, fn):
    """Runs fn() and returns the names of the kernels it launched."""
    core.timing_enable(True)
    core.timing_read()
    try:
        fn()
    finally:
        names = [n for n, _ in core.timing_read()]
        core.timing_enable(False)
    return names


@pytest.mark.parametrize("qset", sorted(QSETS))
@pytest.mark.parametrize("name", sorted(AXES))
def test_thresholds(core, thr_path, name, qset):
    from hdp_b200 import _tables as tb
    ax, x = cached(("base", name), lambda: _baseline(name))
    wt = tb.window_tables(ax.dayofyr, 7)
    q = QSETS[qset]
    want = cached(("thr", name, qset), lambda: oracle.thresholds_batch(x, wt.window_samples(), q))
    if qset == "high" and thr_path in ("default", "net_smem"):
        # the high quantiles of every one of these tables run on the lane-per-cell network kernel
        assert "k_thr_net" in _net_launches(core, lambda: core.thresholds_array(dev(x), wt, q))
    got = core.thresholds_array(dev(x), wt, q).cpu().numpy()
    assert bits_equal(got, want)
    # the NaN on the last sample: NaN in exactly the windows that hold a -1 pad or the last sample itself
    ws = wt.window_samples()
    holds = ((ws < 0) | (ws == len(ax) - 1)).any(1)
    assert np.array_equal(np.isnan(got[0]).all(1), holds) and not np.isnan(got[0][~holds]).any()
    if name != "summer_noleap":
        assert (ws < 0).any()                                # the table has pads for the NaN to reach
    if thr_path == "default" and qset == "high":
        xt = dev(x.T.copy()).t()                             # time-contiguous input
        assert bits_equal(core.thresholds_array(xt, wt, q).cpu().numpy(), want)


def test_thresholds_many_cells_gappy(core):
    # about 5 000 cells of a gappy baseline: many tiles of k_thr_net, every fourth cell with a NaN / infinity handed over to k_thr_seg
    from hdp_b200 import _tables as tb
    ax = ta.gappy("noleap", seed=3)
    wt = tb.window_tables(ax.dayofyr, 7)
    rng = np.random.default_rng(41)
    T, C = len(ax), 5003
    x = (15 + 12 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365) + 3 * rng.standard_normal((T, C), dtype=np.float32)).astype(np.float32)
    bad = np.arange(0, C, 4)
    x[rng.integers(0, T, bad.size), bad] = np.where(rng.random(bad.size) < 0.5, np.nan, np.inf).astype(np.float32)
    x[T - 1, 1::8] = np.nan
    q = QSETS["high"]
    names = _net_launches(core, lambda: core.thresholds_array(dev(x), wt, q))
    assert "k_thr_net" in names and "k_thr_seg" in names
    got = core.thresholds_array(dev(x), wt, q).cpu().numpy()
    sel = np.unique(np.concatenate([np.arange(0, 96), rng.integers(0, C, 160), [C - 2, C - 1]]))
    want = oracle.thresholds_batch(np.ascontiguousarray(x[:, sel]), wt.window_samples(), q)
    assert bits_equal(got[sel], want)


# ------------------------------------------------------------------------------------------ path 2
@pytest.fixture(params=["filter", "nofilter"])
def scan_filter(request, core):
    """With k_scan's run filter (short runs after long breaks dropped before the state machines see them) and with every run fed
    through; both must match the reference bit for bit."""
    from hdp_b200 import _lib
    _lib.lib().hdp_b200_metrics_run_filter(1 if request.param == "filter" else 0)
    yield request.param
    _lib.lib().hdp_b200_metrics_run_filter(1)


def _pattern_masks(T, rng):
    """Hot-day patterns at the run filter's extremes (min_duration up to 32, max_break up to 30)."""
    t = np.arange(T)
    runs = np.zeros(T, bool)
    i = 0
    while i < T:                                             # random runs of 1 .. 40 days, breaks of 1 .. 35
        n = int(rng.integers(1, 41))
        runs[i:i + n] = True
        i += n + int(rng.integers(1, 36))
    return [np.ones(T, bool), np.zeros(T, bool), t % 62 < 32, t % 62 < 31, runs, (t % 33) < 2]


def _run_case(name, C=77, P=3):
    from hdp_b200 import _tables as tb
    ax = AXES[name]()
    rng = np.random.default_rng(len(name) * 7 + 1)
    T = len(ax)
    n_doy = 366 if ax.calendar == "standard" else 365
    z = rng.standard_normal((T, C))
    w = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
        w[t] = 0.8 * w[t - 1] + 0.6 * w[t]
    cyc = 10 * np.sin(2 * np.pi * (ax.dayofyr[:, None] - 110) / 365)
    x = (15 + cyc + 4 * z).astype(np.float32)
    xb = (4 + cyc + 4 * (0.7 * z + 0.7 * w)).astype(np.float32)
    for c, m in enumerate(_pattern_masks(T, rng)):
        x[:, c] = np.where(m, 80.0, -40.0)
        xb[:, c] = np.where(m, 80.0, -40.0)
    x[rng.integers(0, T, 40), rng.integers(0, C, 40)] = np.nan
    thr_cyc = 10 * np.sin(2 * np.pi * (np.arange(n_doy)[None, :, None] - 110) / 365)
    off = np.linspace(1, 5, P)[None, None, :]
    thr = 15 + thr_cyc + off + 0.5 * rng.standard_normal((C, n_doy, 1))
    thr_b = 4 + thr_cyc + off + 0.5 * rng.standard_normal((C, n_doy, 1))
    if name.startswith("summer"):
        north, south = ta.summer_seasons(ax)
    else:
        st = tb.hemisphere_ranges(ax)
        north, south = st.north, st.south
    is_south = (np.arange(C) % 3 == 1).astype(np.uint8)      # both hemispheres in every warp
    return dict(ax=ax, x=x, xb=xb, thr=thr, thr_b=thr_b, dm=tb.doy_map(ax.dayofyr), north=north, south=south, is_south=is_south)


def _defs(kind):
    from hdp_b200 import workloads
    if kind == "readme":
        return workloads.README_DEFS
    rng = np.random.default_rng({"randA": 3, "randB": 8}[kind])
    lmin, bmax = (2, 30) if kind == "randA" else (int(rng.integers(2, 33)), int(rng.integers(0, 31)))
    D = 9
    defs = np.stack([rng.integers(lmin, 33, D), rng.integers(0, bmax + 1, D), rng.integers(0, 4, D)], axis=1)
    defs[0] = [lmin, bmax, 1]
    defs[1] = [32, bmax, 0]
    return defs.tolist()


def _lanes(core, defs, north, south, T):
    from hdp_b200 import _lib
    from hdp_b200._core import _hp, _i32
    info = (ctypes.c_int * 7)()
    df, sn, ss = _i32(defs), _i32(north), _i32(south)
    assert _lib.lib().hdp_b200_metrics_kernel_choice(_hp(df), df.shape[0], _hp(sn), _hp(ss), sn.shape[0], T, info) == 0
    return tuple(info)


@pytest.mark.parametrize("kind", ["readme", "randA", "randB"])
@pytest.mark.parametrize("name", sorted(AXES))
def test_metric_pass(core, scan_filter, monkeypatch, name, kind):
    k = cached(("run", name), lambda: _run_case(name))
    x, thr, dm = k["x"], k["thr"], k["dm"]
    defs = _defs(kind)
    args = (dm, defs, k["north"], k["south"], k["is_south"])
    T = len(k["ax"])
    info = _lanes(core, defs, k["north"], k["south"], T)
    seasons_max = max(np.diff(k["north"], axis=1).max(), np.diff(k["south"], axis=1).max())
    assert info[0] == (8 if seasons_max <= 255 else 16)
    if name.startswith("gappy"):
        assert info[0] == 16                                 # the season to the next year's 1 October
    if kind != "readme":
        assert info[3] == (scan_filter == "filter")          # the run filter at min_duration 2 .. 32, max_break up to 30
    d_x, d_thr = dev(x), dev(thr)
    # u16 metrics
    met = core.metrics_array(d_x, d_thr, *args)
    want = oracle.metrics_batch(x, thr, *args)
    assert np.array_equal(ref_layout(met), want)
    assert want[:, :, :, 0].max() > 0
    # HWO / HWE
    on = core.metrics_array(d_x, d_thr, *args, onset=True)
    assert torch.equal(on[:4], met)
    assert np.array_equal(on[4:].cpu().numpy(), onset_oracle.onset_batch(x, thr, *args))
    # intensity, with the metrics of the same pass
    mo = torch.zeros_like(met)
    heat = core.intensity_array(d_x, d_thr, *args, metrics_out=mo)
    assert torch.equal(mo, met)
    want_h = intensity_oracle.intensity_batch(x, thr, *args)
    assert same_f32(heat_layout(heat), want_h)
    # cold spells: the heatwave pass on negated inputs
    nx, nthr = dev((-x).astype(np.float32)), dev(-thr)
    assert torch.equal(core.metrics_array(d_x, d_thr, *args, cold=True), core.metrics_array(nx, nthr, *args))
    mo_c = torch.zeros_like(met)
    heat_c = core.intensity_array(d_x, d_thr, *args, metrics_out=mo_c, cold=True)
    mo_n = torch.zeros_like(met)
    assert torch.equal(heat_c, core.intensity_array(nx, nthr, *args, metrics_out=mo_n)) and torch.equal(mo_c, mo_n)
    # a time-contiguous view of the samples
    xt = dev(x.T.copy()).t()
    assert torch.equal(core.metrics_array(xt, d_thr, *args), met)
    # the host pipeline in chunks of 32 cells (three chunks, the last one ragged)
    monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", "32")
    met_np = met.cpu().numpy()
    assert np.array_equal(core.metrics_host(x, thr, *args), met_np)
    mo_h = np.zeros_like(met_np)
    heat_h = core.intensity_host(x, thr, *args, metrics_out=mo_h)
    assert np.array_equal(mo_h, met_np) and same_f32(heat_h, heat.cpu().numpy())


@pytest.mark.parametrize("name", sorted(AXES))
def test_compound_pass(core, scan_filter, name):
    from hdp_b200 import workloads
    k = cached(("run", name), lambda: _run_case(name))
    x, xb, thr, thr_b, dm = k["x"], k["xb"], k["thr"], k["thr_b"], k["dm"]
    args = (dm, workloads.README_DEFS, k["north"], k["south"], k["is_south"])
    met = core.compound_metrics_array(dev(x), dev(thr), dev(xb), dev(thr_b), *args)
    mo = torch.zeros_like(met)
    heat = core.compound_intensity_array(dev(x), dev(thr), dev(xb), dev(thr_b), *args, metrics_out=mo)
    assert torch.equal(met, mo)
    want, want_h = compound_oracle(x, thr, xb, thr_b, *args)
    assert np.array_equal(ref_layout(met), want) and want[:, :, :, 0].max() > 0
    assert same_f32(heat.cpu().numpy().transpose(0, 2, 3, 5, 1, 4), want_h)
    mask = core.compound_hot_days_array(dev(x), dev(thr), dev(xb), dev(thr_b), dm).cpu().numpy()
    assert np.array_equal(mask.astype(bool), compound_mask(x, thr, xb, thr_b, dm))


@pytest.mark.parametrize("name", sorted(AXES))
def test_hot_days(core, name):
    k = cached(("run", name), lambda: _run_case(name))
    x, thr, dm = k["x"], k["thr"], k["dm"]
    got = core.hot_days_array(dev(x), dev(thr), dm).cpu().numpy()
    for c in range(x.shape[1]):
        for p in range(thr.shape[2]):
            assert np.array_equal(got[p, :, c].astype(bool), oracle.indicate_hot_days(x[:, c], thr[c, :, p], dm))


# ------------------------------------------------------------------------------------------ limits
def _stride_case(T, C=40, P=2, seed=0):
    rng = np.random.default_rng(seed + T)
    dm = ta.stride_map(T)
    z = rng.standard_normal((T, C))
    for t in range(1, T):
        z[t] = 0.9 * z[t - 1] + 0.45 * z[t]
    x = z.astype(np.float32)
    x[:, 0] = 5.0
    thr = np.linspace(0.2, 0.8, P)[None, None, :] + 0.1 * rng.standard_normal((C, 365, 1))
    n = T // 365 + 1
    north = np.array([[i * 365 + 120, i * 365 + 273] for i in range(n)])
    south = np.array([[i * 365 + 300, i * 365 + 455] for i in range(n)])
    return x, thr, dm, north, south, (np.arange(C) % 2).astype(np.uint8)


def test_scan_word_limit(core, scan_filter):
    # one-day words: K = T.  k_scan keeps K + 1 word records in shared memory; one word more than fit must be refused, not run
    from hdp_b200 import _lib, workloads
    defs = workloads.README_DEFS
    K = ta.scan_word_limit(defs)
    for T, ok in ((K, True), (K + 1, False)):
        x, thr, dm, north, south, is_south = _stride_case(T)
        assert ta.n_words(dm) == T
        args = (dm, defs, north, south, is_south)
        if ok:
            met = core.metrics_array(dev(x), dev(thr), *args)
            assert np.array_equal(ref_layout(met), oracle.metrics_batch(x, thr, *args))
            mo = torch.zeros_like(met)
            heat = core.intensity_array(dev(x), dev(thr), *args, metrics_out=mo)
            assert torch.equal(mo, met) and same_f32(heat_layout(heat), intensity_oracle.intensity_batch(x, thr, *args))
        else:
            for call in (lambda: core.metrics_array(dev(x), dev(thr), *args),
                         lambda: core.intensity_array(dev(x), dev(thr), *args, metrics_out=torch.zeros((4, 2, 6, len(north), 40), dtype=torch.uint16, device="cuda"))):
                with pytest.raises(_lib.HdpB200Error) as e:
                    call()
                assert e.value.code == -2


def test_intensity_word_limit(core):
    # k_intensity alone keeps K int2 word records beside one warp's state: under its own limit it equals the oracle, above it -2
    from hdp_b200 import _lib, workloads
    defs = workloads.README_DEFS
    K = ta.intensity_word_limit(len(defs))
    for T, ok in ((K, True), (K + 1, False)):
        x, thr, dm, north, south, is_south = _stride_case(T, C=33)
        args = (dm, defs, north, south, is_south)
        if ok:
            heat = core.intensity_array(dev(x), dev(thr), *args)
            assert same_f32(heat_layout(heat), intensity_oracle.intensity_batch(x, thr, *args))
        else:
            with pytest.raises(_lib.HdpB200Error) as e:
                core.intensity_array(dev(x), dev(thr), *args)
            assert e.value.code == -2


def test_hot_days_word_limit(core):
    # k_unpack_mask launches one grid row per word: 65 535 words run, one more is refused
    from hdp_b200 import _lib
    for T, ok in ((65535, True), (65536, False)):
        x, thr, dm, *_ = _stride_case(T, C=8, P=1)
        if ok:
            got = core.hot_days_array(dev(x), dev(thr), dm).cpu().numpy()
            for c in range(8):
                assert np.array_equal(got[0, :, c].astype(bool), oracle.indicate_hot_days(x[:, c], thr[c, :, 0], dm))
        else:
            with pytest.raises(_lib.HdpB200Error) as e:
                core.hot_days_array(dev(x), dev(thr), dm)
            assert e.value.code == -2


def test_workspace_bound_without_map(core):
    # *_workspace_bytes with a NULL map promises enough for regular daily calendars only; an 80-year May - September series has
    # six words per year where the bound allows for about 5.7: the pass must return -3 and write nothing
    from hdp_b200 import _lib, workloads
    from hdp_b200._core import _hp, _i32
    L = _lib.lib()
    ax = ta.summer("noleap", years=80, start=1941)
    T, C, P = len(ax), 64, 2
    dm, df = _i32(ax.dayofyr - 1), _i32(workloads.README_DEFS)
    north, south = ta.summer_seasons(ax)
    sn, ss = _i32(north), _i32(south)
    D, Y = df.shape[0], sn.shape[0]
    rng = np.random.default_rng(2)
    x = dev((20 + 4 * rng.standard_normal((T, C))).astype(np.float32))
    thr = dev(22 + rng.standard_normal((C, 365, P)))
    stream = torch.cuda.current_stream().cuda_stream
    for name, planes in (("hdp_b200_metrics", 4), ("hdp_b200_intensity", 3)):
        n_null = getattr(L, name + "_workspace_bytes")(C, T, C, 1, 365, P, D, Y, None)
        n_map = getattr(L, name + "_workspace_bytes")(C, T, C, 1, 365, P, D, Y, _hp(dm))
        assert 0 < n_null < n_map
        ws = torch.empty(n_null, dtype=torch.uint8, device="cuda")
        out = torch.full((planes, P, D, Y, C), 4321, dtype=torch.int32 if planes == 3 else torch.int16, device="cuda")
        if planes == 3:
            out = out.view(torch.float32)
        before = out.clone()
        outs = (out.data_ptr(),) if planes == 4 else (out.data_ptr(), None)
        rc = getattr(L, name)(x.data_ptr(), C, T, C, 1, thr.data_ptr(), 365, P, _hp(dm), _hp(df), D, _hp(sn), _hp(ss), Y, None, *outs,
                              ws.data_ptr(), n_null, stream, 0)
        torch.cuda.synchronize()
        assert rc == -3 and torch.equal(out.view(torch.int16), before.view(torch.int16))
        ws = torch.empty(n_map, dtype=torch.uint8, device="cuda")
        assert getattr(L, name)(x.data_ptr(), C, T, C, 1, thr.data_ptr(), 365, P, _hp(dm), _hp(df), D, _hp(sn), _hp(ss), Y, None, *outs,
                                ws.data_ptr(), n_map, stream, 0) == 0


def _refused(call, outs):
    """call() raises HdpB200Error -1 and leaves every pre-filled output as it was."""
    from hdp_b200 import _lib
    before = [o.clone() if isinstance(o, torch.Tensor) else o.copy() for o in outs]
    with pytest.raises(_lib.HdpB200Error) as e:
        call()
    assert e.value.code == -1
    torch.cuda.synchronize()
    for o, b in zip(outs, before):
        assert torch.equal(o, b) if isinstance(o, torch.Tensor) else np.array_equal(o.view(np.uint8), b.view(np.uint8))


def test_summer_thresholds_with_a_full_year_map(core):
    # thresholds of a May - September baseline have 153 rows; the day-of-year map of a run (dayofyr - 1) reaches 272.  The reference
    # indexes past its table there; the library refuses.
    from hdp_b200 import _tables as tb, workloads
    base = ta.summer("noleap")
    run = ta.summer("noleap", years=5, start=2001)
    rng = np.random.default_rng(4)
    C = 40
    xb = (20 + 4 * rng.standard_normal((len(base), C))).astype(np.float32)
    x = (21 + 4 * rng.standard_normal((len(run), C))).astype(np.float32)
    thr = core.thresholds_array(dev(xb), tb.window_tables(base.dayofyr, 7), [0.9, 0.95])
    assert thr.shape[1] == 153
    dm = tb.doy_map(run.dayofyr)
    north, south = ta.summer_seasons(run)
    args = (dm, workloads.README_DEFS, north, south, None)
    out = torch.full((4, 2, 6, 5, C), 7, dtype=torch.int16, device="cuda").view(torch.uint16)
    heat = torch.full((3, 2, 6, 5, C), 7.0, dtype=torch.float32, device="cuda")
    _refused(lambda: core.metrics_array(dev(x), thr, *args, out=out), [out.view(torch.int16)])
    _refused(lambda: core.intensity_array(dev(x), thr, *args, out=heat), [heat])
    _refused(lambda: core.hot_days_array(dev(x), thr, dm), [])


def test_map_entry_past_the_table_inside_a_word(core, monkeypatch):
    # noleap thresholds (365 rows) with a standard-calendar run: 31 December of a leap year maps to 365, inside the word that starts
    # at 352 (days of year 352 .. 365 are one word).  Every entry point must refuse the map (-1) and write nothing.
    from hdp_b200 import _lib, _tables as tb, workloads
    from hdp_b200._core import _hp, _i32
    run = tb.TimeAxis.date_range("2001-01-01", "2005-12-31", "standard")
    dm = tb.doy_map(run.dayofyr)
    assert dm.max() == 365
    t = int(np.flatnonzero(dm == 352)[3])                    # 2004: its word runs through 31 December
    nb = ta.word_lengths(dm[t:])[0]
    assert dm[t + nb - 1] == 365
    rng = np.random.default_rng(6)
    T, C, P = len(run), 45, 2
    x = (20 + 4 * rng.standard_normal((T, C))).astype(np.float32)
    x[t:t + nb] = 60.0                                       # hot on every day of that word
    thr = 22 + rng.standard_normal((C, 365, P))
    st = tb.hemisphere_ranges(run)
    Y = st.n_years
    defs = workloads.README_DEFS
    args = (dm, defs, st.north, st.south, (np.arange(C) % 2).astype(np.uint8))
    d_x, d_thr = dev(x), dev(thr)

    def u16(shape):
        return torch.full(shape, 7, dtype=torch.int16, device="cuda").view(torch.uint16)
    out, heat, mo = u16((4, P, 6, Y, C)), torch.full((3, P, 6, Y, C), 7.0, device="cuda"), u16((4, P, 6, Y, C))
    cheat = torch.full((2, 3, P, 6, Y, C), 7.0, device="cuda")
    _refused(lambda: core.metrics_array(d_x, d_thr, *args, out=out), [out.view(torch.int16)])
    _refused(lambda: core.intensity_array(d_x, d_thr, *args, out=heat, metrics_out=mo), [heat, mo.view(torch.int16)])
    _refused(lambda: core.compound_metrics_array(d_x, d_thr, d_x, d_thr, *args, out=out), [out.view(torch.int16)])
    _refused(lambda: core.compound_intensity_array(d_x, d_thr, d_x, d_thr, *args, out=cheat, metrics_out=mo),
             [cheat, mo.view(torch.int16)])
    # hot_days through the C ABI, with a pre-filled mask
    L = _lib.lib()
    mask = torch.full((P, T, C), 7, dtype=torch.uint8, device="cuda")
    dm32 = _i32(dm)
    ws = torch.empty(L.hdp_b200_metrics_workspace_bytes(C, T, C, 1, 365, P, 1, 0, _hp(dm32)), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    assert L.hdp_b200_hot_days(d_x.data_ptr(), C, T, C, 1, d_thr.data_ptr(), 365, P, _hp(dm32), mask.data_ptr(), ws.data_ptr(),
                               ws.numel(), stream) == -1
    assert L.hdp_b200_compound_hot_days(d_x.data_ptr(), C, 1, d_x.data_ptr(), C, 1, C, T, d_thr.data_ptr(), d_thr.data_ptr(), 365, P,
                                        _hp(dm32), mask.data_ptr(), ws.data_ptr(), ws.numel(), stream, 0) == -1
    torch.cuda.synchronize()
    assert (mask == 7).all()
    # the host pipeline
    monkeypatch.setenv("HDP_B200_HOST_CHUNK_CELLS", "32")
    out_h = np.full((4, P, 6, Y, C), 7, np.uint16)
    heat_h, mo_h = np.full((3, P, 6, Y, C), 7.0, np.float32), np.full((4, P, 6, Y, C), 7, np.uint16)
    _refused(lambda: core.metrics_host(x, thr, *args, out=out_h), [out_h])
    _refused(lambda: core.intensity_host(x, thr, *args, out=heat_h, metrics_out=mo_h), [heat_h, mo_h])
    _refused(lambda: core.compound_metrics_host(x, thr, x, thr, *args, out=out_h), [out_h])
    # the same run with 366-row thresholds is fine
    thr366 = np.concatenate([thr, thr[:, -1:]], axis=1)
    assert np.array_equal(ref_layout(core.metrics_array(d_x, dev(thr366), *args)), oracle.metrics_batch(x, thr366, *args))
