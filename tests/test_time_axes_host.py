"""The tables of time axes that are not whole continuous years (tests/time_axes.py: mid-year starts, missing days, May - September
subsets, one-day words), without a GPU: invariants of window_tables / doy_map / hemisphere_ranges that the kernels rely on, the
host replay of k_intensity's lane loop (hdp_b200/csrc/intensity.h, tests/intensity_host.cpp) on these axes' day-of-year maps
against the intensity oracle, and the reference's own table builders on the same axes.  tests/test_gpu_time_axes.py runs the
kernels on them."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import intensity_oracle
import time_axes as ta
from hdp_b200 import _tables as tb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

AXES = {
    "mid_noleap": lambda: ta.mid("noleap"),
    "mid_standard": lambda: ta.mid("standard"),
    "gappy_noleap": lambda: ta.gappy("noleap"),
    "gappy_standard": lambda: ta.gappy("standard"),
    "summer_noleap": lambda: ta.summer("noleap"),
    "summer_standard": lambda: ta.summer("standard"),
}


# ------------------------------------------------------------------------------------------------ the axes themselves
def test_axes_are_what_they_say():
    ax = ta.mid("noleap")
    assert (ax.year[0], ax.month[0], ax.day[0]) == (1961, 7, 10) and (ax.year[-1], ax.month[-1], ax.day[-1]) == (1991, 3, 20)
    ax = ta.mid("standard")
    assert (ax.year[0], ax.month[0], ax.day[0], ax.dayofyr[0]) == (1964, 3, 1, 61)
    for cal in ("noleap", "standard"):
        full = tb.TimeAxis.date_range("1961-01-01", "1990-12-31", cal)
        ax = ta.gappy(cal)
        assert 0.01 < 1 - len(ax) / len(full) < 0.02
        for dy, m, d in ta.GAPPY_DROPS.values():
            assert not ((ax.year == 1961 + dy) & (ax.month == m) & (ax.day == d)).any()
        assert not ((ax.year == 1961 + ta.GAPPY_MONTH[0]) & (ax.month == ta.GAPPY_MONTH[1])).any()
        assert ta.gappy(cal).dayofyr.tolist() == ax.dayofyr.tolist()                        # fixed seed
        s = ta.summer(cal)
        assert set(s.month.tolist()) == {5, 6, 7, 8, 9} and len(s) == 30 * 153


# ------------------------------------------------------------------------------------------------ path 1 tables
@pytest.mark.parametrize("name", sorted(AXES))
@pytest.mark.parametrize("radius", [0, 7, 15])
def test_window_tables_invariants(name, radius):
    ax = AXES[name]()
    wt = tb.window_tables(ax.dayofyr, radius)
    ti = wt.time_index
    T = len(ax)
    # every time index exactly once; -1 pads only at the END of a row (a pad reads the last sample, thr_net.cu net_plan)
    assert np.array_equal(np.sort(ti[ti >= 0]), np.arange(T))
    valid = ti >= 0
    assert (valid[:, :-1] | ~valid[:, 1:]).all()
    assert valid[:, 0].all()
    # one day of year per row, rows in first-appearance order, samples of a row in time order
    first = ti[:, 0]
    assert (np.diff(first) > 0).all()
    for d in range(wt.n_doy):
        row = ti[d][valid[d]]
        assert (np.diff(row) > 0).all() and np.unique(ax.dayofyr[row]).size == 1
    assert wt.n_y == np.bincount(np.unique(ax.dayofyr, return_inverse=True)[1]).max()
    # the window of row d: rows d - r .. d + r in the reference's wrap (mirrored above the last row)
    assert wt.width == 2 * radius + 1 and ((wt.win_rows >= 0) & (wt.win_rows < wt.n_doy)).all()
    assert (wt.win_rows[:, radius] == np.arange(wt.n_doy)).all()


def test_window_table_shapes():
    # the row depths that pick the k_thr_net instances: 30 (the exact instance, pads read through time_of), 31 (NY = 32)
    assert tb.window_tables(ta.mid("noleap").dayofyr, 7).n_y == 30
    assert (tb.window_tables(ta.mid("noleap").dayofyr, 7).time_index < 0).any(1).sum() == 111          # 21 March .. 9 July
    assert tb.window_tables(ta.mid("standard").dayofyr, 7).n_y == 31
    g = tb.window_tables(ta.gappy("noleap").dayofyr, 7)
    assert g.n_doy == 365 and g.n_y == 30 and (g.time_index < 0).any(1).sum() > 60                       # pads in arbitrary rows
    s = tb.window_tables(ta.summer("noleap").dayofyr, 7)
    assert s.n_doy == 153 and not (s.time_index < 0).any()
    assert tb.window_tables(ta.summer("standard").dayofyr, 7).n_doy == 154                              # 30 April / 30 September of leap years


# ------------------------------------------------------------------------------------------------ path 2 tables
@pytest.mark.parametrize("name", sorted(AXES))
def test_doy_map_and_words(name):
    ax = AXES[name]()
    dm = tb.doy_map(ax.dayofyr)
    assert np.array_equal(dm, ax.dayofyr - 1)
    nb = ta.word_lengths(dm)
    assert nb.sum() == len(ax) and nb.min() >= 1 and nb.max() <= 32
    t0 = np.concatenate([[0], np.cumsum(nb)[:-1]])
    for t, n in zip(t0, nb):                                          # consecutive days of year inside one 32-day block
        assert np.array_equal(dm[t:t + n], dm[t] + np.arange(n)) and dm[t] // 32 == dm[t + n - 1] // 32
    if name.startswith("gappy"):                                      # the gaps cut the words short
        assert nb.size > ta.n_words(tb.doy_map(tb.TimeAxis.date_range("1961-01-01", "1990-12-31", ax.calendar).dayofyr)) + 50


def test_stride_map_words():
    dm = ta.stride_map(1000)
    assert ta.n_words(dm) == 1000 and (ta.word_lengths(dm) == 1).all()
    assert ta.n_words(np.arange(365)) == 12 and ta.n_words(np.arange(730) % 365) == 24               # one word per 32-day block
    defs = [[3, 0, 0], [3, 1, 1], [32, 30, 2]]
    assert ta.scan_word_limit(defs) == (200 * 1024 - ((12288 + 34 + 33 + 3) & ~3) * 4) // 16 - 1
    assert ta.scan_word_limit([[3, 1, 0]]) == 9725 and ta.intensity_word_limit(6) == 24256


def test_hemisphere_ranges_gappy():
    for cal in ("noleap", "standard"):
        ax = ta.gappy(cal)
        st = tb.hemisphere_ranges(ax)
        for tab in (st.north, st.south):
            assert (tab >= 0).all() and (tab[:, 1] > tab[:, 0]).all() and (tab[1:, 0] >= tab[:-1, 1]).all()   # sorted, disjoint
        # the year without 1 October: its season runs to the NEXT year's 1 October, about 520 days, and the rows behind it shift
        y_oct = 1961 + ta.GAPPY_DROPS["oct1"][0]
        n = st.north
        row = np.flatnonzero(ax.year[n[:, 0]] == y_oct)[0]
        assert ax.year[n[row, 1]] == y_oct + 1 and (ax.month[n[row, 1]], ax.day[n[row, 1]]) == (10, 1)
        assert 500 < n[row, 1] - n[row, 0] < 530
        assert ax.year[n[row + 1, 0]] == y_oct + 2                   # no season starts in the year the long one ends in
        # the year without 1 May: no northern season starts in it
        y_may = 1961 + ta.GAPPY_DROPS["may1"][0]
        assert not (ax.year[n[:, 0]] == y_may).any()
        assert st.n_years < 30
        # trimming keeps every season the south table found (the north one has two fewer)
        assert st.north.shape == st.south.shape


def test_hemisphere_ranges_mid_year_start():
    ax = ta.mid("noleap")
    st = tb.hemisphere_ranges(ax)
    # the first northern season is the one of 1962, in row 0 beside the southern season of 1961/62 (the reference's rows)
    assert (ax.year[st.north[0, 0]], ax.month[st.north[0, 0]]) == (1962, 5)
    assert (ax.year[st.south[0, 0]], ax.month[st.south[0, 0]]) == (1961, 11)
    assert np.diff(st.north, axis=1).max() <= 255 and np.diff(st.south, axis=1).max() <= 255      # k_scan's 8-bit lanes


# ------------------------------------------------------------------------------------------------ intensity.h replay
@pytest.fixture(scope="module")
def replay(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("intensity") / "libintensity_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-shared", "-fPIC", "-I",
                    os.path.join(ROOT, "hdp_b200", "csrc"), os.path.join(ROOT, "tests", "intensity_host.cpp"), "-o", so], check=True)
    L = ctypes.CDLL(so)
    p = ctypes.c_void_p
    L.intensity_host_cell.argtypes = [p, p, p, ctypes.c_int64, p, ctypes.c_int, p, ctypes.c_int, p]

    def run(x, thr, doy_map, defs, seasons):
        x = np.ascontiguousarray(x, np.float32)
        thr = np.ascontiguousarray(thr, np.float64)
        dm = np.ascontiguousarray(doy_map, np.int32)
        df = np.ascontiguousarray(defs, np.int32).reshape(-1, 3)
        sn = np.ascontiguousarray(seasons, np.int32).reshape(-1, 2)
        out = np.full((3, df.shape[0], sn.shape[0]), -7.0, np.float32)
        rc = L.intensity_host_cell(x.ctypes.data, thr.ctypes.data, dm.ctypes.data, x.size, df.ctypes.data, df.shape[0],
                                   sn.ctypes.data, sn.shape[0], out.ctypes.data)
        return rc, out
    return run


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("name", sorted(AXES) + ["stride"])
def test_intensity_replay_on_short_words(replay, name):
    rng = np.random.default_rng(len(name))
    if name == "stride":
        dm = ta.stride_map(4000)
        n_doy = 365
        north = np.array([[i * 365 + 120, i * 365 + 273] for i in range(11)])
        south = np.array([[i * 365 + 300, i * 365 + 455] for i in range(11)])
    else:
        ax = AXES[name]()
        dm = tb.doy_map(ax.dayofyr)
        n_doy = 366 if ax.calendar == "standard" else 365
        if name.startswith("summer"):
            north, south = ta.summer_seasons(ax)
        else:
            st = tb.hemisphere_ranges(ax)
            north, south = st.north, st.south
    T = dm.size
    z = rng.standard_normal(T)
    for t in range(1, T):
        z[t] = 0.8 * z[t - 1] + 0.6 * z[t]
    thr = rng.normal(0.6, 0.3, n_doy)
    x = z.astype(np.float32)
    x[rng.integers(0, T, 20)] = np.nan
    defs = [[3, 0, 0], [3, 1, 1], [1, 0, 0], [5, 2, 3], [2, 30, 1]]
    for seasons in (north, south):
        rc, got = replay(x, thr, dm, defs, seasons)
        assert rc == 0
        want = np.stack([intensity_oracle.heatwave_intensity(x, thr, dm, *d, seasons) for d in defs], axis=1)
        assert np.array_equal(_bits(got), _bits(want))
        assert (got[0] > 0).any()


# ------------------------------------------------------------------------------------------------ the reference's builders
@pytest.fixture(scope="module")
def ref():
    pytest.importorskip("numba")
    from oracle import build as obuild, ref_numba
    if obuild.build_ref() is None or not ref_numba.available():
        pytest.skip("no reference tree and no earlier install")
    thr_mod, met_mod, _ = ref_numba.load()

    class Ref:
        threshold, metric = thr_mod, met_mod

        @staticmethod
        def dates(axis):
            return np.array([ref_numba.FakeDate(int(y), int(m), int(d), int(j), axis.calendar)
                             for y, m, d, j in zip(axis.year, axis.month, axis.day, axis.dayofyr)], dtype=object)
    return Ref


@pytest.mark.reference
@pytest.mark.parametrize("name", sorted(AXES))
def test_table_builders_match_reference(ref, name):
    ax = AXES[name]()
    dates = ref.dates(ax)
    for r in (0, 7):
        assert np.array_equal(tb.window_tables(ax.dayofyr, r).window_samples(), ref.threshold.datetimes_to_windows(dates, r))
    assert np.array_equal(tb.doy_map(ax.dayofyr), ref.metric.build_doy_map(dates))
    for s, e in (((5, 1), (10, 1)), ((11, 1), (4, 1))):
        assert np.array_equal(tb.range_indices(ax, s, e), ref.metric.get_range_indices(dates, s, e))
