"""The heatwave intensity metrics (HWC, HWI, HWP) without a GPU: the per-run / per-season accounting of k_intensity
(hdp_b200/csrc/intensity.h) replayed on the CPU by tests/intensity_host.cpp against the NumPy oracle, the C oracle against the
NumPy oracle, and the new C ABI entry points (exported, ABI version 5, workspace sizes).  The kernel itself is checked by
tests/test_gpu_intensity.py on the GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import intensity_oracle
import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def want_np(x, thr, dm, defs, seasons):
    return np.stack([intensity_oracle.np_intensity(x, thr, dm, *d, seasons) for d in defs], axis=1)      # [3, D, Y]


def check(replay, x, thr, dm, defs, seasons):
    rc, got = replay(x, thr, dm, defs, seasons)
    assert rc == 0
    want = want_np(x, thr, dm, defs, seasons)
    assert np.array_equal(bits(got), bits(want)), (got, want)
    return got


def test_hand_cases(replay):
    thr = np.array([1.0])
    T = 30
    dm = np.zeros(T, np.int64)
    x = np.zeros(T, np.float32)
    x[2:9] = [1.5, 2.25, 3.0, 1.75, 2.5, 1.25, 4.0]               # one 7-day run
    x[10] = 2.0                                                     # break day 9 -> 1-day run 10 (a sub-event of [3, 1, 1])
    x[13:15] = [5.0, 5.0]                                           # 2-day run, never labelled by min_duration 3 without a sub-event
    x[20:30] = 1.5                                                  # a 10-day run open at the end of the series
    defs = [[3, 0, 0], [3, 1, 1], [1, 0, 0], [8, 0, 0]]
    seasons = [[0, 5], [5, 12], [12, 12], [12, 25], [25, 40], [40, 50]]   # a run crossing a season edge, an empty season,
    got = check(replay, x, thr, dm, defs, seasons)                  # a season open at the end, a season past the end
    # [3, 0, 0], season [0, 5): days 2, 3, 4 -> 0.5 + 1.25 + 2.0
    assert got[0, 0, 0] == np.float32(3.75) and got[2, 0, 0] == np.float32(2.0)
    assert got[1, 0, 0] == np.float32(3.75 / 3)
    # season [5, 12): the rest of the run (0.75 + 1.5 + 0.25 + 3.0); the short run at 10 counts for [3, 1, 1] only (branch C)
    assert got[0, 0, 1] == np.float32(5.5) and got[0, 1, 1] == np.float32(6.5) and got[0, 2, 1] == np.float32(6.5)
    assert got[2, 1, 1] == np.float32(3.0)
    assert (got[:, :, 2] == 0).all()                                # empty season
    assert got[0, 0, 3] == np.float32(2.5)                          # [12, 25): the 2-day run is unlabelled, days 20 .. 24
    assert got[0, 2, 3] == np.float32(8.0 + 2.5)                    # ... but labelled by [1, 0, 0]
    assert (got[:, 3, :3] == 0).all() and got[0, 3, 3] == np.float32(2.5)   # [8, 0, 0]: only the last run is long enough
    assert got[0, 0, 4] == np.float32(2.5) and (got[:, :, 5] == 0).all()


def test_break_days_are_not_heatwave_days(replay):
    # break days are cold: they carry no heatwave id (index_heatwaves labels hot runs only) and add nothing
    x = np.array([3, 3, 3, 0, 3, 0, 0, 0, 3, 3, 3], np.float32)
    got = check(replay, x, [1.0], np.zeros(x.size), [[3, 1, 1], [3, 3, 1]], [[0, 11]])
    assert got[0, 0, 0] == 14.0 and got[0, 1, 0] == 14.0 and got[1, 0, 0] == 2.0


def test_nan_and_infinite_samples(replay):
    x = np.array([2, 2, np.nan, 2, 2, 2, np.inf, 2, 2, -np.inf, 2, 2, 2], np.float32)
    thr = np.array([1.0, np.nan])
    dm = np.zeros(x.size, np.int64)
    dm[11] = 1                                                     # NaN threshold: never hot
    got = check(replay, x, thr, dm, [[2, 0, 0], [3, 0, 0]], [[0, 13]])
    assert np.isinf(got[:, 0, 0]).all() and np.isinf(got[:, 1, 0]).all()          # +inf is hot: HWC, HWI, HWP are inf
    got = check(replay, x, thr, dm, [[2, 0, 0], [3, 0, 0]], [[0, 6], [7, 13]])     # the inf day is outside both seasons
    assert got[0, :, 0].tolist() == [5.0, 3.0] and got[0, :, 1].tolist() == [2.0, 2.0]


def test_season_tables(replay):
    x = np.ones(50, np.float32) * 2
    ok = [[0, 10], [10, 20], [-5, -1], [30, 30], [5, 5], [100, 200]]   # unsorted, negative, empty inside another: accepted
    check(replay, x, [1.0], np.zeros(50), [[3, 0, 0]], ok)
    rc, _ = replay(x, [1.0], np.zeros(50), [[3, 0, 0]], [[0, 10], [5, 15]])
    assert rc == -2                                                 # overlapping non-empty seasons
    rc, _ = replay(x, [1.0], np.zeros(50), [[3, 0, 0]], [[0, 10], [-45, -40]])
    assert rc == -2                                                 # [5, 10) after slice clamping


@pytest.mark.parametrize("T", [1, 31, 32, 33, 97, 400, 1500])
def test_random_series_many_definitions(replay, T):
    rng = np.random.default_rng(T)
    for trial in range(12):
        n_doy = int(rng.integers(1, 40))
        dm = np.arange(T) % n_doy
        if trial % 3 == 0:
            dm = (np.arange(T) * 3) % n_doy                           # days of year that are not consecutive: short words
        thr = rng.normal(0.0, 1.0, n_doy)
        z = rng.standard_normal(T)
        for t in range(1, T):
            z[t] = 0.7 * z[t - 1] + 0.7 * z[t]
        x = (z + rng.uniform(-1, 1)).astype(np.float32)
        if trial % 4 == 1:
            x[rng.integers(0, T, max(1, T // 20))] = np.nan
        D = int(rng.integers(1, 33))
        defs = np.stack([rng.integers(0, 7, D), rng.integers(0, 4, D), rng.integers(0, 4, D)], axis=1)
        Y = int(rng.integers(1, 9))
        cuts = np.sort(rng.integers(0, T + 10, 2 * Y))
        seasons = cuts.reshape(Y, 2)[rng.permutation(Y)]               # disjoint, in any order
        seasons = np.where((seasons < T) & (rng.random(seasons.shape) < 0.3), seasons - T, seasons)   # the same, from the end
        if trial % 5 == 0:
            seasons[0] = [seasons[0, 0], seasons[0, 0]]
        check(replay, x, thr, dm, defs, seasons)


def test_c_oracle_equals_numpy_oracle():
    rng = np.random.default_rng(9)
    for trial in range(60):
        T = int(rng.integers(1, 500))
        n_doy = int(rng.integers(1, 20))
        dm = rng.integers(0, n_doy, T)
        thr = rng.normal(0, 1, n_doy)
        thr[rng.integers(0, n_doy)] = np.nan if trial % 4 == 0 else thr[0]
        x = (rng.normal(0.5, 1, T)).astype(np.float32)
        if trial % 3 == 0:
            x[rng.integers(0, T, 3)] = rng.choice([np.nan, np.inf, -np.inf], 3)
        d = (int(rng.integers(0, 6)), int(rng.integers(0, 3)), int(rng.integers(0, 3)))
        seasons = np.sort(rng.integers(-T - 3, T + 4, (int(rng.integers(1, 6)), 2)), axis=1)   # overlapping too: the oracle takes any
        a = intensity_oracle.heatwave_intensity(x, thr, dm, *d, seasons)
        b = intensity_oracle.np_intensity(x, thr, dm, *d, seasons)
        assert np.array_equal(bits(a), bits(b)), trial


def test_intensity_is_positive_exactly_where_there_are_heatwave_days():
    rng = np.random.default_rng(4)
    T, C = 700, 23
    x = rng.normal(0, 1, (T, C)).astype(np.float32)
    thr = rng.normal(0.3, 0.2, (C, 7, 3))
    dm = np.arange(T) % 7
    defs = [[3, 0, 0], [3, 1, 1], [1, 2, 0], [5, 1, 2]]
    north = [[0, 100], [150, 300], [300, 500], [600, 700]]
    south = [[50, 120], [200, 200], [210, 400], [400, 699]]
    south_flag = (np.arange(C) % 2).astype(np.uint8)
    heat = intensity_oracle.intensity_batch(x, thr, dm, defs, north, south, south_flag)
    met = oracle.metrics_batch(x, thr, dm, defs, north, south, south_flag)
    hwf = met[:, :, :, 0, :]
    assert np.array_equal(heat[:, :, :, 0, :] > 0, hwf > 0)
    assert np.array_equal(heat[:, :, :, 2, :] > 0, hwf > 0)
    assert (heat[:, :, :, 1, :] <= heat[:, :, :, 2, :]).all()        # mean <= peak
    for c in (0, 1, C - 1):
        seasons = south if south_flag[c] else north
        for p in range(3):
            for k, d in enumerate(defs):
                want = intensity_oracle.np_intensity(x[:, c], thr[c, :, p], dm, *d, seasons)
                assert np.array_equal(bits(heat[p, k, c]), bits(want))


def test_abi_entry_points():
    from hdp_b200 import _lib
    L = _lib.lib()
    assert L.hdp_b200_abi_version() == 6
    raw = ctypes.CDLL(L._name)
    for name in ("hdp_b200_intensity", "hdp_b200_intensity_host", "hdp_b200_intensity_workspace_bytes"):
        assert hasattr(raw, name)
    w1 = L.hdp_b200_intensity_workspace_bytes(64, 31390, 64, 1, 365, 10, 6, 86, None)
    w2 = L.hdp_b200_intensity_workspace_bytes(128, 31390, 128, 1, 365, 10, 6, 86, None)
    w3 = L.hdp_b200_intensity_workspace_bytes(4096, 31390, 4096, 1, 365, 10, 6, 86, None)
    assert 0 < w1 < w2 < w3
    assert w1 >= L.hdp_b200_metrics_workspace_bytes(64, 31390, 64, 1, 365, 10, 6, 86, None)
    assert L.hdp_b200_intensity_workspace_bytes(-1, 31390, 64, 1, 365, 10, 6, 86, None) == 0
    assert "overlapping" in L.hdp_b200_strerror(-2).decode()
