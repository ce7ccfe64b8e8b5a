"""Which compiled kernel instance each case of tests/test_gpu_instances.py reaches, without a GPU.

k_thr_net is compiled for 24 (samples per row NY, list length K, blocks per window M) instances (HDP_NET_INSTANCES, thr_net.cu) and
k_scan for 46 (accumulator lanes, registers NG, counter planes KS, run-filter constants) instantiations (run_scan, metric.cu).  The
tables below give one input for each, and the host planners (hdp_b200_thresholds_kernel_choice, hdp_b200_metrics_kernel_choice)
must pick exactly that instance for it: so every instance that ships is reachable, and the GPU tests that run these cases against
the oracle run every one of them."""
import ctypes
import os
import re

import numpy as np
import pytest

from hdp_b200 import _lib, _tables as tb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NET = 4

# (NY, K, M) -> (years, radius, q, tm_warps): the network kernel's instance, the table / quantiles that reach it, and the CTA size
# of its tensor-memory variant (0 = k_thr_net only, the lists all fit shared memory).  Every case reaches its instance with a
# noleap calendar (the mirrored year-end program) and with a standard one (leap years: the table-driven irregular program).
# NY = 30 is picked for 30-year baselines only, NY = 16 for up to 16 years, NY = 32 for the rest up to 32; M = 3 when the window
# width is a multiple of 3; K is the shortest list that reaches the deepest requested position from the top of the window.
NET_CASES = {
    (16, 16, 3): (8, 1, (0.45, 0.9), 0),
    (16, 16, 1): (8, 2, (0.67, 0.95), 0),
    (16, 32, 3): (8, 4, (0.6, 0.9), 0),
    (16, 32, 1): (8, 2, (0.26, 0.9), 12),
    (16, 48, 3): (8, 4, (0.37, 0.9), 12),
    (16, 48, 1): (8, 3, (0.19, 0.9), 8),
    (16, 64, 3): (8, 4, (0.15, 0.9), 12),
    (16, 64, 1): (8, 5, (0.3, 0.9), 4),
    (30, 16, 3): (30, 1, (0.86, 0.99), 0),
    (30, 16, 1): (30, 2, (0.92, 0.99), 0),
    (30, 32, 3): (30, 1, (0.68, 0.99), 0),
    (30, 32, 1): (30, 2, (0.81, 0.99), 12),
    (30, 48, 3): (30, 1, (0.5, 0.99), 0),
    (30, 48, 1): (30, 2, (0.7, 0.99), 12),
    (30, 64, 3): (30, 1, (0.32, 0.99), 0),
    (30, 64, 1): (30, 2, (0.6, 0.99), 8),
    (32, 16, 3): (20, 1, (0.78, 0.99), 0),
    (32, 16, 1): (20, 2, (0.87, 0.99), 0),
    (32, 32, 3): (20, 1, (0.51, 0.99), 0),
    (32, 32, 1): (20, 2, (0.71, 0.99), 12),
    (32, 48, 3): (20, 1, (0.24, 0.99), 0),
    (32, 48, 1): (20, 2, (0.55, 0.99), 12),
    (32, 64, 3): (20, 1, (0.07, 0.99), 0),
    (32, 64, 1): (20, 2, (0.39, 0.99), 8),
}
NET_CALENDARS = ("noleap", "standard")


def net_axis(calendar, years):
    return tb.TimeAxis.date_range("1961-01-01", f"{1960 + years}-12-31", calendar)


def thresholds_choice(calendar, years, radius, q):
    ax = net_axis(calendar, years)
    wt = tb.window_tables(ax.dayofyr, radius)
    ti = np.ascontiguousarray(wt.time_index, np.int32)
    wr = np.ascontiguousarray(wt.win_rows, np.int32)
    qq = np.ascontiguousarray(q, np.float64)
    info = (ctypes.c_int * 8)()
    rc = _lib.lib().hdp_b200_thresholds_kernel_choice(ti.ctypes.data_as(ctypes.c_void_p), wr.ctypes.data_as(ctypes.c_void_p), len(ax),
                                                      wt.n_doy, wt.n_y, wt.width, qq.ctypes.data_as(ctypes.c_void_p), qq.size, info)
    assert rc == 0
    return list(info)


def compiled_net_instances():
    """The (NY, K, M) list of HDP_NET_INSTANCES in a full build, read from thr_net.cu."""
    src = open(os.path.join(ROOT, "hdp_b200", "csrc", "thr_net.cu")).read()
    full = src.split("#else", 1)[1].split("#endif", 1)[0]     # (the #ifdef HDP_NET_DEV branch is a reduced set for kernel work)
    row = re.search(r"#define HDP_NET_ROW\(X, ny\)(.*)", full).group(1)
    row_km = [(int(k), int(m)) for k, m in re.findall(r"X\(ny, (\d+), (\d+)\)", row)]
    rows = re.findall(r"HDP_NET_ROW\(X, (\d+)\)", re.search(r"#define HDP_NET_INSTANCES\(X\)(.*)", full).group(1))
    return [(int(ny), k, m) for ny in rows for k, m in row_km]


def test_net_table_covers_every_compiled_instance():
    assert sorted(NET_CASES) == sorted(compiled_net_instances())


@pytest.mark.parametrize("calendar", NET_CALENDARS)
@pytest.mark.parametrize("inst", sorted(NET_CASES))
def test_net_case_reaches_its_instance(inst, calendar):
    years, radius, q, tm_warps = NET_CASES[inst]
    info = thresholds_choice(calendar, years, radius, q)
    assert info[0] == NET and tuple(info[1:4]) == inst, info
    assert info[6] == tm_warps, info
    assert info[5] == radius                                   # the mirrored year-end days (noleap) / the leap-year rows (standard)


# ---------------------------------------------------------------------------------------------------------------- k_scan
# Accumulator registers of k_scan: four definitions per register with 8-bit lanes (seasons of at most 255 days), two with 16-bit
# lanes; the definition count D picks the smallest NG that holds them.
SCAN_NG = {8: (2, 3, 4, 6, 8), 16: (2, 3, 4, 6, 8, 12, 16)}
SCAN_KS = (1, 2, 32)                                           # bit planes of the max_subs counters: max_subs <= 1, <= 3, more
SCAN_FILTER_CONST = ((3, 1), (3, 2))                           # compile-time (LMIN, BMAX): 8-bit lanes, KS = 1, filter on
SCAN_T = 8 * 365


def scan_instances():
    """(lane bits, NG, KS, LMIN, BMAX) of every k_scan instantiation run_scan can launch."""
    out = [(bits, ng, ks, 0, 0) for bits in (8, 16) for ng in SCAN_NG[bits] for ks in SCAN_KS]
    out += [(8, ng, 1, lm, bm) for ng in SCAN_NG[8] for lm, bm in SCAN_FILTER_CONST]
    return out


def scan_seasons(bits):
    """Disjoint season tables of both hemispheres over SCAN_T days: 150-day seasons (8-bit lanes) or 290 / 280-day ones
    (16-bit lanes); the last southern season runs past the end of the series."""
    if bits == 8:
        north = [[y * 365 + 100, y * 365 + 250] for y in range(8)]
        south = [[y * 365 + 280, y * 365 + 430] for y in range(8)]
    else:
        north = [[y * 365 + 10, y * 365 + 300] for y in range(8)]
        south = [[y * 365 + 200, y * 365 + 480] for y in range(8)]
    return north, south


def scan_case(bits, ng, ks, lmin, bmax):
    """Definitions [D, 3] that reach the instantiation (bits, ng, ks, lmin, bmax), and the season tables."""
    per = 4 if bits == 8 else 2
    menu = SCAN_NG[bits]
    i = menu.index(ng)
    lo = (menu[i - 1] * per + 1) if i else 1
    hi = ng * per
    D = hi if ks == 32 else max(lo, hi - 1)                    # full registers, and a last register with a free lane
    rng = np.random.default_rng(1000 * bits + 10 * ng + ks + lmin + 7 * bmax)
    subs_max = {1: 1, 2: 3, 32: 9}[ks]
    if lmin:                                                   # the filter constants: smallest min_duration 3, largest max_break
        l0, b0 = lmin, bmax
    else:                                                      # run-time filter values, or the filter off (a 1-day definition)
        l0, b0 = [(2, 0), (4, 3), (1, 1), (6, 5), (3, 4)][(ng + ks) % 5]
    defs = np.stack([rng.integers(l0, l0 + 5, D), rng.integers(0, b0 + 1, D), rng.integers(0, subs_max + 1, D)], axis=1)
    defs[rng.integers(0, D)] = [l0, b0, subs_max]
    if D > 1:
        defs[rng.integers(0, D)] = [l0 + 1, b0, 0]
    north, south = scan_seasons(bits)
    return defs.astype(np.int32), north, south


def metrics_choice(defs, north, south, T=SCAN_T):
    df = np.ascontiguousarray(defs, np.int32)
    sn, ss = np.ascontiguousarray(north, np.int32).reshape(-1, 2), np.ascontiguousarray(south, np.int32).reshape(-1, 2)
    info = (ctypes.c_int * 7)()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)            # noqa: E731
    rc = _lib.lib().hdp_b200_metrics_kernel_choice(p(df), df.shape[0], p(sn), p(ss), sn.shape[0], T, info)
    return rc, list(info)


@pytest.fixture
def run_filter_on():
    L = _lib.lib()
    L.hdp_b200_metrics_run_filter(1)
    yield
    L.hdp_b200_metrics_run_filter(1)


def test_scan_table_covers_46_instantiations():
    inst = scan_instances()
    assert len(inst) == len(set(inst)) == 46


@pytest.mark.parametrize("inst", scan_instances(), ids=lambda i: "b{}_ng{}_ks{}_f{}{}".format(*i))
def test_scan_case_reaches_its_instantiation(inst, run_filter_on):
    bits, ng, ks, lmin, bmax = inst
    defs, north, south = scan_case(*inst)
    rc, info = metrics_choice(defs, north, south)
    assert rc == 0
    filter_on = int(defs[:, 0].min() >= 2 and defs[:, 0].min() <= 32 and defs[:, 1].max() <= 30)
    assert info == [bits, ng, ks, filter_on, lmin, bmax, 1], (info, defs.tolist())
    if lmin:                                                   # with the filter off the same definitions run the generic code
        _lib.lib().hdp_b200_metrics_run_filter(0)
        assert metrics_choice(defs, north, south)[1] == [bits, ng, ks, 0, 0, 0, 1]


def test_scan_choice_boundaries(run_filter_on):
    defs = [[1, 0, 0], [8000, 0, 0], [1, 0, 0], [8000, 0, 0]]
    assert metrics_choice(defs, [[0, 255]], [[10, 265]])[1][:3] == [8, 2, 1]        # 255 days: 8-bit lanes
    assert metrics_choice(defs, [[0, 256]], [[10, 265]])[1][:3] == [16, 2, 1]       # 256 days: 16-bit lanes
    T = 65700
    assert metrics_choice(defs, [[0, 65535]], [[0, 65535]], T)[0] == 0                 # the longest season the u16 output holds
    assert metrics_choice(defs, [[0, 65536]], [[0, 10]], T)[0] == -2
    assert metrics_choice(defs, [[0, 10], [5, 20], [8, 30]], [[0, 5]])[1][6] == 3     # overlapping seasons: one launch per pass
    assert metrics_choice([[3, 1, 0]] * 33, [[0, 10]], [[0, 10]])[0] == -2            # more definitions than HDP_B200_MAX_DEFINITIONS
    assert metrics_choice([[3, 1, 0]], [[0, 10]], [[0, 10]], -1)[0] == -1
    assert metrics_choice([[8191, 0, 0]], [[0, 10]], [[0, 10]])[0] == -2              # min_duration beyond the look-up tables
