"""HWO / HWE (hdp_b200_metrics with HDP_B200_ONSET) by the reference's building blocks: oracle.indicate_hot_days, then
oracle.index_heatwaves (both pinned to the reference), then the first and last day with an id > 0 of every season slice (Python
slice semantics, the slice hw_ts[a:b] that heatwave_frequency counts), 0xFFFF where there is none.  Test infrastructure: nothing
here is part of the product."""
import numpy as np

import oracle

NO_DAY = 0xFFFF


def onset_of_ids(hw, seasons):
    """int64 id series -> uint16 [2, Y]: HWO, HWE of every season hw[a:b] (NumPy's basic slicing is Python's)."""
    out = np.full((2, len(seasons)), NO_DAY, np.uint16)
    for y, (a, b) in enumerate(seasons):
        days = np.flatnonzero(hw[int(a):int(b)] > 0)
        if days.size:
            out[:, y] = days[0], days[-1]
    return out


def onset_batch(measure_tc, thresholds_cdp, doy_map, defs, seasons_north, seasons_south, is_south):
    """uint16 [2, P, D, Y, C]: planes 4 and 5 of the library's u16 output with HDP_B200_ONSET."""
    x = np.asarray(measure_tc, np.float32)
    thr = np.asarray(thresholds_cdp, np.float64)
    T, C = x.shape
    assert np.shape(doy_map) == (T,), "doy_map needs one entry per day of measure_tc [T, C]"
    P = thr.shape[2]
    df = np.asarray(defs, np.int64).reshape(-1, 3)
    sn, ss = np.asarray(seasons_north).reshape(-1, 2), np.asarray(seasons_south).reshape(-1, 2)
    south = np.zeros(C, np.uint8) if is_south is None else np.asarray(is_south)
    out = np.empty((2, P, df.shape[0], sn.shape[0], C), np.uint16)
    for c in range(C):
        seasons = ss if south[c] else sn
        for p in range(P):
            hot = oracle.indicate_hot_days(x[:, c], thr[c, :, p], doy_map)
            for d, (lmin, brk, subs) in enumerate(df):
                out[:, p, d, :, c] = onset_of_ids(oracle.index_heatwaves(hot, lmin, brk, subs), seasons)
    return out


def cold_onset_batch(measure_tc, thresholds_cdp, *args):
    """CSO / CSE: the heatwave result on negated inputs."""
    return onset_batch((-np.asarray(measure_tc, np.float32)).astype(np.float32), -np.asarray(thresholds_cdp, np.float64), *args)


def compound_onset_batch(xa, ta, xb, tb, doy_map, defs, north, south, is_south, cold=False):
    """Compound HWO / HWE by the masked-input construction of tests/test_compound_host.py: percentile p of the compound result is the
    single-measure result of where(M_p, x_a, NaN) against thr_a (negated for cold)."""
    from test_compound_host import compound_mask
    M = compound_mask(xa, ta, xb, tb, doy_map, cold)
    s = -1.0 if cold else 1.0
    planes = []
    for p in range(M.shape[0]):
        ma = np.where(M[p], s * np.asarray(xa, np.float32), np.float32(np.nan)).astype(np.float32)
        planes.append(onset_batch(ma, s * np.asarray(ta)[:, :, p:p + 1], doy_map, defs, north, south, is_south)[:, 0])
    return np.stack(planes, axis=1)
