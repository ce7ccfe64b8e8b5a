"""Heatwave spatial extent (hdp_b200_extent) by the reference's building blocks: oracle.indicate_hot_days, then oracle.index_heatwaves
(both pinned to the reference), then for every cell and season slice hw[a:b] (Python slice semantics, the slice heatwave_frequency
counts) w_c added on the days with an id > 0.  The cold result is this on negated inputs.  Test infrastructure: nothing here is part
of the product."""
import numpy as np

import oracle


def extent_of_ids(hw, seasons, w, row):
    """Adds w to row[t] for every day t of a season slice hw[a:b] with an id > 0."""
    days = np.arange(hw.size)
    for a, b in seasons:
        sl = slice(int(a), int(b))
        row[days[sl][hw[sl] > 0]] += w


def extent_batch(measure_tc, thresholds_cdp, doy_map, defs, seasons_north, seasons_south, is_south, weights=None, regions=None,
                 n_regions=1):
    """int64 [R, P, D, T]: d_ext of one hdp_b200_extent call on zeros."""
    x = np.asarray(measure_tc, np.float32)
    thr = np.asarray(thresholds_cdp, np.float64)
    T, C = x.shape
    P = thr.shape[2]
    df = np.asarray(defs, np.int64).reshape(-1, 3)
    sn, ss = np.asarray(seasons_north).reshape(-1, 2), np.asarray(seasons_south).reshape(-1, 2)
    south = np.zeros(C, np.uint8) if is_south is None else np.asarray(is_south)
    w = np.ones(C, np.int64) if weights is None else np.asarray(weights).astype(np.int64)
    r = np.zeros(C, np.int64) if regions is None else np.asarray(regions).astype(np.int64)
    out = np.zeros((n_regions, P, df.shape[0], T), np.int64)
    for c in range(C):
        if not 0 <= r[c] < n_regions or w[c] == 0:
            continue
        seasons = ss if south[c] else sn
        for p in range(P):
            hot = oracle.indicate_hot_days(x[:, c], thr[c, :, p], doy_map)
            for d, (lmin, brk, subs) in enumerate(df):
                extent_of_ids(oracle.index_heatwaves(hot, lmin, brk, subs), seasons, w[c], out[r[c], p, d])
    return out


def cold_extent_batch(measure_tc, thresholds_cdp, *args, **kw):
    """The cold-spell extent: the heatwave result on negated inputs."""
    return extent_batch((-np.asarray(measure_tc, np.float32)).astype(np.float32), -np.asarray(thresholds_cdp, np.float64), *args, **kw)
