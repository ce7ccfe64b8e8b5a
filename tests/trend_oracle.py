"""The trend statistics of hdp_b200_trend (include/hdp_b200.h) restated with NumPy: the explicit list of valid pairs, one sort of the
slopes, and the median, rank and Mann-Kendall rules of the contract.  Test infrastructure, not part of the product."""
import math

import numpy as np

NAMES = ("slope", "intercept", "slope_low", "slope_high", "mk_s", "mk_var", "mk_p", "n")


def key(v):
    """The order-preserving uint64 key of float64 values (-0.0 before +0.0): the order the contract sorts in."""
    u = np.ascontiguousarray(v, np.float64).view(np.uint64)
    return np.where(u >> np.uint64(63), ~u, u | np.uint64(1 << 63))


def sort(v):
    v = np.asarray(v, np.float64)
    return v[np.argsort(key(v), kind="stable")]


def median(a):
    """a sorted ascending: a[m/2] for odd m, (a[m/2-1] + a[m/2]) * 0.5 for even m"""
    m = a.size
    return float(a[m // 2]) if m % 2 else float((a[m // 2 - 1] + a[m // 2]) * 0.5)


def ranks(N, var, zq):
    """(Rl, Ru) of N slopes: Sen (1968), as scipy.stats.theilslopes, with var divided by 18 (not scaled by 1/18.)"""
    sigma = math.sqrt(max(var, 0.0))
    Ru = min(int(np.rint((N - zq * sigma) / 2)), N - 1)
    Rl = max(int(np.rint((N + zq * sigma) / 2)) - 1, 0)
    return Rl, Ru


def valid_of(y, missing=None):
    y = np.asarray(y)
    if y.dtype == np.uint16:
        return np.ones(y.shape, bool) if missing is None else y != missing
    return np.isfinite(y)


def series(y, zq, missing=None):
    """The eight outputs of one series y[0 .. Y-1] (uint16 or float32), as float64."""
    idx = np.flatnonzero(valid_of(y, missing))
    v = np.asarray(y)[idx].astype(np.float64)
    n = v.size
    var_tie = (v[:, None] == v[None, :]).sum(1) if n else np.zeros(0, np.int64)
    tie = int(((var_tie - 1) * (2 * var_tie + 5)).sum())
    var = float(n * (n - 1) * (2 * n + 5) - tie) / 18.0
    if n < 2:
        return np.array([np.nan, np.nan, np.nan, np.nan, 0.0, var, np.nan, float(n)])
    i, j = np.triu_indices(n, 1)
    d = v[j] - v[i]
    a = sort(d / (idx[j] - idx[i]).astype(np.float64))
    N = a.size
    slope = median(a)
    intercept = median(sort(v)) - slope * median(idx.astype(np.float64))
    S = int(np.sign(d).sum())
    z = (S - np.sign(S)) / math.sqrt(var) if var > 0 else 0.0
    p = math.erfc(abs(z) * 0.7071067811865476)
    Rl, Ru = ranks(N, var, zq)
    return np.array([slope, intercept, a[Rl], a[Ru], float(S), var, p, float(n)])


def trend_batch(x, zq, missing=None):
    """x [rows, Y, C] -> float64 [8, rows, C]"""
    x = np.asarray(x)
    rows, _, C = x.shape
    out = np.empty((8, rows, C))
    for r in range(rows):
        for c in range(C):
            out[:, r, c] = series(x[r, :, c], zq, missing)
    return out
