"""Daily time axes that are not whole continuous years - test infrastructure, not product code.

Every builder only indexes the fields of a :class:`hdp_b200._tables.TimeAxis` built by ``TimeAxis.date_range``, so the axes are
what a user gets from a calendar-aware time coordinate after ``isel``: model runs that start and end mid-year (``mid``), station
or observational series with missing days (``gappy``), May - September subsets (``summer``).  ``stride_map`` is a day-of-year map
whose words are one day long, and ``scan_word_limit`` / ``intensity_word_limit`` restate how many words k_scan and k_intensity
keep in shared memory (hdp_b200/csrc/metric.cu run_scan, intensity.cu run_intensity)."""
from __future__ import annotations

import numpy as np

from hdp_b200 import _tables as tb


def subset(ax: tb.TimeAxis, keep) -> tb.TimeAxis:
    keep = np.asarray(keep)
    return tb.TimeAxis(ax.year[keep], ax.month[keep], ax.day[keep], ax.dayofyr[keep], ax.calendar)


def mid(calendar: str) -> tb.TimeAxis:
    """Starts and ends mid-year and mid-block.  noleap: 10 July 1961 - 20 March 1991 (30 samples in most rows, 29 from 21 March to
    9 July: -1 pads in 111 rows); standard: 1 March 1964 (a leap year) - 15 January 1995 (31 samples per row)."""
    if calendar == "noleap":
        return tb.TimeAxis.date_range("1961-07-10", "1991-03-20", "noleap")
    return tb.TimeAxis.date_range("1964-03-01", "1995-01-15", calendar)


# what gappy() drops besides the random days: (year offset, month, day) of single dates, and one whole month
GAPPY_DROPS = {"dec31": (4, 12, 31), "jan1": (9, 1, 1), "oct1": (12, 10, 1), "may1": (19, 5, 1)}
GAPPY_MONTH = (6, 8)


def gappy(calendar: str, seed: int = 1, years: int = 30, start: int = 1961) -> tb.TimeAxis:
    """``years`` whole years from 1 January ``start`` without about 1 % of the days (at random), one whole month of one year
    (GAPPY_MONTH), one 31 December and one 1 January (the rows the window wraps through), one 1 October (that year's northern
    season then runs to the next year's 1 October) and, in another year, one 1 May (the season rows shift)."""
    ax = tb.TimeAxis.date_range(f"{start}-01-01", f"{start + years - 1}-12-31", calendar)
    rng = np.random.default_rng(seed)
    keep = rng.random(len(ax)) >= 0.01
    for dy, m, d in GAPPY_DROPS.values():
        keep &= ~((ax.year == start + dy) & (ax.month == m) & (ax.day == d))
    keep &= ~((ax.year == start + GAPPY_MONTH[0]) & (ax.month == GAPPY_MONTH[1]))
    # the dates that shape the season tables stay where GAPPY_DROPS does not remove them, so the tables are the ones described
    for m, d in ((5, 1), (10, 1), (11, 1), (4, 1)):
        keep |= (ax.month == m) & (ax.day == d) & ~np.isin(ax.year, [start + dy for dy, mm, dd in GAPPY_DROPS.values() if (mm, dd) == (m, d)])
    return subset(ax, keep)


def summer(calendar: str, years: int = 30, start: int = 1961) -> tb.TimeAxis:
    """1 May - 30 September of every year."""
    ax = tb.TimeAxis.date_range(f"{start}-01-01", f"{start + years - 1}-12-31", calendar)
    return subset(ax, (ax.month >= 5) & (ax.month <= 9))


def summer_seasons(ax: tb.TimeAxis):
    """Explicit per-year season tables of a summer axis (hemisphere_ranges finds no 1 October there): north = the whole summer
    [1 May, 1 October), south = [1 June, 1 September) of every year."""
    years = np.unique(ax.year)
    north = np.array([[np.flatnonzero(ax.year == y)[0], np.flatnonzero(ax.year == y)[-1] + 1] for y in years])
    south = np.array([[np.flatnonzero((ax.year == y) & (ax.month == 6))[0], np.flatnonzero((ax.year == y) & (ax.month == 9))[0]]
                      for y in years])
    return north, south


def stride_map(T: int, n_doy: int = 365) -> np.ndarray:
    """Day-of-year map (3 t) mod n_doy: no two neighbouring days have consecutive days of year, so every word is one day."""
    return (3 * np.arange(T, dtype=np.int64)) % n_doy


def word_lengths(doy_map) -> np.ndarray:
    """word_length (hdp_b200/csrc/seams.h) replayed: the lengths of the hot-day words the metric pass cuts the series into."""
    dm = np.asarray(doy_map, np.int64)
    T = dm.size
    out = []
    t = 0
    while t < T:
        nb = 1
        while t + nb < T and nb < 32 and dm[t + nb] == dm[t] + nb and (dm[t + nb] & 31) != 0:
            nb += 1
        out.append(nb)
        t += nb
    return np.array(out, np.int64)


def n_words(doy_map) -> int:
    return int(word_lengths(doy_map).size)


def scan_word_limit(defs) -> int:
    """The most words run_scan (metric.cu) launches k_scan for: its shared memory holds 8 warps' queues (3 x 16 x 32 u32 each), the
    definition tables (max min_duration + 2 and max max_break + 2 u32, rounded up to 4) and K + 1 int4 word records, at most
    200 KB."""
    df = np.asarray(defs, np.int64).reshape(-1, 3)
    lut = int(df[:, 0].max()) + 2 + int(df[:, 1].max()) + 2
    fixed = ((8 * 3 * 16 * 32 + lut + 3) & ~3) * 4
    return (200 * 1024 - fixed) // 16 - 1


def intensity_word_limit(D: int) -> int:
    """The most words run_intensity (intensity.cu) launches k_intensity for: K int2 word records (rounded up to 16 bytes) and one
    warp's state (D x 32 x (32-byte IndexState + 24-byte IntensityAcc)) within 200 KB."""
    return (200 * 1024 - D * 32 * 56) // 8
