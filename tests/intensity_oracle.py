"""CPU oracle of the heatwave intensity metrics (HWC, HWI, HWP) - TEST INFRASTRUCTURE, not product code.

Two restatements of the contract in include/hdp_b200.h (hdp_b200_intensity):

* ``intensity_oracle.c`` (built on the unchanged ``oracle/hdp_oracle.c``: its hot-day and ``index_heatwaves`` code), compiled on
  first use into a temporary directory and loaded through ctypes - the checker of the GPU tests;
* :func:`np_intensity`, a NumPy second opinion for small cases, from the id series of ``oracle.index_heatwaves``.
"""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from typing import Optional

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_i64 = ctypes.c_int64
_p = ctypes.c_void_p
_LIB: Optional[ctypes.CDLL] = None


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="hdp_intensity_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libintensity_oracle.so")
        src = os.path.join(HERE, "intensity_oracle.c")
        # the compilers and OpenMP fallback of oracle/build.py
        cmds = [[cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fvisibility=hidden", *omp, "-I", os.path.join(ROOT, "oracle"),
                 "-o", out, src, "-lm"]
                for cc in ("/usr/bin/gcc", shutil.which("gcc"), os.environ.get("CC"), shutil.which("cc")) if cc
                for omp in (["-fopenmp"], [])]
        errors = []
        for cmd in cmds:
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode == 0:
                break
            errors.append(" ".join(cmd) + "\n" + r.stderr)
        else:
            raise RuntimeError("could not build the intensity oracle:\n" + "\n".join(errors))
        L = ctypes.CDLL(out)
        L.hdp_oracle_heatwave_intensity.argtypes = [_p, _p, _p, _i64, _i64, _i64, _i64, _p, _i64, _p]
        L.hdp_oracle_intensity_batch.argtypes = [_p, _i64, _i64, _i64, _i64, _p, _i64, ctypes.c_int, _p, _p, ctypes.c_int,
                                                 _p, _p, _i64, _p, _p, ctypes.c_int]
        _LIB = L
    return _LIB


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_p)


def _c(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


def heatwave_intensity(measure, threshold, doy_map, min_duration, max_break, max_subs, season_ranges) -> np.ndarray:
    """One cell, one definition: -> float32[3, Y] = [HWC, HWI, HWP]."""
    m, th, dm = _c(measure, np.float32), _c(threshold, np.float64), _c(doy_map, np.int64)
    rng = _c(season_ranges, np.int64).reshape(-1, 2)
    out = np.empty((3, rng.shape[0]), np.float32)
    rc = lib().hdp_oracle_heatwave_intensity(_ptr(m), _ptr(th), _ptr(dm), m.size, int(min_duration), int(max_break),
                                             int(max_subs), _ptr(rng), rng.shape[0], _ptr(out))
    assert rc == 0
    return out


def intensity_batch(measure_tc, thresholds_cdp, doy_map, defs, seasons_north, seasons_south, is_south, threads: int = 0) -> np.ndarray:
    """Every (percentile, definition, cell) -> float32 ``[P, D, C, 3, Y]`` (HWC, HWI, HWP), the layout of ``oracle.metrics_batch``."""
    meas = np.asarray(measure_tc)
    assert meas.dtype == np.float32 and meas.ndim == 2
    T, C = meas.shape
    thr = _c(thresholds_cdp, np.float64)
    assert thr.shape[0] == C
    n_doy, P = thr.shape[1], thr.shape[2]
    dm = _c(doy_map, np.int64)
    df = _c(defs, np.int64).reshape(-1, 3)
    sn, ss = _c(seasons_north, np.int64).reshape(-1, 2), _c(seasons_south, np.int64).reshape(-1, 2)
    south = np.zeros(C, np.uint8) if is_south is None else _c(is_south, np.uint8)
    Y = sn.shape[0]
    out = np.empty((P, df.shape[0], C, 3, Y), np.float32)
    ld_t, ld_c = (s // 4 for s in meas.strides)
    rc = lib().hdp_oracle_intensity_batch(_ptr(meas), C, T, ld_t, ld_c, _ptr(thr), n_doy, P, _ptr(dm), _ptr(df), df.shape[0],
                                          _ptr(sn), _ptr(ss), Y, _ptr(south), _ptr(out), threads)
    assert rc == 0
    return out


def np_intensity(measure, threshold, doy_map, min_duration, max_break, max_subs, season_ranges) -> np.ndarray:
    """Second opinion on :func:`heatwave_intensity`, from the id series of ``oracle.index_heatwaves``: -> float32[3, Y]."""
    m = np.asarray(measure, np.float32)
    th = np.asarray(threshold, np.float64)
    dm = np.asarray(doy_map, np.int64)
    with np.errstate(invalid="ignore"):
        hot = m.astype(np.float64) > th[dm]
        e = m.astype(np.float64) - th[dm]
    hw = oracle.index_heatwaves(hot, min_duration, max_break, max_subs)
    T = m.size
    rng = np.asarray(season_ranges, np.int64).reshape(-1, 2)
    out = np.zeros((3, rng.shape[0]), np.float32)
    for y, (a, b) in enumerate(rng):
        lo, hi, _ = slice(int(a), int(b)).indices(T)
        S, days, peak = np.float64(0.0), 0, np.float64(0.0)
        t = lo
        while t < hi:
            if hw[t] <= 0:
                t += 1
                continue
            r = np.float64(0.0)
            while t < hi and hw[t] > 0:                           # one block of consecutive heatwave days
                r = r + e[t]
                peak = max(peak, e[t])
                days += 1
                t += 1
            S = S + r
        out[:, y] = [np.float32(S), np.float32(S / np.float64(days)) if days else np.float32(0.0), np.float32(peak)]
    return out
