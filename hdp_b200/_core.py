"""Array-level API over the C ABI: torch CUDA tensors (device memory + streams) in, tensors out.

These are the two seams of the reference that the CUDA library replaces:

* :func:`thresholds_array`  <- ``compute_percentiles`` gufunc + its per-block wrapper
  (reference hdp/threshold.py:52-93)
* :func:`metrics_array`     <- ``compute_heatwave_metrics`` + the percentile x definition sweep
  (reference hdp/metric.py:304-369)
* :func:`hot_days_array`    <- ``indicate_hot_days`` (reference hdp/metric.py:280-301)
* :func:`intensity_array`   heatwave intensity (HWC, HWI, HWP: cumulative, mean and peak exceedance of the threshold over the
  heatwave days of a season), which the reference does not have; optionally with the four metrics from the same pass
* ``cold=True`` on the metric and intensity calls: cold spells (CSF ... CSA, CSC ... CSP), the same sweep over the days below the
  threshold, which the reference does not have either
* :func:`compound_metrics_array`, :func:`compound_intensity_array`: compound (day-night) heatwaves, the same sweep over the days on
  which two measures (e.g. tmax and tmin) both exceed their own thresholds
* ``onset=True`` on the metric, intensity and compound calls: two more uint16 planes, HWO and HWE, the day of the season of its first
  and last heatwave day (0xFFFF without one)
* :func:`extent_array`: the heatwave spatial extent, the daily weighted number of cells of each region on a heatwave day
* :func:`trend_array`: Theil-Sen slope, its confidence interval and the Mann-Kendall test of every season series of a metric or
  intensity output (or any ``[..., Y, C]`` array)
* :func:`index_heatwaves_array`, :func:`season_metrics_array` <- ``index_heatwaves`` and ``heatwave_frequency`` / ``number`` /
  ``duration`` / ``average`` (reference hdp/metric.py:11-172), the building blocks the hot path never materialises

plus ``*_host`` variants that take NumPy (host) arrays and run the chunked copy/compute pipeline of
the library.  PyTorch is used only for device allocations and the current stream.  All compute happens
in libhdp_b200.so; there is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._tables import WindowTables

METRIC_NAMES = ("HWF", "HWN", "HWD", "HWA")      # plane order of the metric output (reference metric.py:336-340)
INTENSITY_NAMES = ("HWC", "HWI", "HWP")          # plane order of the intensity output
COLD_METRIC_NAMES = ("CSF", "CSN", "CSD", "CSA")  # the same planes of a cold-spell pass (cold=True)
COLD_INTENSITY_NAMES = ("CSC", "CSI", "CSP")
COLD = 0x100                                      # HDP_B200_COLD, OR-ed into the unit code of the metric entry points
ONSET_NAMES = ("HWO", "HWE")                      # planes 4 and 5 of the metric output with onset=True
COLD_ONSET_NAMES = ("CSO", "CSE")
ONSET = 0x200                                     # HDP_B200_ONSET, OR-ed in the same way
NO_DAY = 0xFFFF                                   # HWO / HWE of a season without heatwave days
MAX_REGIONS = 256                                 # HDP_B200_MAX_REGIONS: regions of the extent calls

_workspaces = {}


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("hdp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def _workspace(device, nbytes: int):
    """Per-device scratch tensor, grown on demand (the C ABI never allocates)."""
    torch = _torch()
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        _workspaces.pop(key, None)
        ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def release_workspaces() -> None:
    _workspaces.clear()


def _i32(a) -> np.ndarray:
    a = np.asarray(a)
    if a.size and (a.max() > np.iinfo(np.int32).max or a.min() < np.iinfo(np.int32).min):
        raise ValueError("index table does not fit int32")
    return np.ascontiguousarray(a, dtype=np.int32)


def _hp(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def _check_measure(x, name: str):
    torch = _torch()
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 2):
        raise TypeError(f"{name} must be a 2-D float32 CUDA tensor [T, C] (any strides)")
    if x.numel() and (x.stride(0) < 0 or x.stride(1) < 0):
        raise ValueError(f"{name} must have non-negative strides")


def _strides(x):
    T, C = x.shape
    ld_t = x.stride(0) if T > 1 else max(C, 1)
    ld_c = x.stride(1) if C > 1 else 1
    return int(ld_t), int(ld_c)


def _unit_code(units) -> int:
    """``units`` of the samples handed to the kernels: they are converted to Celsius as they are loaded (the unit step of
    format_standard_measures, reference hdp/measure.py:136-149, fused into the load stage)."""
    if units is None:
        return 0
    try:
        return TEMPERATURE_UNIT_CODES[units]
    except KeyError:
        raise ValueError(f"units must be one of {sorted(TEMPERATURE_UNIT_CODES)}") from None


def thresholds_array(temps, tables: WindowTables, percentiles: Sequence[float], out=None, units=None):
    """``temps`` f32 ``[T_b, C]`` -> thresholds f64 ``[C, n_doy, P]`` (reference dims (<cells>, doy, percentile)).
    ``units``: 'degC' (default), 'degK' or 'degF' samples - see :func:`_unit_code`."""
    torch = _torch()
    unit = _unit_code(units)
    _check_measure(temps, "temps")
    L = _lib.lib()
    T_b, C = temps.shape
    q = np.ascontiguousarray(percentiles, dtype=np.float64).ravel()
    ti, wr = _i32(tables.time_index), _i32(tables.win_rows)
    n_doy, n_y, W, P = tables.n_doy, tables.n_y, tables.width, int(q.size)
    ld_t, ld_c = _strides(temps)
    if out is None:
        out = torch.empty((C, n_doy, P), dtype=torch.float64, device=temps.device)
    elif not (out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (C, n_doy, P)):
        raise TypeError("out must be a contiguous float64 CUDA tensor [C, n_doy, P]")
    with torch.cuda.device(temps.device):
        nbytes = L.hdp_b200_thresholds_workspace_bytes(C, T_b, ld_t, ld_c, n_doy, n_y, W, P, unit)
        ws = _workspace(temps.device, nbytes)
        rc = L.hdp_b200_thresholds(temps.data_ptr(), C, T_b, ld_t, ld_c, _hp(ti), _hp(wr), n_doy, n_y, W, _hp(q), P,
                                   out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream, unit)
    _lib.check(rc, "hdp_b200_thresholds")
    return out


def _metric_tables(doy_map, defs, season_north, season_south, T):
    dm = _i32(doy_map).ravel()
    df = _i32(defs).reshape(-1, 3)
    sn, ss = _i32(season_north).reshape(-1, 2), _i32(season_south).reshape(-1, 2)
    if sn.shape != ss.shape:
        raise ValueError("northern and southern season tables must have the same number of rows")
    if dm.size != T:
        raise ValueError("doy_map must have one entry per time step")
    return dm, df, sn, ss


def _check_thr(thr, C):
    torch = _torch()
    if not (isinstance(thr, torch.Tensor) and thr.is_cuda and thr.dtype == torch.float64 and thr.dim() == 3
            and thr.is_contiguous() and thr.shape[0] == C):
        raise TypeError("thresholds must be a contiguous float64 CUDA tensor [C, n_doy, P]")


def _south_tensor(is_south, C, device):
    if is_south is None:
        return None
    torch = _torch()
    south_t = torch.as_tensor(np.ascontiguousarray(is_south, dtype=np.uint8) if not isinstance(is_south, torch.Tensor) else is_south)
    south_t = south_t.to(device=device, dtype=torch.uint8).contiguous()
    if south_t.numel() != C:
        raise ValueError("is_south must have one entry per cell")
    return south_t


def _device_out(out, dtype, shape, device, message):
    torch = _torch()
    if out is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if not (out.is_cuda and out.dtype == dtype and out.is_contiguous() and tuple(out.shape) == shape):
        raise TypeError(message)
    return out


def _names(pairs, name):
    return (name,) if len(pairs) == 1 else (f"{name}_a", f"{name}_b")


def _check_pairs(pairs):
    """(T, C, n_doy, P) of one (measure, thresholds) pair of CUDA tensors, or of the two of a compound call: f32 ``[T, C]`` measures
    of one shape and device, f64 ``[C, n_doy, P]`` thresholds of one shape."""
    for (x, _), name in zip(pairs, _names(pairs, "measure")):
        _check_measure(x, name)
    x0, t0 = pairs[0]
    if any(tuple(x.shape) != tuple(x0.shape) or x.device != x0.device for x, _ in pairs[1:]):
        raise ValueError("measure_a and measure_b must have the same shape [T, C] and device")
    T, C = x0.shape
    for _, thr in pairs:
        _check_thr(thr, C)
    if any(tuple(thr.shape) != tuple(t0.shape) for _, thr in pairs[1:]):
        raise ValueError("thresholds_a and thresholds_b must have the same shape [C, n_doy, P]")
    return T, C, int(t0.shape[1]), int(t0.shape[2])


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _flags(units, cold, onset):
    return _unit_code(units) | (COLD if cold else 0) | (ONSET if onset else 0)


def _check_onset(met, intensity, onset):
    if onset and intensity and met is None:
        raise ValueError("onset=True needs metrics_out: HWO and HWE are planes of the uint16 metric output")


def _metric_pass(pairs, doy_map, defs, season_north, season_south, is_south, units, met, heat, intensity, cold, onset=False):
    """hdp_b200_metrics, or with ``intensity`` hdp_b200_intensity, on one (measure, thresholds) pair of CUDA tensors; hdp_b200_compound
    on two.  ``met`` / ``heat``: the uint16 metrics / float32 intensity output (``[2, 3, P, D, Y, C]`` for two pairs) or None; the
    metrics are allocated unless the intensity pass runs without them.  Returns the intensity output of the intensity pass, else the
    metrics.  ``cold``: the cold-spell pass; ``onset``: the metrics have six planes, HWO and HWE behind the four."""
    torch = _torch()
    _check_onset(met, intensity, onset)
    unit = _flags(units, cold, onset)
    planes = 6 if onset else 4
    T, C, n_doy, P = _check_pairs(pairs)
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south, T)
    L = _lib.lib()
    D, Y = int(df.shape[0]), int(sn.shape[0])
    dev = pairs[0][0].device
    south_t = _south_tensor(is_south, C, dev)
    compound = len(pairs) == 2
    if intensity:
        heat = _device_out(heat, torch.float32, (2, 3, P, D, Y, C) if compound else (3, P, D, Y, C), dev,
                           f"out must be a contiguous float32 CUDA tensor [{'2, ' if compound else ''}3, P, D, Y, C]")
    if met is not None or not intensity:
        met = _device_out(met, torch.uint16, (planes, P, D, Y, C), dev,
                          f"{'metrics_out' if intensity else 'out'} must be a contiguous uint16 CUDA tensor [{planes}, P, D, Y, C]")
    tables = (_hp(dm), _hp(df), D, _hp(sn), _hp(ss), Y, _ptr(south_t))
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        if compound:
            name = "hdp_b200_compound"
            (xa, ta), (xb, tb) = pairs
            (ld_ta, ld_ca), (ld_tb, ld_cb) = _strides(xa), _strides(xb)
            ws = _workspace(dev, L.hdp_b200_compound_workspace_bytes(C, T, ld_ca, ld_cb, n_doy, P, D, Y, _hp(dm)))
            rc = L.hdp_b200_compound(xa.data_ptr(), ld_ta, ld_ca, xb.data_ptr(), ld_tb, ld_cb, C, T, ta.data_ptr(), tb.data_ptr(), n_doy,
                                     P, *tables, _ptr(met), _ptr(heat), ws.data_ptr(), ws.numel(), stream, unit)
        else:
            name = "hdp_b200_intensity" if intensity else "hdp_b200_metrics"
            (x, thr), = pairs
            ld_t, ld_c = _strides(x)
            outs = (heat.data_ptr(), _ptr(met)) if intensity else (met.data_ptr(),)
            ws = _workspace(dev, getattr(L, name + "_workspace_bytes")(C, T, ld_t, ld_c, n_doy, P, D, Y, _hp(dm)))
            rc = getattr(L, name)(x.data_ptr(), C, T, ld_t, ld_c, thr.data_ptr(), n_doy, P, *tables, *outs, ws.data_ptr(), ws.numel(),
                                  stream, unit)
    _lib.check(rc, name)
    return heat if intensity else met


def metrics_array(measure, thresholds, doy_map, defs, season_north, season_south, is_south=None, out=None, units=None, *,
                  cold=False, onset=False):
    """``measure`` f32 ``[T, C]``, ``thresholds`` f64 ``[C, n_doy, P]`` -> uint16 ``[4, P, D, Y, C]``
    (planes HWF, HWN, HWD, HWA; the reference's int64 ``[P, D, C, 4, Y]`` is ``out.permute(1, 2, 4, 0, 3)`` widened).
    ``units`` of the measure's samples as for :func:`thresholds_array`.  ``cold=True``: cold spells - the same rules over the
    days with ``measure < threshold``, planes CSF, CSN, CSD, CSA (the season tables are used as given; the cold season of a
    hemisphere is usually the other one's warm season).  ``onset=True``: uint16 ``[6, P, D, Y, C]``, planes 4 and 5 HWO and HWE
    (CSO, CSE): the day of the season (0 = its first day) of its first and last heatwave day, :data:`NO_DAY` where HWF is 0."""
    return _metric_pass([(measure, thresholds)], doy_map, defs, season_north, season_south, is_south, units, out, None, False, cold,
                        onset)


def intensity_array(measure, thresholds, doy_map, defs, season_north, season_south, is_south=None, out=None, metrics_out=None,
                    units=None, *, cold=False, onset=False):
    """Heatwave intensity: ``measure`` f32 ``[T, C]``, ``thresholds`` f64 ``[C, n_doy, P]`` -> float32 ``[3, P, D, Y, C]``, planes
    HWC (cumulative), HWI (mean) and HWP (peak) exceedance ``measure - threshold`` over the heatwave days of every season (the
    days HWF counts; 0 where there are none).  ``metrics_out``: an optional uint16 CUDA tensor ``[4, P, D, Y, C]`` that also
    receives exactly what :func:`metrics_array` returns, from the same pass.  The non-empty seasons of each hemisphere's table must
    be disjoint (every table compute_hemisphere_ranges builds is).  ``cold=True``: CSC, CSI, CSP - the deficit
    ``threshold - measure`` over the cold-spell days (and CSF ... CSA in ``metrics_out``), see :func:`metrics_array`.  ``onset=True``:
    ``metrics_out`` (required) is ``[6, P, D, Y, C]`` with HWO and HWE, as for :func:`metrics_array`."""
    return _metric_pass([(measure, thresholds)], doy_map, defs, season_north, season_south, is_south, units, metrics_out, out, True,
                        cold, onset)


def compound_metrics_array(measure_a, thresholds_a, measure_b, thresholds_b, doy_map, defs, season_north, season_south, is_south=None,
                           out=None, units=None, *, cold=False, onset=False):
    """Compound heatwaves: :func:`metrics_array` over the days on which BOTH ``measure_a > thresholds_a`` and
    ``measure_b > thresholds_b`` (e.g. tmax and tmin: hot days and hot nights) -> uint16 ``[4, P, D, Y, C]``.  The two measures are
    f32 ``[T, C]`` CUDA tensors (any strides each), the two thresholds f64 ``[C, n_doy, P]`` of the same shape: percentile p of A is
    paired with percentile p of B.  ``units`` applies to both measures; ``cold=True``: days on which both are below their
    thresholds (CSF ... CSA); ``onset=True``: ``[6, P, D, Y, C]`` with HWO and HWE of the compound days."""
    return _metric_pass([(measure_a, thresholds_a), (measure_b, thresholds_b)], doy_map, defs, season_north, season_south, is_south,
                        units, out, None, False, cold, onset)


def compound_intensity_array(measure_a, thresholds_a, measure_b, thresholds_b, doy_map, defs, season_north, season_south, is_south=None,
                             out=None, metrics_out=None, units=None, *, cold=False, onset=False):
    """Intensity of the compound heatwaves of :func:`compound_metrics_array`: float32 ``[2, 3, P, D, Y, C]``, block 0 = HWC, HWI, HWP
    of measure A (its exceedance ``measure_a - thresholds_a`` over the compound heatwave days, as :func:`intensity_array` computes
    it), block 1 = the same for measure B.  ``metrics_out``: an optional uint16 CUDA tensor ``[4, P, D, Y, C]`` that also receives
    what :func:`compound_metrics_array` returns, from the same pass.  ``cold``: the deficits over the compound cold spells.
    ``onset=True``: ``metrics_out`` (required) is ``[6, P, D, Y, C]``."""
    return _metric_pass([(measure_a, thresholds_a), (measure_b, thresholds_b)], doy_map, defs, season_north, season_south, is_south,
                        units, metrics_out, out, True, cold, onset)


def _hot_days(pairs, doy_map, units=None, cold=False):
    """The hot-day mask uint8 ``[P, T, C]`` of one (measure, thresholds) pair (hdp_b200_hot_days) or the compound mask of two
    (hdp_b200_compound_hot_days)."""
    torch = _torch()
    T, C, n_doy, P = _check_pairs(pairs)
    dm = _i32(doy_map).ravel()
    if dm.size != T:
        raise ValueError("doy_map must have one entry per time step")
    L = _lib.lib()
    dev = pairs[0][0].device
    out = torch.empty((P, T, C), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        if len(pairs) == 2:
            name = "hdp_b200_compound_hot_days"
            (xa, ta), (xb, tb) = pairs
            (ld_ta, ld_ca), (ld_tb, ld_cb) = _strides(xa), _strides(xb)
            ws = _workspace(dev, L.hdp_b200_compound_workspace_bytes(C, T, ld_ca, ld_cb, n_doy, P, 1, 0, _hp(dm)))
            rc = L.hdp_b200_compound_hot_days(xa.data_ptr(), ld_ta, ld_ca, xb.data_ptr(), ld_tb, ld_cb, C, T, ta.data_ptr(), tb.data_ptr(),
                                              n_doy, P, _hp(dm), out.data_ptr(), ws.data_ptr(), ws.numel(), stream,
                                              _unit_code(units) | (COLD if cold else 0))
        else:
            name = "hdp_b200_hot_days"
            (x, thr), = pairs
            ld_t, ld_c = _strides(x)
            ws = _workspace(dev, L.hdp_b200_metrics_workspace_bytes(C, T, ld_t, ld_c, n_doy, P, 1, 0, _hp(dm)))
            rc = L.hdp_b200_hot_days(x.data_ptr(), C, T, ld_t, ld_c, thr.data_ptr(), n_doy, P, _hp(dm), out.data_ptr(), ws.data_ptr(),
                                     ws.numel(), stream)
    _lib.check(rc, name)
    return out


def compound_hot_days_array(measure_a, thresholds_a, measure_b, thresholds_b, doy_map, units=None, *, cold=False):
    """The compound mask of every percentile: uint8 ``[P, T, C]``, 1 where both measures exceed their thresholds (``cold``: are
    below them)."""
    return _hot_days([(measure_a, thresholds_a), (measure_b, thresholds_b)], doy_map, units, cold)


def hot_days_array(measure, thresholds, doy_map):
    """``indicate_hot_days`` for every percentile: uint8 ``[P, T, C]``."""
    return _hot_days([(measure, thresholds)], doy_map)


# ----------------------------------------------------------------------------------------------
# the building blocks of path 2 under the reference's names (reference hdp/metric.py:11-172), csrc/seams.cu
# ----------------------------------------------------------------------------------------------

def index_heatwaves_array(hot, defs):
    """``index_heatwaves`` (reference hdp/metric.py:11-60) for S series x D definitions: ``hot`` bool / uint8 CUDA tensor
    ``[S, T]`` (non-zero = hot day), ``defs`` ``[D, 3]`` -> int64 ``[S, D, T]`` heatwave ids (0 = no heatwave)."""
    torch = _torch()
    if not (isinstance(hot, torch.Tensor) and hot.is_cuda and hot.dim() == 2 and hot.dtype in (torch.uint8, torch.bool)):
        raise TypeError("hot must be a 2-D bool / uint8 CUDA tensor [S, T]")
    hot = hot.contiguous().view(torch.uint8)
    df = _i32(defs).reshape(-1, 3)
    S, T = hot.shape
    D = int(df.shape[0])
    out = torch.empty((S, D, T), dtype=torch.int64, device=hot.device)
    with torch.cuda.device(hot.device):
        rc = _lib.lib().hdp_b200_index_heatwaves(hot.data_ptr(), S, T, _hp(df), D, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "hdp_b200_index_heatwaves")
    return out


def season_metrics_array(hw, season_ranges, want=METRIC_NAMES):
    """``heatwave_frequency`` / ``number`` / ``duration`` / ``average`` (reference hdp/metric.py:63-172) of S id series: ``hw`` int64
    CUDA tensor ``[S, T]`` (ANY ids), ``season_ranges`` ``[Y, 2]`` (Python slice semantics) -> dict of the metrics named in
    ``want``: HWF, HWN, HWD int64 ``[S, Y]``, HWA float64 ``[S, Y]`` (before the truncation of compute_heatwave_metrics)."""
    torch = _torch()
    if not (isinstance(hw, torch.Tensor) and hw.is_cuda and hw.dim() == 2 and hw.dtype == torch.int64):
        raise TypeError("hw must be a 2-D int64 CUDA tensor [S, T]")
    hw = hw.contiguous()
    rng = np.ascontiguousarray(season_ranges, dtype=np.int64).reshape(-1, 2)
    S, T = hw.shape
    Y = int(rng.shape[0])
    d_rng = torch.as_tensor(rng).to(hw.device)
    out = {name: torch.empty((S, Y), dtype=torch.float64 if name == "HWA" else torch.int64, device=hw.device) for name in want}
    ptr = lambda name: out[name].data_ptr() if name in out else None
    with torch.cuda.device(hw.device):
        rc = _lib.lib().hdp_b200_season_metrics(hw.data_ptr(), S, T, d_rng.data_ptr(), Y, ptr("HWF"), ptr("HWN"), ptr("HWD"), ptr("HWA"),
                                                torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "hdp_b200_season_metrics")
    return out


# ----------------------------------------------------------------------------------------------
# hdp.measure's elementwise pre-pass on the device (reference hdp/measure.py:10-94, 183-194)
# ----------------------------------------------------------------------------------------------

def _f32_dense(x, name: str):
    torch = _torch()
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
        raise TypeError(f"{name} must be a contiguous float32 CUDA tensor")
    return x


def _measure_call(fn_name: str, temp, rh, flag, out):
    torch = _torch()
    temp = _f32_dense(temp, "temp")
    if rh is not None:
        rh = _f32_dense(rh, "rh")
        if rh.shape != temp.shape:
            raise ValueError("temp and rh must have the same shape")
    out = torch.empty_like(temp) if out is None else _f32_dense(out, "out")
    if out.shape != temp.shape:
        raise ValueError("out must have the shape of temp")
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    with torch.cuda.device(temp.device):
        if fn_name == "hdp_b200_heat_index":
            rc = L.hdp_b200_heat_index(temp.data_ptr(), rh.data_ptr(), temp.numel(), out.data_ptr(), stream)
        elif fn_name == "hdp_b200_heat_index_measure":
            rc = L.hdp_b200_heat_index_measure(temp.data_ptr(), rh.data_ptr(), temp.numel(), int(flag), out.data_ptr(), stream)
        else:
            rc = L.hdp_b200_to_celsius(temp.data_ptr(), temp.numel(), int(flag), out.data_ptr(), stream)
    _lib.check(rc, fn_name)
    return out


def heat_index_array(temp_f, rh_pct, out=None):
    """``heat_index`` ufunc (reference hdp/measure.py:61-94): degF and % in, degF out, float32, bit-identical."""
    return _measure_call("hdp_b200_heat_index", temp_f, rh_pct, 0, out)


def heat_index_measure_array(temp_c, rh, rh_is_fraction: bool = False, out=None):
    """The ``{name}_hi`` measure of ``format_standard_measures`` (reference hdp/measure.py:183-194) in one pass:
    degC -> degF, heat index against rh (% or g/g), degF -> degC."""
    return _measure_call("hdp_b200_heat_index_measure", temp_c, rh, 1 if rh_is_fraction else 0, out)


TEMPERATURE_UNIT_CODES = {"degC": 0, "C": 0, "degK": 1, "K": 1, "degF": 2, "F": 2}


def to_celsius_array(temp, units: str, out=None):
    """``convert_temp_units`` (reference hdp/measure.py:10-41, 136-149) in float32, like the reference's array arithmetic."""
    return _measure_call("hdp_b200_to_celsius", temp, None, TEMPERATURE_UNIT_CODES[units], out)


# ----------------------------------------------------------------------------------------------
# variants the reference declares but does not implement (hdp/threshold.py:105-110), and the figure deck's reduction
# ----------------------------------------------------------------------------------------------

def thresholds_no_season_array(temps, percentiles: Sequence[float], units=None):
    """``no_season``: one percentile set per cell over the WHOLE baseline -> f64 ``[C, 1, P]`` (day-of-year axis of length 1;
    use ``doy_map = zeros(T)`` with :func:`metrics_array`).  Same kernels, same quantile arithmetic, one pooled window."""
    from ._tables import no_season_tables
    return thresholds_array(temps, no_season_tables(temps.shape[0]), percentiles, units=units)


def fixed_thresholds(n_cells: int, value: float, device="cuda"):
    """``fixed_value``: the same threshold everywhere and all year -> f64 ``[C, 1, 1]`` (``doy_map = zeros(T)``)."""
    torch = _torch()
    return torch.full((int(n_cells), 1, 1), float(value), dtype=torch.float64, device=device)


def weighted_spatial_mean(metrics, weights):
    """``compute_weighted_spatial_mean`` of the reference's figure deck (hdp/graphics/figure.py:14-15) for the metric planes:
    uint16 ``[..., C]`` and per-cell weights (cos(latitude) of every flattened cell) -> float64 ``[...]``."""
    torch = _torch()
    if not (isinstance(metrics, torch.Tensor) and metrics.is_cuda and metrics.dtype == torch.uint16 and metrics.is_contiguous()):
        raise TypeError("metrics must be a contiguous uint16 CUDA tensor [..., C]")
    C = int(metrics.shape[-1])
    w = torch.as_tensor(np.ascontiguousarray(weights, dtype=np.float64) if not isinstance(weights, torch.Tensor) else weights)
    w = w.to(device=metrics.device, dtype=torch.float64).contiguous()
    if w.numel() != C:
        raise ValueError("one weight per cell")
    rows = metrics.numel() // max(C, 1)
    out = torch.empty(metrics.shape[:-1], dtype=torch.float64, device=metrics.device)
    with torch.cuda.device(metrics.device):
        rc = _lib.lib().hdp_b200_weighted_mean(metrics.data_ptr(), rows, C, w.data_ptr(), float(w.sum().item()), out.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "hdp_b200_weighted_mean")
    return out


# ----------------------------------------------------------------------------------------------
# host-buffer variants (NumPy in, NumPy out; the library pipelines H2D / kernels / D2H over cell chunks)
# ----------------------------------------------------------------------------------------------

def _host_measure(x: np.ndarray, name: str):
    x = np.asarray(x)
    if x.dtype != np.float32 or x.ndim != 2:
        raise TypeError(f"{name} must be a 2-D float32 array [T, C]")
    T, C = x.shape
    if any(s % 4 for s in x.strides):                   # not a whole number of elements (views of packed records)
        x = np.ascontiguousarray(x)
    ld_t = x.strides[0] // 4 if T > 1 else max(C, 1)
    ld_c = x.strides[1] // 4 if C > 1 else 1
    if ld_t <= 0 or ld_c <= 0 or (ld_c != 1 and ld_t != 1):   # reversed / broadcast / doubly strided views: one dense copy
        x = np.ascontiguousarray(x)
        ld_t, ld_c = max(C, 1), 1
    return x, int(ld_t), int(ld_c)


# Device-resident copies of thresholds this process computed, so that the reference workflow compute_thresholds ->
# compute_group_metrics does not send them back over PCIe.  Keyed by the identity of the host array the library itself
# allocated and returned READ-ONLY (nobody can change its contents behind the cache; a writable copy is a different
# array and misses); the entry dies with the array.  Bounded: oldest entries go first.
_resident = {}                       # id(ndarray) -> (weakref, data pointer, shape, device tensor)
RESIDENT_BYTES_MAX = 24 << 30


def _resident_put(host: np.ndarray, dev) -> None:
    import weakref
    key = id(host)
    _resident[key] = (weakref.ref(host, lambda _r, k=key: _resident.pop(k, None)), host.ctypes.data, host.shape, dev)
    total = sum(e[3].numel() * 8 for e in _resident.values())
    for k in list(_resident):
        if total <= RESIDENT_BYTES_MAX or k == key:
            continue
        total -= _resident[k][3].numel() * 8
        del _resident[k]


def resident_thresholds(thr: np.ndarray):
    """The device copy of ``thr`` if ``thr`` is (a same-shape contiguous view of) an array :func:`thresholds_host` returned."""
    root = thr
    while isinstance(getattr(root, "base", None), np.ndarray):
        root = root.base
    e = _resident.get(id(root))
    if e is None or e[0]() is not root or root.flags.writeable:
        return None
    if thr.ctypes.data != e[1] or tuple(thr.shape) != tuple(e[2]) or not thr.flags.c_contiguous:
        return None
    return e[3]


def release_resident() -> None:
    _resident.clear()


def thresholds_host(temps: np.ndarray, tables: WindowTables, percentiles: Sequence[float], out: Optional[np.ndarray] = None,
                    keep=None, units=None) -> np.ndarray:
    """Host arrays in, host array out (chunked copy/compute pipeline inside the library).  ``keep``: a float64 CUDA tensor
    ``[C, n_doy, P]`` that also receives the thresholds, or True to let the library allocate one and remember it for the
    metric pass (the returned array is then read-only, see :func:`resident_thresholds`)."""
    torch = _torch()
    L = _lib.lib()
    temps, ld_t, ld_c = _host_measure(temps, "temps")
    T_b, C = temps.shape
    q = np.ascontiguousarray(percentiles, dtype=np.float64).ravel()
    ti, wr = _i32(tables.time_index), _i32(tables.win_rows)
    remember = keep is True and out is None
    if keep is True:
        keep = torch.empty((C, tables.n_doy, q.size), dtype=torch.float64, device="cuda") if remember else None
    if keep is not None and not (keep.is_cuda and keep.dtype == torch.float64 and keep.is_contiguous()
                                 and tuple(keep.shape) == (C, tables.n_doy, q.size)):
        raise TypeError("keep must be a contiguous float64 CUDA tensor [C, n_doy, P]")
    if out is None:
        out = np.empty((C, tables.n_doy, q.size), np.float64)
    assert out.flags.c_contiguous and out.dtype == np.float64 and out.shape == (C, tables.n_doy, q.size)
    rc = L.hdp_b200_thresholds_host(_hp(temps), C, T_b, ld_t, ld_c, _hp(ti), _hp(wr), tables.n_doy, tables.n_y,
                                    tables.width, _hp(q), int(q.size), _hp(out), keep.data_ptr() if keep is not None else None,
                                    _unit_code(units))
    _lib.check(rc, "hdp_b200_thresholds_host")
    if remember:
        out.flags.writeable = False
        _resident_put(out, keep)
    return out


def _host_out(out, dtype, shape, message):
    if out is None:
        return np.empty(shape, dtype)
    if not (isinstance(out, np.ndarray) and out.flags.c_contiguous and out.dtype == dtype and out.shape == shape):
        raise TypeError(message)
    return out


def _host_thresholds(thresholds, C):
    """(host array or None, device tensor or None) of one threshold argument of a host call: a CUDA tensor is used where it is, a
    host array that :func:`thresholds_host` returned with ``keep=True`` through its device copy."""
    torch = _torch()
    if isinstance(thresholds, torch.Tensor):
        _check_thr(thresholds, C)
        return None, thresholds
    thr = np.ascontiguousarray(thresholds, dtype=np.float64)
    if thr.ndim != 3 or thr.shape[0] != C:
        raise TypeError("thresholds must be float64 [C, n_doy, P]")
    return thr, resident_thresholds(thr)


def _metric_pass_host(pairs, doy_map, defs, season_north, season_south, is_south, units, met, heat, intensity, cold, onset=False):
    """:func:`_metric_pass` with host arrays: hdp_b200_metrics_host or hdp_b200_intensity_host on one (measure, thresholds) pair,
    hdp_b200_compound_host on two; each threshold as for :func:`metrics_host`."""
    _torch()
    _check_onset(met, intensity, onset)
    planes = 6 if onset else 4
    xs = [_host_measure(x, name) for (x, _), name in zip(pairs, _names(pairs, "measure"))]      # (samples, ld_t, ld_c)
    if any(x.shape != xs[0][0].shape for x, _, _ in xs[1:]):
        raise ValueError("measure_a and measure_b must have the same shape [T, C]")
    T, C = xs[0][0].shape
    thrs = [_host_thresholds(thr, C) for _, thr in pairs]                                       # (host, device)
    shapes = [tuple((d if h is None else h).shape) for h, d in thrs]
    if any(shape != shapes[0] for shape in shapes[1:]):
        raise ValueError("thresholds_a and thresholds_b must have the same shape [C, n_doy, P]")
    n_doy, P = int(shapes[0][1]), int(shapes[0][2])
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south, T)
    south = None if is_south is None else np.ascontiguousarray(is_south, dtype=np.uint8)
    D, Y = df.shape[0], sn.shape[0]
    compound = len(pairs) == 2
    if intensity:
        heat = _host_out(heat, np.float32, (2, 3, P, D, Y, C) if compound else (3, P, D, Y, C),
                         f"out must be a C-contiguous float32 array [{'2, ' if compound else ''}3, P, D, Y, C]")
    if met is not None or not intensity:
        met = _host_out(met, np.uint16, (planes, P, D, Y, C),
                        f"{'metrics_out' if intensity else 'out'} must be a C-contiguous uint16 array [{planes}, P, D, Y, C]")
    hp = lambda h: _hp(h) if h is not None else None                # noqa: E731
    tables = (_hp(dm), _hp(df), D, _hp(sn), _hp(ss), Y, hp(south))
    if compound:
        name = "hdp_b200_compound_host"
        ((a, ld_ta, ld_ca), (b, ld_tb, ld_cb)), ((h_a, d_a), (h_b, d_b)) = xs, thrs
        rc = _lib.lib().hdp_b200_compound_host(_hp(a), ld_ta, ld_ca, _hp(b), ld_tb, ld_cb, C, T, hp(h_a), _ptr(d_a), hp(h_b), _ptr(d_b),
                                               n_doy, P, *tables, hp(met), hp(heat), _flags(units, cold, onset))
    else:
        name = "hdp_b200_intensity_host" if intensity else "hdp_b200_metrics_host"
        ((x, ld_t, ld_c),), ((h_thr, d_thr),) = xs, thrs
        outs = (_hp(heat), hp(met)) if intensity else (_hp(met),)
        rc = getattr(_lib.lib(), name)(_hp(x), C, T, ld_t, ld_c, hp(h_thr), _ptr(d_thr), n_doy, P, *tables, *outs,
                                       _flags(units, cold, onset))
    _lib.check(rc, name)
    return heat if intensity else met


def compound_metrics_host(measure_a: np.ndarray, thresholds_a, measure_b: np.ndarray, thresholds_b, doy_map, defs, season_north,
                          season_south, is_south=None, out: Optional[np.ndarray] = None, units=None, *, cold=False,
                          onset=False) -> np.ndarray:
    """Host-array counterpart of :func:`compound_metrics_array` (both measures' cells of a chunk cross PCIe once).  Each threshold
    as for :func:`metrics_host`: a host array, a CUDA tensor, or a resident copy."""
    return _metric_pass_host([(measure_a, thresholds_a), (measure_b, thresholds_b)], doy_map, defs, season_north, season_south, is_south,
                             units, out, None, False, cold, onset)


def compound_intensity_host(measure_a: np.ndarray, thresholds_a, measure_b: np.ndarray, thresholds_b, doy_map, defs, season_north,
                            season_south, is_south=None, out: Optional[np.ndarray] = None, metrics_out: Optional[np.ndarray] = None,
                            units=None, *, cold=False, onset=False) -> np.ndarray:
    """Host-array counterpart of :func:`compound_intensity_array`: float32 ``[2, 3, P, D, Y, C]``."""
    return _metric_pass_host([(measure_a, thresholds_a), (measure_b, thresholds_b)], doy_map, defs, season_north, season_south, is_south,
                             units, metrics_out, out, True, cold, onset)


def metrics_host(measure: np.ndarray, thresholds, doy_map, defs, season_north, season_south,
                 is_south=None, out: Optional[np.ndarray] = None, units=None, *, cold=False, onset=False) -> np.ndarray:
    """``thresholds``: float64 ``[C, n_doy, P]`` as a host array, or as a CUDA tensor (device-resident: no upload).  A host
    array that :func:`thresholds_host` returned with ``keep=True`` is recognised and its device copy used.  ``cold`` and ``onset`` as
    for :func:`metrics_array`."""
    return _metric_pass_host([(measure, thresholds)], doy_map, defs, season_north, season_south, is_south, units, out, None, False, cold,
                             onset)


def intensity_host(measure: np.ndarray, thresholds, doy_map, defs, season_north, season_south, is_south=None,
                   out: Optional[np.ndarray] = None, metrics_out: Optional[np.ndarray] = None, units=None, *,
                   cold=False, onset=False) -> np.ndarray:
    """Host-array counterpart of :func:`intensity_array`: float32 ``[3, P, D, Y, C]`` (HWC, HWI, HWP); ``metrics_out`` an
    optional uint16 host array ``[4, P, D, Y, C]`` that also receives what :func:`metrics_host` returns (the samples cross PCIe
    once for both).  Thresholds as for :func:`metrics_host` (host array, CUDA tensor, or a resident copy); ``cold`` and ``onset``
    as for :func:`intensity_array`."""
    return _metric_pass_host([(measure, thresholds)], doy_map, defs, season_north, season_south, is_south, units, metrics_out, out, True,
                             cold, onset)


def _extent_cells(weights, regions, n_regions, C):
    """uint32 weights and int32 regions of C cells as contiguous NumPy arrays (None stays None), and the region count."""
    R = int(n_regions)
    if not 1 <= R <= MAX_REGIONS:
        raise ValueError(f"n_regions must be in 1 .. {MAX_REGIONS}")
    w = r = None
    if weights is not None:
        w = np.asarray(weights.cpu() if hasattr(weights, "cpu") else weights).ravel()
        if w.size != C:
            raise ValueError("weights must have one entry per cell")
        if not np.issubdtype(w.dtype, np.integer) or (w.size and (w.min() < 0 or w.max() > 0xFFFFFFFF)):
            raise ValueError("weights must be integers in 0 .. 2**32 - 1")
        w = np.ascontiguousarray(w, dtype=np.uint32)
    if regions is not None:
        r = np.asarray(regions.cpu() if hasattr(regions, "cpu") else regions).ravel()
        if r.size != C:
            raise ValueError("regions must have one entry per cell")
        if not np.issubdtype(r.dtype, np.integer):
            raise ValueError("regions must be integers")
        r = np.ascontiguousarray(np.where((r < 0) | (r >= R), -1, r), dtype=np.int32)     # outside [0, R): in no region
    return w, r, R


def extent_array(measure, thresholds, doy_map, defs, season_north, season_south, is_south=None, weights=None, regions=None, n_regions=1,
                 out=None, metrics_out=None, units=None, *, cold=False):
    """Heatwave spatial extent: ``measure`` f32 ``[T, C]``, ``thresholds`` f64 ``[C, n_doy, P]`` -> int64 ``[R, P, D, T]``, the sum of
    the weights of the cells of region r for which day t is a heatwave day that HWF counts (inside the cell's season, heatwave id >
    0).  ``weights``: integer weights ``[C]`` (uint32; None = 1 each, a cell count); ``regions``: integer region ``[C]`` of every cell
    (None = all in region 0; a value outside ``[0, n_regions)`` = in no region).  The result is ADDED to ``out`` when it is given (a
    contiguous int64 CUDA tensor ``[R, P, D, T]``): the sums are exact, so a loop over cell ranges into one ``out`` gives the result of
    one call.  ``metrics_out``: an optional uint16 CUDA tensor ``[4, P, D, Y, C]`` that also receives what :func:`metrics_array`
    returns, from the same pass.  The non-empty seasons of each hemisphere's table must be disjoint.  ``cold=True``: the cold-spell
    days."""
    torch = _torch()
    unit = _flags(units, cold, False)
    T, C, n_doy, P = _check_pairs([(measure, thresholds)])
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south, T)
    D, Y = int(df.shape[0]), int(sn.shape[0])
    w, r, R = _extent_cells(weights, regions, n_regions, C)
    dev = measure.device
    south_t = _south_tensor(is_south, C, dev)
    w_t = None if w is None else torch.from_numpy(w.view(np.int32)).to(dev)      # (bits of the uint32 weights)
    r_t = None if r is None else torch.from_numpy(r).to(dev)
    if out is None:
        out = torch.zeros((R, P, D, T), dtype=torch.int64, device=dev)
    elif not (out.is_cuda and out.dtype == torch.int64 and out.is_contiguous() and tuple(out.shape) == (R, P, D, T)):
        raise TypeError("out must be a contiguous int64 CUDA tensor [R, P, D, T]")
    if metrics_out is not None:
        metrics_out = _device_out(metrics_out, torch.uint16, (4, P, D, Y, C), dev, "metrics_out must be a contiguous uint16 CUDA tensor "
                                  "[4, P, D, Y, C]")
    L = _lib.lib()
    ld_t, ld_c = _strides(measure)
    with torch.cuda.device(dev):
        ws = _workspace(dev, L.hdp_b200_extent_workspace_bytes(C, T, ld_t, ld_c, n_doy, P, D, Y, R, _hp(dm)))
        rc = L.hdp_b200_extent(measure.data_ptr(), C, T, ld_t, ld_c, thresholds.data_ptr(), n_doy, P, _hp(dm), _hp(df), D, _hp(sn), _hp(ss),
                               Y, _ptr(south_t), _ptr(w_t), _ptr(r_t), R, out.data_ptr(), _ptr(metrics_out), ws.data_ptr(), ws.numel(),
                               torch.cuda.current_stream().cuda_stream, unit)
    _lib.check(rc, "hdp_b200_extent")
    return out


def extent_host(measure: np.ndarray, thresholds, doy_map, defs, season_north, season_south, is_south=None, weights=None, regions=None,
                n_regions=1, out: Optional[np.ndarray] = None, metrics_out: Optional[np.ndarray] = None, units=None, *,
                cold=False) -> np.ndarray:
    """Host-array counterpart of :func:`extent_array` (the pipeline of :func:`metrics_host`): int64 ``[R, P, D, T]`` NumPy out.  ``out``
    is OVERWRITTEN here, not added to.  Thresholds as for :func:`metrics_host` (host array, CUDA tensor, or a resident copy)."""
    _torch()
    x, ld_t, ld_c = _host_measure(measure, "measure")
    T, C = x.shape
    h_thr, d_thr = _host_thresholds(thresholds, C)
    n_doy, P = int((d_thr if h_thr is None else h_thr).shape[1]), int((d_thr if h_thr is None else h_thr).shape[2])
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south, T)
    D, Y = int(df.shape[0]), int(sn.shape[0])
    w, r, R = _extent_cells(weights, regions, n_regions, C)
    south = None if is_south is None else np.ascontiguousarray(is_south, dtype=np.uint8)
    out = _host_out(out, np.int64, (R, P, D, T), "out must be a C-contiguous int64 array [R, P, D, T]")
    if metrics_out is not None:
        metrics_out = _host_out(metrics_out, np.uint16, (4, P, D, Y, C), "metrics_out must be a C-contiguous uint16 array [4, P, D, Y, C]")
    hp = lambda h: _hp(h) if h is not None else None                # noqa: E731
    rc = _lib.lib().hdp_b200_extent_host(_hp(x), C, T, ld_t, ld_c, hp(h_thr), _ptr(d_thr), n_doy, P, _hp(dm), _hp(df), D, _hp(sn), _hp(ss),
                                         Y, hp(south), hp(w), hp(r), R, _hp(out), hp(metrics_out), _flags(units, cold, False))
    _lib.check(rc, "hdp_b200_extent_host")
    return out


def host_release() -> None:
    """Free the streams and device buffers the ``*_host`` entry points keep between calls."""
    release_resident()
    _lib.lib().hdp_b200_host_release()


# ----------------------------------------------------------------------------------------------
# trend statistics of season series (csrc/trend.cu)
# ----------------------------------------------------------------------------------------------

TREND_NAMES = ("slope", "intercept", "slope_low", "slope_high", "mk_s", "mk_var", "mk_p", "n")   # plane order of the trend output
DTYPE_U16, DTYPE_F32 = 1, 2                                      # HDP_B200_DTYPE_U16, HDP_B200_DTYPE_F32
TREND_MAX_Y = 512


def _trend_args(dtype_name: str, shape, missing, alpha):
    """(dtype code, rows, Y, C, missing code, zq) of a trend call on ``[..., Y, C]`` values."""
    if len(shape) < 2:
        raise ValueError("values must be [..., Y, C]")
    if dtype_name == "uint16":
        if missing is not None and not (0 <= int(missing) <= 0xFFFF):
            raise ValueError("missing must be a uint16 value or None")
        code, miss = DTYPE_U16, -1 if missing is None else int(missing)
    elif dtype_name == "float32":
        if missing is not None:
            raise ValueError("missing applies to uint16 values; in float32 values every non-finite value is missing")
        code, miss = DTYPE_F32, -1
    else:
        raise TypeError("values must be uint16 or float32")
    if not 0.0 < alpha < 1.0:
        raise ValueError("alpha must be in (0, 1)")
    from statistics import NormalDist
    zq = NormalDist().inv_cdf(alpha / 2)
    Y, C = int(shape[-2]), int(shape[-1])
    rows = int(np.prod(shape[:-2], dtype=np.int64))
    return code, rows, Y, C, miss, zq


def trend_array(values, *, missing=None, alpha=0.05):
    """Trend of every season series of ``values``, a contiguous uint16 or float32 CUDA tensor ``[..., Y, C]`` (e.g. the metric output
    ``[M, P, D, Y, C]``): float64 ``[8, ..., C]``, planes :data:`TREND_NAMES` - the Theil-Sen slope per season, its intercept at season
    0, the bounds of its Sen (1968) ``1 - alpha`` confidence interval, and the Mann-Kendall S, variance (tie-corrected) and two-sided
    p-value, and the number of valid seasons.  ``missing``: the uint16 value of a missing season (:data:`NO_DAY` for HWO / HWE), or
    None; in float32 values every non-finite value is missing.  Y <= 512.  The exact rules are those of hdp_b200_trend in
    include/hdp_b200.h."""
    torch = _torch()
    if not (isinstance(values, torch.Tensor) and values.is_cuda and values.is_contiguous()):
        raise TypeError("values must be a contiguous uint16 or float32 CUDA tensor [..., Y, C]")
    code, rows, Y, C, miss, zq = _trend_args(str(values.dtype).replace("torch.", ""), tuple(values.shape), missing, alpha)
    out = torch.empty((8, *values.shape[:-2], C), dtype=torch.float64, device=values.device)
    with torch.cuda.device(values.device):
        rc = _lib.lib().hdp_b200_trend(values.data_ptr(), code, rows, Y, C, miss, zq, out.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "hdp_b200_trend")
    return out


TREND_CHUNK_BYTES = 1 << 28


def trend_host(values: np.ndarray, *, missing=None, alpha=0.05) -> np.ndarray:
    """:func:`trend_array` on a host array ``[..., Y, C]`` (uint16 or float32): uploaded in chunks of whole rows (about
    :data:`TREND_CHUNK_BYTES` each), float64 ``[8, ..., C]`` NumPy out."""
    torch = _torch()
    x = np.ascontiguousarray(values)
    code, rows, Y, C, miss, zq = _trend_args(str(x.dtype), x.shape, missing, alpha)
    out = np.empty((8, rows, C), np.float64)
    flat = x.reshape(rows, Y, C)
    step = max(1, TREND_CHUNK_BYTES // max(1, Y * C * x.itemsize))
    for r0 in range(0, rows, step):
        dev = torch.as_tensor(flat[r0:r0 + step]).cuda()
        out[:, r0:r0 + dev.shape[0]] = trend_array(dev, missing=missing, alpha=alpha).cpu().numpy()
    return out.reshape(8, *x.shape[:-2], C)


def launch_count() -> int:
    return int(_lib.lib().hdp_b200_launch_count())


KERNEL_NAMES = {1: "normalize", 2: "k_thr_generic", 3: "k_hot_words", 4: "k_scan", 5: "k_unpack_mask",
                6: "k_thr_seg", 7: "k_thr_ranked", 8: "k_measure", 9: "k_thr_cand", 10: "k_thr_net", 11: "k_seam",
                12: "k_intensity", 13: "k_hot_pair", 14: "k_trend", 15: "k_extent_prefix"}


def timing_enable(on: bool) -> None:
    """Bracket every kernel launch of the library with CUDA events on its launching stream."""
    _lib.lib().hdp_b200_timing_enable(1 if on else 0)


def timing_read(cap: int = 65536):
    """[(kernel name, milliseconds), ...] of the launches recorded since the last read (waits for them)."""
    ids = (ctypes.c_int * cap)()
    ms = (ctypes.c_float * cap)()
    n = _lib.lib().hdp_b200_timing_read(ids, ms, cap)
    return [(KERNEL_NAMES.get(ids[i], str(ids[i])), float(ms[i])) for i in range(n)]
