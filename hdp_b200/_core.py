"""Array-level API over the C ABI: torch CUDA tensors (device memory + streams) in, tensors out.

These are the two seams of the reference that the CUDA library replaces:

* :func:`thresholds_array`  <- ``compute_percentiles`` gufunc + its per-block wrapper
  (reference hdp/threshold.py:52-93)
* :func:`metrics_array`     <- ``compute_heatwave_metrics`` + the percentile x definition sweep
  (reference hdp/metric.py:304-369)
* :func:`hot_days_array`    <- ``indicate_hot_days`` (reference hdp/metric.py:280-301)
* :func:`intensity_array`   heatwave intensity (HWC, HWI, HWP: cumulative, mean and peak exceedance of the threshold over the
  heatwave days of a season), which the reference does not have; optionally with the four metrics from the same pass
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


def _metric_tables(doy_map, defs, season_north, season_south):
    dm = _i32(doy_map).ravel()
    df = _i32(defs).reshape(-1, 3)
    sn, ss = _i32(season_north).reshape(-1, 2), _i32(season_south).reshape(-1, 2)
    if sn.shape != ss.shape:
        raise ValueError("northern and southern season tables must have the same number of rows")
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


def _metric_pass(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, met, heat, intensity):
    """hdp_b200_metrics, or with ``intensity`` hdp_b200_intensity, on CUDA tensors.  ``met`` / ``heat``: the uint16 metrics /
    float32 intensity output or None; the metrics are allocated unless the intensity pass runs without them.  Returns the
    intensity output of the intensity pass, else the metrics."""
    torch = _torch()
    unit = _unit_code(units)
    _check_measure(measure, "measure")
    T, C = measure.shape
    _check_thr(thresholds, C)
    n_doy, P = int(thresholds.shape[1]), int(thresholds.shape[2])
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south)
    if dm.size != T:
        raise ValueError("doy_map must have one entry per time step")
    L = _lib.lib()
    D, Y = int(df.shape[0]), int(sn.shape[0])
    south_t = _south_tensor(is_south, C, measure.device)
    if intensity:
        heat = _device_out(heat, torch.float32, (3, P, D, Y, C), measure.device,
                           "out must be a contiguous float32 CUDA tensor [3, P, D, Y, C]")
    if met is not None or not intensity:
        met = _device_out(met, torch.uint16, (4, P, D, Y, C), measure.device,
                          f"{'metrics_out' if intensity else 'out'} must be a contiguous uint16 CUDA tensor [4, P, D, Y, C]")
    outs = (heat.data_ptr(), met.data_ptr() if met is not None else None) if intensity else (met.data_ptr(),)
    name = "hdp_b200_intensity" if intensity else "hdp_b200_metrics"
    ld_t, ld_c = _strides(measure)
    with torch.cuda.device(measure.device):
        nbytes = getattr(L, name + "_workspace_bytes")(C, T, ld_t, ld_c, n_doy, P, D, Y, _hp(dm))
        ws = _workspace(measure.device, nbytes)
        rc = getattr(L, name)(measure.data_ptr(), C, T, ld_t, ld_c, thresholds.data_ptr(), n_doy, P, _hp(dm),
                              _hp(df), D, _hp(sn), _hp(ss), Y, south_t.data_ptr() if south_t is not None else None,
                              *outs, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream, unit)
    _lib.check(rc, name)
    return heat if intensity else met


def metrics_array(measure, thresholds, doy_map, defs, season_north, season_south, is_south=None, out=None, units=None):
    """``measure`` f32 ``[T, C]``, ``thresholds`` f64 ``[C, n_doy, P]`` -> uint16 ``[4, P, D, Y, C]``
    (planes HWF, HWN, HWD, HWA; the reference's int64 ``[P, D, C, 4, Y]`` is ``out.permute(1, 2, 4, 0, 3)`` widened).
    ``units`` of the measure's samples as for :func:`thresholds_array`."""
    return _metric_pass(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, out, None, False)


def intensity_array(measure, thresholds, doy_map, defs, season_north, season_south, is_south=None, out=None, metrics_out=None,
                    units=None):
    """Heatwave intensity: ``measure`` f32 ``[T, C]``, ``thresholds`` f64 ``[C, n_doy, P]`` -> float32 ``[3, P, D, Y, C]``, planes
    HWC (cumulative), HWI (mean) and HWP (peak) exceedance ``measure - threshold`` over the heatwave days of every season (the
    days HWF counts; 0 where there are none).  ``metrics_out``: an optional uint16 CUDA tensor ``[4, P, D, Y, C]`` that also
    receives exactly what :func:`metrics_array` returns, from the same pass.  The non-empty seasons of each hemisphere's table must
    be disjoint (every table compute_hemisphere_ranges builds is)."""
    return _metric_pass(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, metrics_out, out, True)


def hot_days_array(measure, thresholds, doy_map):
    """``indicate_hot_days`` for every percentile: uint8 ``[P, T, C]``."""
    torch = _torch()
    _check_measure(measure, "measure")
    T, C = measure.shape
    _check_thr(thresholds, C)
    L = _lib.lib()
    n_doy, P = int(thresholds.shape[1]), int(thresholds.shape[2])
    dm = _i32(doy_map).ravel()
    if dm.size != T:
        raise ValueError("doy_map must have one entry per time step")
    out = torch.empty((P, T, C), dtype=torch.uint8, device=measure.device)
    ld_t, ld_c = _strides(measure)
    with torch.cuda.device(measure.device):
        nbytes = L.hdp_b200_metrics_workspace_bytes(C, T, ld_t, ld_c, n_doy, P, 1, 0, _hp(dm))
        ws = _workspace(measure.device, nbytes)
        rc = L.hdp_b200_hot_days(measure.data_ptr(), C, T, ld_t, ld_c, thresholds.data_ptr(), n_doy, P, _hp(dm),
                                 out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "hdp_b200_hot_days")
    return out


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


def _metric_pass_host(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, met, heat, intensity):
    """:func:`_metric_pass` with host arrays: hdp_b200_metrics_host, or with ``intensity`` hdp_b200_intensity_host."""
    torch = _torch()
    measure, ld_t, ld_c = _host_measure(measure, "measure")
    T, C = measure.shape
    d_thr = None
    if isinstance(thresholds, torch.Tensor):
        _check_thr(thresholds, C)
        d_thr, thr = thresholds, None
        n_doy, P = int(d_thr.shape[1]), int(d_thr.shape[2])
    else:
        thr = np.ascontiguousarray(thresholds, dtype=np.float64)
        if thr.ndim != 3 or thr.shape[0] != C:
            raise TypeError("thresholds must be float64 [C, n_doy, P]")
        n_doy, P = thr.shape[1], thr.shape[2]
        d_thr = resident_thresholds(thr)
    dm, df, sn, ss = _metric_tables(doy_map, defs, season_north, season_south)
    if dm.size != T:
        raise ValueError("doy_map must have one entry per time step")
    south = None if is_south is None else np.ascontiguousarray(is_south, dtype=np.uint8)
    D, Y = df.shape[0], sn.shape[0]
    if intensity:
        heat = _host_out(heat, np.float32, (3, P, D, Y, C), "out must be a C-contiguous float32 array [3, P, D, Y, C]")
    if met is not None or not intensity:
        met = _host_out(met, np.uint16, (4, P, D, Y, C),
                        f"{'metrics_out' if intensity else 'out'} must be a C-contiguous uint16 array [4, P, D, Y, C]")
    outs = (_hp(heat), _hp(met) if met is not None else None) if intensity else (_hp(met),)
    name = "hdp_b200_intensity_host" if intensity else "hdp_b200_metrics_host"
    rc = getattr(_lib.lib(), name)(_hp(measure), C, T, ld_t, ld_c, _hp(thr) if thr is not None else None,
                                   d_thr.data_ptr() if d_thr is not None else None, n_doy, P, _hp(dm), _hp(df), D, _hp(sn), _hp(ss), Y,
                                   _hp(south) if south is not None else None, *outs, _unit_code(units))
    _lib.check(rc, name)
    return heat if intensity else met


def metrics_host(measure: np.ndarray, thresholds, doy_map, defs, season_north, season_south,
                 is_south=None, out: Optional[np.ndarray] = None, units=None) -> np.ndarray:
    """``thresholds``: float64 ``[C, n_doy, P]`` as a host array, or as a CUDA tensor (device-resident: no upload).  A host
    array that :func:`thresholds_host` returned with ``keep=True`` is recognised and its device copy used."""
    return _metric_pass_host(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, out, None, False)


def intensity_host(measure: np.ndarray, thresholds, doy_map, defs, season_north, season_south, is_south=None,
                   out: Optional[np.ndarray] = None, metrics_out: Optional[np.ndarray] = None, units=None) -> np.ndarray:
    """Host-array counterpart of :func:`intensity_array`: float32 ``[3, P, D, Y, C]`` (HWC, HWI, HWP); ``metrics_out`` an
    optional uint16 host array ``[4, P, D, Y, C]`` that also receives what :func:`metrics_host` returns (the samples cross PCIe
    once for both).  Thresholds as for :func:`metrics_host` (host array, CUDA tensor, or a resident copy)."""
    return _metric_pass_host(measure, thresholds, doy_map, defs, season_north, season_south, is_south, units, metrics_out, out, True)


def host_release() -> None:
    """Free the streams and device buffers the ``*_host`` entry points keep between calls."""
    release_resident()
    _lib.lib().hdp_b200_host_release()


def launch_count() -> int:
    return int(_lib.lib().hdp_b200_launch_count())


KERNEL_NAMES = {1: "normalize", 2: "k_thr_generic", 3: "k_hot_words", 4: "k_scan", 5: "k_unpack_mask",
                6: "k_thr_seg", 7: "k_thr_ranked", 8: "k_measure", 9: "k_thr_cand", 10: "k_thr_net", 11: "k_seam",
                12: "k_intensity"}


def timing_enable(on: bool) -> None:
    """Bracket every kernel launch of the library with CUDA events on its launching stream."""
    _lib.lib().hdp_b200_timing_enable(1 if on else 0)


def timing_read(cap: int = 65536):
    """[(kernel name, milliseconds), ...] of the launches recorded since the last read (waits for them)."""
    ids = (ctypes.c_int * cap)()
    ms = (ctypes.c_float * cap)()
    n = _lib.lib().hdp_b200_timing_read(ids, ms, cap)
    return [(KERNEL_NAMES.get(ids[i], str(ids[i])), float(ms[i])) for i in range(n)]
