"""hdp.metric on B200 (reference hdp/metric.py).

Same function names, arguments, output variables, dims ``(percentile, definition, <cells>, time)``, coordinates,
dtypes (int64) and attributes as the reference.  The per-cell / per-percentile / per-definition Python -> Numba calls
(`compute_heatwave_metrics`, metric.py:304-341, swept at :357-369) are replaced by ONE call into libhdp_b200.so that
covers the whole sweep; the per-day heatwave id array is never built.
"""
from __future__ import annotations

import numpy as np

from . import _core, _layout, _tables, xr
from .utils import add_history, get_version, time_axis_of

METRIC_ATTRS = {          # metric.py:473-492
    "HWF": {"units": "heatwave days", "long_name": "Heatwave Frequency",
            "description": "Number of days that fall within heatwave during a heatwave season"},
    "HWD": {"units": "heatwave days", "long_name": "Heatwave Duration",
            "description": "Length of longest heatwave during a heatwave season"},
    "HWN": {"units": "heatwave events", "long_name": "Heatwave Number",
            "description": "Number of distinct heatwaves during a heatwave season"},
    "HWA": {"units": "heatwave events", "long_name": "Heatwave Average",
            "description": "Average length of heatwaves during a heatwave season"},
}

# The opt-in intensity variables (compute_individual_metrics(..., intensity=True)); their units are the measure's.
_EXCEEDANCE = "exceedance e = measure - threshold (float64) on the days that fall within a heatwave during a heatwave season"
INTENSITY_ATTRS = {
    "HWC": {"long_name": "Heatwave Cumulative Intensity",
            "description": f"Sum of the {_EXCEEDANCE}, added heatwave by heatwave in time order; 0 without heatwave days"},
    "HWI": {"long_name": "Heatwave Mean Intensity",
            "description": f"Cumulative intensity divided by the heatwave frequency: mean of the {_EXCEEDANCE}; 0 without heatwave days"},
    "HWP": {"long_name": "Heatwave Peak Intensity",
            "description": f"Largest {_EXCEEDANCE}; 0 without heatwave days"},
}


# ----------------------------------------------------------------------------------------------
# The building blocks under the reference's names (its unit tests import exactly these: hdp/tests/test_index_heatwaves.py,
# test_heatwave_{frequency,number,duration,average}.py).  Host arrays in and out like the Numba functions, computed on the GPU
# (csrc/seams.cu); compute_group_metrics does not go through them - its fused kernels never build the id series.
# ----------------------------------------------------------------------------------------------

def _to_device(a: np.ndarray):
    import torch
    _core._torch()                                                  # raises without a CUDA device: there is no CPU path
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def index_heatwaves(hot_days_ts, min_duration: int, max_break: int, max_subs: int) -> np.ndarray:
    """metric.py:11-60: bool / 0-1 series of hot days -> int64 series of heatwave ids (0 = no heatwave)."""
    hot = np.asarray(hot_days_ts)
    if hot.ndim != 1:
        raise ValueError("hot_days_ts must be one-dimensional")
    hot = (hot != 0).astype(np.uint8)                               # `if hot_days_ts[i]`, metric.py:29
    out = _core.index_heatwaves_array(_to_device(hot[None, :]), [[min_duration, max_break, max_subs]])
    return out[0, 0].cpu().numpy()


def _season_metric(hw_ts, season_ranges, name: str) -> np.ndarray:
    hw = np.asarray(hw_ts)
    if hw.ndim != 1:
        raise ValueError("hw_ts must be one-dimensional")
    rng = np.asarray(season_ranges, dtype=np.int64).reshape(-1, 2)
    if name in ("HWD", "HWA") and rng.shape[0]:
        # a season whose slice hw_ts[a:b] is empty: the reference's np.max / np.mean of nothing raise
        T = hw.size
        lo = np.clip(np.where(rng[:, 0] < 0, rng[:, 0] + T, rng[:, 0]), 0, T)
        hi = np.clip(np.where(rng[:, 1] < 0, rng[:, 1] + T, rng[:, 1]), 0, T)
        if np.any(hi <= lo):
            if name == "HWD":
                raise ValueError("zero-size array to reduction operation maximum which has no identity")
            raise ZeroDivisionError("division by zero")
    out = _core.season_metrics_array(_to_device(hw.astype(np.int64)[None, :]), rng, want=(name,))
    return out[name][0].cpu().numpy()


def heatwave_number(hw_ts, season_ranges) -> np.ndarray:
    """metric.py:63-82 (HWN): distinct non-zero ids in every season slice, int64[Y]."""
    return _season_metric(hw_ts, season_ranges, "HWN")


def heatwave_frequency(hw_ts, season_ranges) -> np.ndarray:
    """metric.py:85-102 (HWF): days with id > 0 in every season slice, int64[Y]."""
    return _season_metric(hw_ts, season_ranges, "HWF")


def heatwave_duration(hw_ts, season_ranges) -> np.ndarray:
    """metric.py:105-137 (HWD): most days carrying one id inside every season slice, int64[Y]."""
    return _season_metric(hw_ts, season_ranges, "HWD")


def heatwave_average(hw_ts, season_ranges) -> np.ndarray:
    """metric.py:140-172 (HWA): mean number of days per id inside every season slice, float64[Y]."""
    return _season_metric(hw_ts, season_ranges, "HWA")


def indicate_hot_days(measure, threshold, doy_map) -> np.ndarray:
    """metric.py:280-301: ``measure[t] > threshold[doy_map[t]]`` (float32 against float64, compared in double; NaN -> False)."""
    m = np.asarray(measure)
    if m.ndim != 1:
        raise ValueError("measure must be one-dimensional")
    m32 = m.astype(np.float32)
    if m.dtype != np.float32 and not np.array_equal(m32.astype(np.float64), m.astype(np.float64), equal_nan=True):
        raise TypeError("measure must be float32 (or exactly representable in it): the device path compares float32 samples")
    thr = np.ascontiguousarray(threshold, dtype=np.float64).reshape(1, -1, 1)
    out = _core.hot_days_array(_to_device(m32.reshape(-1, 1)), _to_device(thr), np.asarray(doy_map))
    return out[0, :, 0].cpu().numpy().astype(bool)


def build_doy_map(times) -> np.ndarray:
    """metric.py:265-277"""
    axis = times if isinstance(times, _tables.TimeAxis) else _tables.TimeAxis.from_datetimes(list(times))
    return _tables.doy_map(axis.dayofyr)


def get_range_indices(times, start: tuple, end: tuple) -> np.ndarray:
    """metric.py:175-209"""
    axis = times if isinstance(times, _tables.TimeAxis) else _tables.TimeAxis.from_datetimes(list(times))
    return _tables.range_indices(axis, start, end)


def compute_hemisphere_ranges(measure):
    """metric.py:212-262: ``int[year, end_points, lat, lon]`` season table, South for lat < 0."""
    axis = time_axis_of(measure)
    st = _tables.hemisphere_ranges(axis)
    lat, lon = np.asarray(xr.coord_values(measure, "lat")), np.asarray(xr.coord_values(measure, "lon"))
    ranges = np.where((lat < 0)[None, None, :, None], st.south[:, :, None, None], st.north[:, :, None, None])
    ranges = np.broadcast_to(ranges, (st.n_years, 2, lat.size, lon.size)).copy()
    return xr.DataArray(ranges, dims=["year", "end_points", "lat", "lon"],
                        coords={"year": st.years, "end_points": ["start", "finish"], "lat": lat, "lon": lon})


def compute_heatwave_metrics(measure, threshold, doy_map, min_duration, max_break, max_subs, season_ranges) -> np.ndarray:
    """Array-level seam of the reference kernel (metric.py:304-341) on the GPU, one cell, one definition:
    float32[t], float64[doy], int[t], 3 ints, int[y, 2] -> int64[4, y] = [HWF, HWN, HWD, HWA]."""
    x = np.ascontiguousarray(measure, dtype=np.float32).reshape(-1, 1)
    thr = np.ascontiguousarray(threshold, dtype=np.float64).reshape(1, -1, 1)
    out = _core.metrics_host(x, thr, doy_map, [[min_duration, max_break, max_subs]], season_ranges, season_ranges)
    return out[:, 0, 0, :, 0].astype(np.int64)


def _year_times(years: np.ndarray, calendar: str):
    if xr.HAVE_XARRAY:                 # pragma: no cover - cftime Jan-1 stamps, metric.py:463-465
        import cftime
        import xarray
        start_ts = cftime.datetime(int(years[0]), 1, 1, calendar=calendar)
        end_ts = cftime.datetime(int(years[-1]), 1, 1, calendar=calendar)
        return xarray.date_range(start_ts, end_ts, periods=years.size, use_cftime=True)
    n = years.size
    return _tables.TimeAxis(np.asarray(years, np.int64), np.ones(n, np.int64), np.ones(n, np.int64), np.ones(n, np.int64), calendar)


# dtype of the metric variables.  The reference's are int64 (hdp/tests/test_workflow.py:57) and so is the default; at CMIP scale that
# widening is 10.7 GB per measure and the largest single cost of the drop-in call (tools/api_e2e.py).  A caller that can live with
# the library's native encoding sets `hdp_b200.metric.METRIC_DTYPE = np.uint16` (values are <= the longest season, < 65536).
METRIC_DTYPE = np.int64


def _widen_int64(a: np.ndarray) -> np.ndarray:
    """uint16 -> int64 of one metric plane ([P, D, Y, C], C-contiguous).  The reference's metrics are int64
    (hdp/tests/test_workflow.py:57); at CMIP scale that is 2.7 GB in and 10.7 GB out per measure, so the widening is split
    over the leading axis across threads (NumPy releases the GIL inside the copy)."""
    out = np.empty(a.shape, dtype=np.int64)
    n = a.shape[0] if a.ndim else 0
    if a.size < (1 << 22) or n < 2:
        np.copyto(out, a, casting="unsafe")
        return out
    import os
    from concurrent.futures import ThreadPoolExecutor
    workers = max(1, min(n, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
    with ThreadPoolExecutor(workers) as pool:
        list(pool.map(lambda i: np.copyto(out[i], a[i], casting="unsafe"), range(n)))
    return out


def _metric_sweep(measure, threshold, hw_definitions, time_axis, doy_map=None, intensity=False):
    """The percentile x definition x cell sweep of compute_heatwave_metrics_wrapper (metric.py:344-369) as ONE library call:
    -> ((uint16 [4, P, D, Y, C], float32 [3, P, D, Y, C] or None), season tables, cell dims, cell shape, P, D).  With
    ``intensity`` the call is the intensity pass, which also returns the intensity metrics."""
    st = _tables.hemisphere_ranges(time_axis)                       # compute_hemisphere_ranges, :410
    if doy_map is None:
        doy_map = _tables.doy_map(time_axis.dayofyr)                # build_doy_map, :413
    x, cell_dims, cell_shape = _layout.to_time_cells(xr.values_of(measure), tuple(measure.dims), require_float32=True)
    south = _tables.is_south(_layout.cell_latitudes(xr.coord_values(measure, "lat"), cell_dims, cell_shape))

    # thresholds [<cells in the measure's order>, doy, percentile] -> [C, n_doy, P]; exact coordinate join like apply_ufunc
    thr_dims = tuple(threshold.dims)
    want = [*cell_dims, "doy", "percentile"]
    if sorted(thr_dims) != sorted(want):
        raise ValueError(f"threshold dims {thr_dims} do not match measure dims {tuple(measure.dims)}")
    for d in cell_dims:
        if not np.array_equal(np.asarray(xr.coord_values(threshold, d)), np.asarray(xr.coord_values(measure, d))):
            raise ValueError(f"cannot align measure and threshold exactly along '{d}'")
    thr_vals = np.transpose(xr.values_of(threshold), [thr_dims.index(d) for d in want]).astype(np.float64, copy=False)
    n_doy, P = thr_vals.shape[-2], thr_vals.shape[-1]
    thr_cdp = np.ascontiguousarray(thr_vals).reshape(-1, n_doy, P)

    defs = np.asarray(hw_definitions, dtype=np.int64).reshape(-1, 3)
    if intensity:
        out = np.empty((4, P, defs.shape[0], st.n_years, x.shape[1]), np.uint16)
        heat = _core.intensity_host(x, thr_cdp, doy_map, defs, st.north, st.south, south, metrics_out=out)   # float32 [3, P, D, Y, C]
    else:
        out, heat = _core.metrics_host(x, thr_cdp, doy_map, defs, st.north, st.south, south), None       # uint16 [4, P, D, Y, C]
    return (out, heat), st, cell_dims, cell_shape, P, defs.shape[0]


def compute_heatwave_metrics_wrapper(measure, threshold, doy_map, hw_definitions):
    """metric.py:344-369: the four metrics of every cell for every percentile and definition as one int64 array with dims
    ``(percentile, definition, <cells>, metric, year)``; ``metric`` = HWF, HWN, HWD, HWA in this order (:336-340)."""
    dm = None if doy_map is None else np.asarray(getattr(doy_map, "values", doy_map))
    (out, _), st, cell_dims, cell_shape, P, D = _metric_sweep(measure, threshold, hw_definitions, time_axis_of(measure), dm)
    data = out.astype(np.int64).transpose(1, 2, 4, 0, 3).reshape(P, D, *cell_shape, 4, st.n_years)
    coords = {"definition": [f"{hw_def[0]}-{hw_def[1]}-{hw_def[2]}" for hw_def in hw_definitions],      # :347-350
              "percentile": np.asarray(xr.coord_values(threshold, "percentile"))}
    return xr.DataArray(data, dims=["percentile", "definition", *cell_dims, "metric", "year"], coords=coords)


def compute_individual_metrics(measure, threshold, hw_definitions: list, include_threshold: bool = True, check_variables: bool = True,
                               *, intensity: bool = False):
    """metric.py:372-506.  ``intensity=True`` adds three float32 variables to the four metrics (which stay identical): HWC, HWI
    and HWP, the cumulative, mean and peak exceedance ``measure - threshold`` over the heatwave days of every season, in the
    measure's units (see hdp_b200_intensity in include/hdp_b200.h for the exact arithmetic).  Same dims and coords as HWF."""
    time_axis = time_axis_of(measure)
    if check_variables:                                             # :393-398
        assert "hdp_type" in threshold.attrs
        assert threshold.attrs["hdp_type"] == "threshold"
        assert threshold.attrs["baseline_variable"] == measure.attrs["baseline_variable"]
        assert threshold.attrs["baseline_calendar"] == time_axis.calendar

    combined_history = ""                                           # :400-408
    if "history" in measure.attrs:
        for entry in measure.attrs["history"].split("\n"):
            if entry != '':
                combined_history += (f"(Measure) {entry}\n")
    if "history" in threshold.attrs:
        for entry in threshold.attrs["history"].split("\n"):
            if entry != '':
                combined_history += (f"(Threshold) {entry}\n")

    (out, heat), st, cell_dims, cell_shape, P, D = _metric_sweep(measure, threshold, hw_definitions, time_axis, intensity=intensity)
    Y = st.n_years

    coords = dict(xr.non_time_coords(measure))
    coords["definition"] = [f"{hw_def[0]}-{hw_def[1]}-{hw_def[2]}" for hw_def in hw_definitions]   # :432
    coords["percentile"] = np.asarray(xr.coord_values(threshold, "percentile"))
    coords["time"] = _year_times(st.years, time_axis.calendar)
    dims = ["percentile", "definition", *cell_dims, "time"]
    data_vars = {}
    for i, name in enumerate(_core.METRIC_NAMES):                   # HWF=0, HWN=1, HWD=2, HWA=3, :454-461
        wide = out[i] if np.dtype(METRIC_DTYPE) == np.uint16 else _widen_int64(out[i]).astype(METRIC_DTYPE, copy=False)   # [P, D, Y, C]
        plane = wide.transpose(0, 1, 3, 2).reshape(P, D, *cell_shape, Y)                # view: no host transposition
        data_vars[name] = xr.DataArray(plane, dims=dims, coords=coords)
    if intensity:
        for i, name in enumerate(_core.INTENSITY_NAMES):            # float32 [P, D, Y, C]
            data_vars[name] = xr.DataArray(heat[i].transpose(0, 1, 3, 2).reshape(P, D, *cell_shape, Y), dims=dims, coords=coords)
    ds = xr.Dataset(data_vars)
    ds.attrs.update({
        "description": f"Heatwave metric dataset generated by Heatwave Diagnostics Package (HDP v{get_version()})",
        "hdp_version": get_version(),
        "hdp_type": "metric"
    })
    for name, attrs in METRIC_ATTRS.items():
        ds[name].attrs.update(attrs)
    if intensity:
        for name, attrs in INTENSITY_ATTRS.items():
            ds[name].attrs.update({"units": measure.attrs["units"], **attrs} if "units" in measure.attrs else attrs)
    xr.set_coord_attrs(ds, "percentile", {"range": "(0, 1)"})
    xr.set_coord_attrs(ds, "definition", {
        "first_number": "Minimum number of consecutively hot days",
        "second_number": "Maximum number of break days after first wave",
        "third_number": "Minimum number of consecutively hot days after the break"
    })
    for variable in ds:
        ds[variable].attrs["history"] = combined_history
        add_history(ds[variable], f"Heatwave metrics generated by HDP v{get_version()}")
    return ds


def compute_group_metrics(measures, thresholds, hw_definitions: list, include_threshold: bool = False, check_variables: bool = True,
                          *, intensity: bool = False):
    """metric.py:509-523: every measure against every threshold of the same baseline variable.  ``intensity=True`` adds the
    HWC / HWI / HWP variables of :func:`compute_individual_metrics` under the same ``{measure}.{threshold}.{metric}`` names."""
    metric_sets = []
    for measure_name in list(measures.keys()):
        measure = measures[measure_name]
        for threshold_name in list(thresholds.keys()):
            threshold = thresholds[threshold_name]
            if threshold.attrs["baseline_variable"] == measure.attrs["baseline_variable"]:
                hw_metrics = compute_individual_metrics(measure, threshold, hw_definitions, include_threshold, check_variables,
                                                        intensity=intensity)
                var_renames = {name: f"{measure_name}.{threshold_name}.{name}" for name in list(hw_metrics.keys())}
                metric_sets.append(hw_metrics.rename(var_renames))
    aggr_ds = xr.merge(metric_sets)
    aggr_ds.attrs["variable_naming_desc"] = "(heat measure).(threshold used).(heatwave metric)"
    aggr_ds.attrs["variable_naming_delimeter"] = "."
    return aggr_ds


def compute_metrics_io(output_path: str, measure_path: str, measure_var: str, threshold_path: str, hw_definitions: list,
                       include_threshold: bool = False, override_threshold_var: str = None, overwrite: bool = False) -> None:
    """hdp/metric.py:526-590: metrics from netCDF files / zarr stores, written back to disk.  The reference's wrapper does not run
    as shipped (``overwrite`` and ``makedirs`` are undefined, ``threshold_var`` is unset when an override is given); this one
    does what it sets out to do (``overwrite`` is the argument the reference forgot to declare).  netCDF / zarr need xarray;
    without it (this image) use :func:`hdp_b200.io.compute_metrics_io`, the same flow on memory-mapped ``.npy`` files."""
    import os
    from pathlib import Path
    output_path, measure_path, threshold_path = Path(output_path), Path(measure_path), Path(threshold_path)
    check_variables = True
    threshold_var = override_threshold_var
    if override_threshold_var is None:                              # :562-564
        threshold_var = f"threshold_{measure_var}"
        check_variables = False
    if output_path.exists() and not overwrite:
        raise FileExistsError(f"Overwrite parameter set to False and file exists at '{output_path}'.")
    if not output_path.parent.exists():
        if overwrite:
            os.makedirs(output_path.parent, exist_ok=True)
        else:
            raise FileExistsError(f"Overwrite parameter set to False and directory '{output_path.parent}' does not exist.")
    if output_path.suffix not in [".zarr", ".nc"]:
        raise ValueError(f"File type '{output_path.suffix}' from '{output_path}' not supported.")
    if not xr.HAVE_XARRAY:
        raise RuntimeError("reading netCDF / zarr needs xarray; hdp_b200.io.compute_metrics_io streams .npy files without it")
    import xarray                                                   # pragma: no cover - no xarray in the build image

    def _open(path, var):                                           # pragma: no cover
        return (xarray.open_zarr(path) if path.suffix == ".zarr" and path.is_dir() else xarray.open_dataset(path))[var]
    metric_ds = compute_individual_metrics(_open(measure_path, measure_var), _open(threshold_path, threshold_var), hw_definitions,
                                           include_threshold=include_threshold, check_variables=check_variables)   # pragma: no cover
    if output_path.suffix == ".zarr":                               # pragma: no cover
        metric_ds.to_zarr(output_path, mode="w" if overwrite else "w-")
    else:                                                           # pragma: no cover
        metric_ds.to_netcdf(output_path)
