#!/usr/bin/env python
"""tools/run_cold.py [cells] [reps] [workload ...] - the cold-spell pass next to the heatwave pass on the same synthetic field.

For each workload: thresholds for its percentiles (cmip6_1deg: 0.90 ... 0.99) and for their mirror 1 - q (0.01 ... 0.10), with
the per-kernel CUDA-event times of each; then per-kernel times (k_hot_words, k_scan, k_intensity) of one hdp_b200_intensity call
that also writes the integer metrics, heatwave (high q) and cold-spell (mirrored q, cold=True, swapped season tables) calls
alternated rep by rep; and the mean HWF / CSF behind them, since k_scan's and k_intensity's work grows with the day density.
Prints one JSON object with the card's name and power limit."""
import json, os, subprocess, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hdp_b200 import _core, synth, workloads, _tables as tb

cells = int(sys.argv[1]) if len(sys.argv) > 1 else 0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
names = sys.argv[3:] or ["cmip6_1deg", "wide_sweep"]
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
result = {"device": torch.cuda.get_device_name(), "nvidia_smi": smi[0] if smi else "not read", "reps": reps, "workloads": {}}


def timed(fn):
    """fn() once with kernel timing on: {kernel: ms summed over its launches}."""
    torch.cuda.synchronize()
    _core.timing_enable(True); _core.timing_read()
    fn()
    torch.cuda.synchronize()
    by = {}
    for n, ms in _core.timing_read():
        by[n] = by.get(n, 0.0) + ms
    _core.timing_enable(False)
    return by


def mean_of(runs):
    keys = sorted({k for r in runs for k in r})
    return {k: round(float(np.mean([r.get(k, 0.0) for r in runs])), 3) for k in keys}


for name in names:
    wl = workloads.get(name)
    lat, _ = synth.grid_latitudes(wl.n_lat, wl.n_lon)
    if cells:
        lat = lat[np.linspace(0, wl.cells - 1, cells).astype(np.int64)]
    C = lat.size
    q_warm = np.asarray(wl.percentiles, np.float64)
    q_cold = np.round(1.0 - q_warm[::-1], 12)
    base = synth.gridded_field(lat, wl.base_axis().dayofyr, seed=1234, offset=5.0, device="cuda")
    wt = wl.window_tables()
    thr = {}
    thr_ms = {"warm": [], "cold": []}
    for r in range(reps + 1):                                       # the first round warms up
        for kind, q in (("warm", q_warm), ("cold", q_cold)):
            t = timed(lambda: thr.__setitem__(kind, _core.thresholds_array(base, wt, q)))
            if r:
                thr_ms[kind].append(t)
    del base
    run = synth.gridded_field(lat, wl.run_axis().dayofyr, seed=1235, offset=5.0, trend=4.0, device="cuda")
    st, dm = wl.seasons(), tb.doy_map(wl.run_axis().dayofyr)
    south = torch.as_tensor((lat < 0).astype(np.uint8), device="cuda")
    args = {"warm": (dm, wl.defs, st.north, st.south, south), "cold": (dm, wl.defs, st.south, st.north, south)}
    met = heat = None                                               # one pair of output buffers for both directions (wide_sweep: 53 GB)
    mean_f, checksum = {}, {}
    for k in ("warm", "cold"):
        met = _core.metrics_array(run, thr[k], *args[k], out=met, cold=k == "cold")
        heat = _core.intensity_array(run, thr[k], *args[k], out=heat, metrics_out=met, cold=k == "cold")
        mean_f[k] = round(float(met[0].double().mean()), 3)
        checksum[k] = float(heat[0].double().sum())
    pass_ms = {"warm": [], "cold": []}
    for _ in range(reps):
        for k in ("warm", "cold"):
            pass_ms[k].append(timed(lambda: _core.intensity_array(run, thr[k], *args[k], out=heat, metrics_out=met, cold=k == "cold")))
    season_days = {k: round(float(np.mean([b - a for a, b in np.concatenate([args[k][2], args[k][3]])])), 1) for k in args}
    result["workloads"][name] = {
        "cells": C, "T": run.shape[0], "P": q_warm.size, "D": len(wl.defs), "Y": st.n_years,
        "q_warm": q_warm.round(4).tolist(), "q_cold": q_cold.round(4).tolist(),
        "thresholds_kernel_ms": {k: mean_of(v) for k, v in thr_ms.items()},
        "intensity_call_kernel_ms": {k: mean_of(v) for k, v in pass_ms.items()},
        "mean_HWF_CSF_days_per_season": mean_f,
        "mean_season_days": season_days,
        "checksum_HWC_CSC": checksum,
    }
    del thr, met, heat, run
    _core.release_workspaces()
    torch.cuda.empty_cache()

print(json.dumps(result, indent=1))
