#!/usr/bin/env python
"""tools/run_intensity.py [cells] [reps] [workload ...] - the intensity pass (thresholds computed once): per-kernel CUDA-event
times of k_hot_words, k_scan and k_intensity for one hdp_b200_intensity call that also writes the integer metrics, next to the
algorithmic floor of the intensity output; then, for the first workload, the wall time of intensity_host with metrics_out next
to metrics_host alone for one full-size measure.  Prints one JSON object with the card's name and power limit."""
import json, os, subprocess, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hdp_b200 import _core, synth, workloads, _tables as tb

HBM_GBS = 6547.5                      # copy bandwidth measured on a B200 (SURVEY.md section 8d)

cells = int(sys.argv[1]) if len(sys.argv) > 1 else 0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
names = sys.argv[3:] or ["cmip6_1deg", "wide_sweep"]
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
result = {"device": torch.cuda.get_device_name(), "nvidia_smi": smi[0] if smi else "not read", "reps": reps, "workloads": {}}

for i, name in enumerate(names):
    wl = workloads.get(name)
    lat, _ = synth.grid_latitudes(wl.n_lat, wl.n_lon)
    if cells:
        lat = lat[np.linspace(0, wl.cells - 1, cells).astype(np.int64)]
    C = lat.size
    base = synth.gridded_field(lat, wl.base_axis().dayofyr, seed=1234, offset=5.0, device="cuda")
    run = synth.gridded_field(lat, wl.run_axis().dayofyr, seed=1235, offset=5.0, trend=4.0, device="cuda")
    st, dm = wl.seasons(), tb.doy_map(wl.run_axis().dayofyr)
    south = torch.as_tensor((lat < 0).astype(np.uint8), device="cuda")
    thr = _core.thresholds_array(base, wl.window_tables(), wl.percentiles)
    del base
    args = (dm, wl.defs, st.north, st.south, south)
    met = _core.metrics_array(run, thr, *args)
    heat = _core.intensity_array(run, thr, *args, metrics_out=torch.empty_like(met))
    torch.cuda.synchronize()
    _core.timing_enable(True); _core.timing_read()
    for _ in range(reps):
        _core.intensity_array(run, thr, *args, out=heat, metrics_out=met)
    torch.cuda.synchronize()
    by = {}
    for n, ms in _core.timing_read():
        by.setdefault(n, []).append(ms)
    _core.timing_enable(False)
    ms = {k: round(float(np.sum(v)) / reps, 3) for k, v in by.items()}
    T, n_doy, P, D, Y = run.shape[0], thr.shape[1], len(wl.percentiles), len(wl.defs), st.n_years
    b_int = C * (4 * T + 8 * n_doy * P + 12 * Y * P * D)
    floor_ms = b_int / HBM_GBS / 1e6
    entry = {"cells": C, "T": T, "P": P, "D": D, "Y": Y, "kernel_ms_per_measure": ms,
             "B_int_GB": round(b_int / 1e9, 2), "floor_ms_at_6547.5GBs": round(floor_ms, 2),
             "k_intensity_over_floor": round(ms.get("k_intensity", float("nan")) / floor_ms, 1),
             "checksum_HWC": float(heat[0].double().sum())}
    if i == 0:
        x_h = run.cpu().numpy()
        thr_h = thr.cpu().numpy()
        del run
        torch.cuda.empty_cache()
        met_h = np.empty(tuple(met.shape), np.uint16)
        _core.intensity_host(x_h[:, :4096], thr_h[:4096], dm, wl.defs, st.north, st.south, south[:4096].cpu().numpy())   # warm-up
        wall = {}
        for label, fn in (("metrics_host", lambda: _core.metrics_host(x_h, thr_h, *args[:-1], south.cpu().numpy(), out=met_h)),
                          ("intensity_host_with_metrics_out", lambda: _core.intensity_host(x_h, thr_h, *args[:-1], south.cpu().numpy(),
                                                                                           metrics_out=met_h))):
            fn()
            t0 = time.perf_counter()
            fn()
            wall[label] = round(time.perf_counter() - t0, 3)
        entry["host_wall_s_one_measure_pageable"] = wall
        _core.host_release()
    result["workloads"][name] = entry
    del thr, met, heat
    _core.release_workspaces()
    torch.cuda.empty_cache()

print(json.dumps(result, indent=1))
