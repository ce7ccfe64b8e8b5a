#!/usr/bin/env python
"""tools/run_compound.py [cells] [reps] - the compound pass next to two single-measure passes, full-size cmip6_1deg by default.

tmax is a seasonal cycle plus a persistent unit-variance anomaly, times 3 degC; tmin is the same cycle 10 degC lower with an anomaly
correlated with tmax's (0.75 a_tmax + 0.66 fresh noise), and the measured correlation of the two anomalies is reported.  Thresholds:
the seasonal cycle of each field plus 3 degC times the normal quantiles of the README percentiles 0.90 ... 0.99.  Per rep,
alternated: one hdp_b200_compound call (integer metrics and both intensity blocks) and, for each measure, one hdp_b200_intensity
call that also writes the integer metrics; per-kernel CUDA-event times of each, the mean compound HWF next to the single-measure
HWF, and the bytes k_hot_pair must move.  Prints one JSON object with the card's name and power limit."""
import json, os, subprocess, sys
import numpy as np
from statistics import NormalDist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hdp_b200 import _core, workloads, _tables as tb

cells = int(sys.argv[1]) if len(sys.argv) > 1 else 0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
w = workloads.get("cmip6_1deg")
C = cells or w.cells
ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
T, P, D = len(ax), len(w.percentiles), len(w.defs)
g = torch.Generator(device="cuda").manual_seed(2015)
doy = torch.as_tensor(ax.dayofyr, device="cuda", dtype=torch.float32)[:, None]
cyc = 10 * torch.sin(2 * np.pi * (doy - 110) / 365)
za = torch.randn((T, C), device="cuda", generator=g)
for t in range(1, 4):                                               # a little persistence: runs of hot days
    za[t:] = 0.5 * za[t:] + 0.5 * za[:-t]
za /= za.std()
zb = 0.75 * za + (1 - 0.75 ** 2) ** 0.5 * torch.randn((T, C), device="cuda", generator=g)
rho = float(torch.corrcoef(torch.stack([za[:, ::97].flatten(), zb[:, ::97].flatten()]))[0, 1])
xa = (25 + cyc + 3 * za).float().contiguous()
xb = (15 + cyc + 3 * zb).float().contiguous()
del za, zb
qz = torch.tensor([NormalDist().inv_cdf(float(q)) for q in w.percentiles], device="cuda", dtype=torch.float64)
cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
ta = (25 + cyc_d[None, :, None] + 3 * qz[None, None, :]).expand(C, 365, P).contiguous()
tbh = (15 + cyc_d[None, :, None] + 3 * qz[None, None, :]).expand(C, 365, P).contiguous()
st = tb.hemisphere_ranges(ax)
is_south = ((np.arange(C) // w.n_lon) < w.n_lat // 2).astype(np.uint8)
args = (tb.doy_map(ax.dayofyr), w.defs, st.north, st.south, is_south)
Y = len(st.north)
met = torch.empty((4, P, D, Y, C), dtype=torch.uint16, device="cuda")
met_a, met_b = torch.empty_like(met), torch.empty_like(met)
heat = torch.empty((2, 3, P, D, Y, C), dtype=torch.float32, device="cuda")
heat_a, heat_b = torch.empty_like(heat[0]), torch.empty_like(heat[0])


def timed(fn):
    torch.cuda.synchronize()
    _core.timing_enable(True); _core.timing_read()
    fn()
    torch.cuda.synchronize()
    by = {}
    for n, ms in _core.timing_read():
        by[n] = by.get(n, 0.0) + ms
    _core.timing_enable(False)
    return by


def compound():
    _core.compound_intensity_array(xa, ta, xb, tbh, *args, out=heat, metrics_out=met)


def singles():
    _core.intensity_array(xa, ta, *args, out=heat_a, metrics_out=met_a)
    _core.intensity_array(xb, tbh, *args, out=heat_b, metrics_out=met_b)


compound(); singles()                                               # warm-up: module loads, workspace growth
runs_c, runs_s = [], []
for _ in range(reps):
    runs_c.append(timed(compound))
    runs_s.append(timed(singles))
mean = lambda runs: {k: round(float(np.mean([r.get(k, 0.0) for r in runs])), 3) for k in sorted({k for r in runs for k in r})}  # noqa: E731
hwf = lambda m: float(m[0].double().mean())                         # noqa: E731
bytes_pair = 2 * 4 * T * C + 2 * 8 * 365 * P * C
result = {
    "device": torch.cuda.get_device_name(), "nvidia_smi": smi[0] if smi else "not read", "reps": reps,
    "workload": "cmip6_1deg", "cells": C, "days": T, "percentiles": P, "definitions": D, "seasons": Y,
    "anomaly_correlation_tmax_tmin": round(rho, 4),
    "mean_hwf": {"compound": round(hwf(met), 4), "tmax": round(hwf(met_a), 4), "tmin": round(hwf(met_b), 4)},
    "kernel_ms_compound_call": mean(runs_c), "kernel_ms_two_single_calls": mean(runs_s),
    "runs_compound": runs_c, "runs_single": runs_s,
    "hot_pair_bytes_without_words": bytes_pair,
}
print(json.dumps(result))
