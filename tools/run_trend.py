#!/usr/bin/env python
"""tools/run_trend.py [cells] [reps] [out.json] - k_trend (hdp_b200_trend) on full-size cmip6_1deg (P 10, D 6, 86 seasons) by default.

One synthetic tmax-like field with a warming trend: a seasonal cycle, a persistent unit-variance anomaly times 3 degC, and 0.03 degC per
year; thresholds the seasonal cycle plus 3 degC times the normal quantiles of the percentiles.  One intensity_array call with onset=True
gives the 6 uint16 metric planes [6, P, D, Y, C] and the 3 float32 intensity planes.  Then, per rep and timed with CUDA events:
  u16    trend_array of planes 0 - 3 (no sentinel) and of planes 4 - 5 (missing 0xFFFF): the two calls of one measure
  f32    trend_array of the 3 intensity planes (non-finite = missing)
  y251   trend_array of a float32 [10, 251, C] field of Poisson counts with a trend and 10 % NaN
with the slope pairs (sum of n(n-1)/2 over the series), pair evaluations (8 radix passes over every pair) per second and the bytes read
and written.  Beside them, labelled CPU: the NumPy oracle's time per series (tests/trend_oracle.py) on this host, for 200 series of each
kind (100 of y251).  Prints one JSON object with the card's name and power limit, and writes it to out.json when given."""
import json
import os
import subprocess
import sys
import time
from statistics import NormalDist

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from hdp_b200 import _core, _tables as tb, workloads  # noqa: E402
from trend_oracle import trend_batch  # noqa: E402

cells = int(sys.argv[1]) if len(sys.argv) > 1 else 0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
out_path = sys.argv[3] if len(sys.argv) > 3 else None
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
base = workloads.get("cmip6_1deg")
C = cells or base.cells
ax = tb.TimeAxis.daily((2015, 1, 1), 31390, "noleap")
T = len(ax)
g = torch.Generator(device="cuda").manual_seed(2015)
doy = torch.as_tensor(ax.dayofyr, device="cuda", dtype=torch.float32)[:, None]
year = torch.as_tensor(ax.year - ax.year[0], device="cuda", dtype=torch.float32)[:, None]
z = torch.randn((T, C), device="cuda", generator=g)
for t in range(1, 4):
    z[t:] = 0.5 * z[t:] + 0.5 * z[:-t]
z /= z.std()
x = (25 + 10 * torch.sin(2 * np.pi * (doy - 110) / 365) + 3 * z + 0.03 * year).float().contiguous()
del z
cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
st = tb.hemisphere_ranges(ax)
is_south = ((np.arange(C) // base.n_lon) < base.n_lat // 2).astype(np.uint8)
q = np.asarray(base.percentiles, np.float64)
zs = torch.as_tensor([NormalDist().inv_cdf(v) for v in q], device="cuda", dtype=torch.float64)
thr = (25 + cyc_d[None, :, None] + 3 * zs[None, None, :]).expand(C, 365, q.size).contiguous()
dm = tb.doy_map(ax.dayofyr)
defs = np.asarray(base.defs)
P, D, Y = q.size, len(defs), len(st.north)
met = torch.empty((6, P, D, Y, C), dtype=torch.uint16, device="cuda")
heat = _core.intensity_array(x, thr, dm, defs, st.north, st.south, is_south, metrics_out=met, onset=True)
del x
torch.cuda.synchronize()

rng = np.random.default_rng(251)
lam = rng.uniform(0.5, 8.0, (10, 1, C)) + 0.01 * np.arange(251)[None, :, None]
f251 = rng.poisson(lam).astype(np.float32)
f251[rng.random(f251.shape) < 0.1] = np.nan
y251 = torch.as_tensor(f251).cuda()

cases = {"u16": [(met[:4], None), (met[4:], _core.NO_DAY)], "f32": [(heat, None)], "y251": [(y251, None)]}


def timed(calls):
    torch.cuda.synchronize()
    _core.timing_enable(True)
    _core.timing_read()
    outs = [_core.trend_array(v, missing=m) for v, m in calls]
    torch.cuda.synchronize()
    ms = sum(t for n, t in _core.timing_read() if n == "k_trend")
    _core.timing_enable(False)
    return ms, outs


result = {"card": smi, "cells": C, "seasons": Y, "P": P, "D": D, "reps": reps, "cases": {}}
for name, calls in cases.items():
    times = []
    for _ in range(reps + 1):                                       # the first call warms up
        ms, outs = timed(calls)
        times.append(ms)
    n = torch.cat([o[7].reshape(-1) for o in outs])
    pairs = int((n * (n - 1) / 2).sum().item())
    series = int(n.numel())
    bytes_in = sum(v.numel() * v.element_size() for v, _ in calls)
    bytes_out = sum(o.numel() * 8 for o in outs)
    best = min(times[1:])
    result["cases"][name] = {
        "k_trend_ms": times[1:], "series": series, "mean_valid_seasons": float(n.double().mean().item()), "slope_pairs": pairs,
        "slope_pairs_per_s": pairs / (best / 1e3), "pair_evaluations_per_s": 8 * pairs / (best / 1e3),
        "bytes_read": bytes_in, "bytes_written": bytes_out, "GB_per_s": (bytes_in + bytes_out) / (best / 1e3) / 1e9,
        "mean_slope": float(torch.nanmean(outs[0][0]).item()), "share_p_below_0.05": float((outs[0][6] < 0.05).double().mean().item()),
    }
    # the NumPy oracle on 200 series of the same data, on this host's CPU
    v, m = calls[0]
    flat = v.reshape(-1, v.shape[-2], v.shape[-1])
    sample = np.ascontiguousarray(flat[:20, :, :10].cpu().numpy())        # 200 series (100 for y251)
    zq = NormalDist().inv_cdf(0.025)
    t0 = time.perf_counter()
    want = trend_batch(sample, zq, m)
    cpu_s = time.perf_counter() - t0
    got = _core.trend_array(torch.as_tensor(sample).cuda(), missing=m).cpu().numpy()
    result["cases"][name]["cpu_oracle_us_per_series"] = cpu_s / (sample.shape[0] * sample.shape[2]) * 1e6
    result["cases"][name]["oracle_sample_equal"] = bool(np.array_equal(np.nan_to_num(got[[0, 1, 2, 3, 4, 5, 7]], nan=-7.0),
                                                                        np.nan_to_num(want[[0, 1, 2, 3, 4, 5, 7]], nan=-7.0)))
line = json.dumps(result)
print(line)
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(line + "\n")
