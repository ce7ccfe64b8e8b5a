#!/usr/bin/env python
"""tools/run_onset.py [cells] [reps] [out.json] - k_scan with and without HWO / HWE (onset=True), full-size cmip6_1deg (P 10, D 6) and
wide_sweep (P 20, D 24) by default.

One synthetic tmax-like field for both workloads: a seasonal cycle plus a persistent unit-variance anomaly, times 3 degC; thresholds
the seasonal cycle plus 3 degC times the normal quantiles of the workload's percentiles.  Per workload and rep, alternated: one
metrics_array call without the flag and one with it, per-kernel CUDA-event times of each.  Planes 0 - 3 of the two outputs must be
identical.  Also the mean HWO and HWE per hemisphere over the seasons that have a heatwave day (a sanity line: 0 = May 1 in the north,
Nov 1 in the south).  Prints one JSON object with the card's name and power limit, and writes it to out.json when given."""
import json
import os
import subprocess
import sys
from statistics import NormalDist

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from hdp_b200 import _core, _tables as tb, workloads  # noqa: E402

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
z = torch.randn((T, C), device="cuda", generator=g)
for t in range(1, 4):                                               # a little persistence: runs of hot days
    z[t:] = 0.5 * z[t:] + 0.5 * z[:-t]
z /= z.std()
x = (25 + 10 * torch.sin(2 * np.pi * (doy - 110) / 365) + 3 * z).float().contiguous()
del z
cyc_d = 10 * torch.sin(2 * np.pi * (torch.arange(365, device="cuda", dtype=torch.float64) - 110) / 365)
st = tb.hemisphere_ranges(ax)
is_south = ((np.arange(C) // base.n_lon) < base.n_lat // 2).astype(np.uint8)
Y = len(st.north)


def timed(fn):
    torch.cuda.synchronize()
    _core.timing_enable(True)
    _core.timing_read()
    fn()
    torch.cuda.synchronize()
    by = {}
    for n, ms in _core.timing_read():
        by[n] = by.get(n, 0.0) + ms
    _core.timing_enable(False)
    return by


def day_means(plane, south):
    """mean of the u16 plane [P, D, Y, C] over the seasons with a heatwave day, per hemisphere"""
    s = torch.as_tensor(south.astype(bool), device="cuda")
    tot = {"north": [0.0, 0], "south": [0.0, 0]}
    for p in range(plane.shape[0]):
        v = plane[p].view(torch.int16).to(torch.int32) & 0xFFFF
        ok = v != _core.NO_DAY
        for name, m in (("north", ~s), ("south", s)):
            sel = ok & m
            tot[name][0] += float(torch.where(sel, v, 0).double().sum())
            tot[name][1] += int(sel.sum())
    return {k: round(a / max(n, 1), 3) for k, (a, n) in tot.items()}


result = {"device": torch.cuda.get_device_name(), "nvidia_smi": smi[0] if smi else "not read", "reps": reps, "cells": C, "days": T,
          "seasons": Y, "workloads": {}}
for name in ("cmip6_1deg", "wide_sweep"):
    w = workloads.get(name)
    P, D = len(w.percentiles), len(w.defs)
    qz = torch.tensor([NormalDist().inv_cdf(float(q)) for q in w.percentiles], device="cuda", dtype=torch.float64)
    thr = (25 + cyc_d[None, :, None] + 3 * qz[None, None, :]).expand(C, 365, P).contiguous()
    args = (tb.doy_map(ax.dayofyr), w.defs, st.north, st.south, is_south)
    plain = torch.empty((4, P, D, Y, C), dtype=torch.uint16, device="cuda")
    onset = torch.empty((6, P, D, Y, C), dtype=torch.uint16, device="cuda")
    run_plain = lambda: _core.metrics_array(x, thr, *args, out=plain)                       # noqa: E731
    run_onset = lambda: _core.metrics_array(x, thr, *args, out=onset, onset=True)           # noqa: E731
    run_plain(), run_onset()                                        # warm-up: module loads, workspace growth
    runs_p, runs_o = [], []
    for _ in range(reps):
        runs_p.append(timed(run_plain))
        runs_o.append(timed(run_onset))
    assert torch.equal(plain, onset[:4]), "planes 0 - 3 differ from the call without onset"
    mean = lambda runs: {k: round(float(np.mean([r.get(k, 0.0) for r in runs])), 3) for k in sorted({k for r in runs for k in r})}  # noqa: E731
    mp, mo = mean(runs_p), mean(runs_o)
    result["workloads"][name] = {
        "percentiles": P, "definitions": D,
        "kernel_ms_plain": mp, "kernel_ms_onset": mo, "k_scan_ratio": round(mo["k_scan"] / mp["k_scan"], 4),
        "runs_plain": runs_p, "runs_onset": runs_o,
        "mean_hwf": round(float(plain[0].double().mean()), 4),
        "mean_HWO_days": day_means(onset[4], is_south), "mean_HWE_days": day_means(onset[5], is_south),
        "seasons_without_heatwave_day": round(float((onset[4].view(torch.int16) == -1).double().mean()), 4),
    }
    del plain, onset, thr
    torch.cuda.empty_cache()
    _core.release_workspaces()
print(json.dumps(result))
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(json.dumps(result) + "\n")
