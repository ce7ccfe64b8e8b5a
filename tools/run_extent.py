#!/usr/bin/env python
"""tools/run_extent.py [cells] [reps] [out.json] - the heatwave spatial extent (extent_array) against the plain metric pass
(metrics_array), full-size cmip6_1deg (P 10, D 6) and wide_sweep (P 20, D 24) by default.

The field of tools/run_onset.py: a seasonal cycle plus a persistent unit-variance anomaly, times 3 degC; thresholds the seasonal
cycle plus 3 degC times the normal quantiles of the workload's percentiles.  One region, weight 1 per cell (the extent is a cell
count).  Per workload and rep, alternated: one metrics_array call and one extent_array call with metrics_out, each timed twice: as a
whole call (CUDA events around it) and per kernel (the library's per-launch events).  The u16 planes of both must be identical, and
the extent must satisfy its invariant sum_t ext = sum_y,c HWF.  Prints one JSON object with the card's name and power limit, and
writes it to out.json when given."""
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


def per_kernel(fn):
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


def whole(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


result = {"device": torch.cuda.get_device_name(), "nvidia_smi": smi[0] if smi else "not read", "reps": reps, "cells": C, "days": T,
          "seasons": Y, "workloads": {}}
for name in ("cmip6_1deg", "wide_sweep"):
    w = workloads.get(name)
    P, D = len(w.percentiles), len(w.defs)
    qz = torch.tensor([NormalDist().inv_cdf(float(q)) for q in w.percentiles], device="cuda", dtype=torch.float64)
    thr = (25 + cyc_d[None, :, None] + 3 * qz[None, None, :]).expand(C, 365, P).contiguous()
    args = (tb.doy_map(ax.dayofyr), w.defs, st.north, st.south, is_south)
    plain = torch.empty((4, P, D, Y, C), dtype=torch.uint16, device="cuda")
    met = torch.empty((4, P, D, Y, C), dtype=torch.uint16, device="cuda")
    ext = torch.zeros((1, P, D, T), dtype=torch.int64, device="cuda")
    run_plain = lambda: _core.metrics_array(x, thr, *args, out=plain)                       # noqa: E731

    def run_extent():
        ext.zero_()
        _core.extent_array(x, thr, *args, out=ext, metrics_out=met)
    run_plain(), run_extent()                                       # warm-up: module loads, workspace growth
    k_p, k_e, w_p, w_e = [], [], [], []
    for _ in range(reps):
        k_p.append(per_kernel(run_plain))
        k_e.append(per_kernel(run_extent))
        w_p.append(whole(run_plain))
        w_e.append(whole(run_extent))
    assert torch.equal(plain, met), "the u16 planes differ from the call without the extent"
    hwf_total = plain[0].to(torch.int64).sum(dim=(2, 3))
    assert torch.equal(ext[0].sum(dim=-1), hwf_total), "sum over days of the extent != sum of HWF"
    mean = lambda runs: {k: round(float(np.mean([r.get(k, 0.0) for r in runs])), 3) for k in sorted({k for r in runs for k in r})}  # noqa: E731
    mp, me = mean(k_p), mean(k_e)
    share = ext[0].double() / C                                     # [P, D, T]
    result["workloads"][name] = {
        "percentiles": P, "definitions": D,
        "kernel_ms_plain": mp, "kernel_ms_extent": me, "k_scan_ratio": round(me["k_scan"] / mp["k_scan"], 4),
        "call_ms_plain": round(float(np.mean(w_p)), 3), "call_ms_extent": round(float(np.mean(w_e)), 3),
        "call_ratio": round(float(np.mean(w_e) / np.mean(w_p)), 4),
        "runs_kernel_plain": k_p, "runs_kernel_extent": k_e, "runs_call_ms_plain": w_p, "runs_call_ms_extent": w_e,
        "planes_0_3_identical": True, "invariant_sum_t_ext_eq_sum_hwf": True,
        "mean_extent_share": round(float(share.mean()), 5),
        "mean_extent_share_first_percentile_first_definition": round(float(share[0, 0].mean()), 5),
        "max_daily_extent_share": round(float(share.max()), 5),
    }
    del plain, met, ext, thr
    torch.cuda.empty_cache()
    _core.release_workspaces()
print(json.dumps(result))
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(json.dumps(result) + "\n")
