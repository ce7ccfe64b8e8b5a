#!/usr/bin/env python
"""bench.py - grid-cell-years/s of the two HDP hot paths (thresholds + heatwave metrics) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--scaling weak|strong]
                    [--dump-outputs DIR]

One "step" = thresholds for every measure of the workload, then the full percentile x definition metric
sweep for every measure (BASELINE.json configs[1]: CMIP6-like 180x360, 30 y + 86 y, 3 measures, 10 x 6).
With N > 1 (torchrun, one rank per GPU) the cells of ONE job are sharded across the ranks with hdp_b200.shard
(contiguous ranges of the flattened cell index, no collective on the data path) and the output gather over
NCCL / NVLink is timed beside it:
    weak   (default)  the job is N ensemble members of the grid, flattened (member, cell); per-GPU work is fixed
    strong            the job is one grid; every rank owns 1/N of its cells
Extra records in the same line: `strong` (N > 1), `lens50` (BASELINE configs[2], N >= 4) and, at N = 1,
`configs` with the other named workloads.  Prints ONE JSON line on rank 0.  DESIGN.md "Measurement" explains every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "grid-cell-years/s (threshold+metric)"
UNIT = "grid-cell-years/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cmip6_1deg")
    ap.add_argument("--cells", type=int, default=0, help="override the number of cells per GPU (debugging only)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="target CPU time per path for the cpu_baseline sample")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="what N > 1 ranks share (see the module docstring)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra records (strong / lens50 / configs)")
    ap.add_argument("--no-gather", action="store_true", help="skip the output gather timing (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (a fixed sample of cells) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference times a CPU sample of other cells")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(label: str, cells: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel(s) in `label`, from the committed ncu
    `--set full` capture of this round (profiles/traffic.json, written by tools/ncu_summary.py), scaled to `cells`."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        k = json.load(f)["kernels"]
    names = [n for n in label.split("+") if n in k]             # (the hand-over pass of k_thr_seg behind k_thr_cand is not captured: ~0 bytes)
    if not names:
        return None
    return sum(k[n]["dram_bytes"] * cells / k[n]["cells"] for n in names)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms.  It is started before the warm-up (nvidia-smi needs a few
    hundred ms to deliver its first line) and `stop(t0, t1)` keeps the samples whose timestamps fall inside the timed region
    [t0, t1] (time.time()); a region shorter than the sampling period falls back to the samples within 0.5 s around it, which
    were taken under the same load (warm-up steps before, end-to-end steps after)."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_id: str):
        self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", gpu_id, f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.file, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self, t0: float, t1: float):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)                                   # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.file.flush()
        self.file.seek(0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in self.file.read().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[1]), float(parts[2]), [n for n, v in zip(names, parts[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        self.file.close()
        os.unlink(self.file.name)
        inside = [r for r in rows if t0 <= r[0] <= t1]
        where = "timed region"
        if not inside:
            inside = [r for r in rows if t0 - 0.5 <= r[0] <= t1 + 0.5]
            where = "within 0.5 s of the timed region (region shorter than the sampling period)"
        if inside:
            out.update(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=float(max(r[2] for r in inside)),
                       reasons=sorted({n for r in inside for n in r[3]}), samples=len(inside), sampled=where)
        return out


# --------------------------------------------------------------------------------------------------
# CPU legs: the reference's own Numba kernels under a process pool (oracle/_ref + oracle/ref_pool.py), else the oracle port
# --------------------------------------------------------------------------------------------------
def host_cores() -> int:
    """Cores this process may run on.  torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs are meant to use every
    host core, so they ask for this many workers / threads explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def bind_to_gpu_numa_node(gpu_id: str):
    """Multi-GPU boxes have several NUMA nodes: run this rank on the cores next to its GPU, so that the pinned host buffers of
    the end-to-end leg are allocated (first touch) in the memory its PCIe root is attached to.  Returns the previous affinity
    (the CPU baseline leg restores it: it is meant to use every host core)."""
    try:
        import pynvml
        previous = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByUUID(gpu_id) if gpu_id.startswith("GPU-") else pynvml.nvmlDeviceGetHandleByIndex(int(gpu_id))
        n_words = (max(previous) + 64) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, n_words)
        cpus = {64 * w + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1} & previous
        if cpus:
            os.sched_setaffinity(0, cpus)
        return previous
    except Exception:                                      # no NVML / no permission: stay where we are
        return None


def cpu_tables(wl):
    from hdp_b200 import _tables as tb
    wt = wl.window_tables()
    if not wl.run_years:
        return wt, None, None
    return wt, tb.doy_map(wl.run_axis().dayofyr), wl.seasons()


def port_pass(wl, base, run, is_south, threads=None):
    """One pass of the oracle port (oracle/hdp_oracle.c, OpenMP over cells) on [T, n] host arrays.
    Returns (seconds thresholds, seconds metrics, thresholds, metrics)."""
    import oracle
    threads = threads or host_cores()
    wt, dm, st = cpu_tables(wl)
    win = wt.window_samples()
    t0 = time.perf_counter()
    thr = oracle.thresholds_batch(base, win, wl.percentiles, threads)
    t1 = time.perf_counter()
    met = None
    if run is not None:
        met = oracle.metrics_batch(run, thr, dm, wl.defs, st.north, st.south, is_south, threads)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, thr, met


def reference_pool():
    """The reference's own Numba kernels, one worker process per host core (None when oracle/_ref is absent)."""
    try:
        from oracle import ref_numba, ref_pool
        if not ref_numba.available():
            return None
        return ref_pool.RefPool(host_cores())
    except Exception as e:                                 # noqa: BLE001 - no numba / spawn failure: fall back to the port
        print(f"reference pool unavailable ({type(e).__name__}: {e}); timing the oracle port instead", file=sys.stderr)
        return None


def reference_pass(pool, wl, base, run, is_south):
    """The same pass through the reference's kernels (hdp/threshold.py:52-93, hdp/metric.py:304-369)."""
    wt, dm, st = cpu_tables(wl)
    thr, t_thr = pool.thresholds(base, wt.window_samples(), wl.percentiles)
    met, t_met = (None, 0.0)
    if run is not None:
        met, t_met = pool.metrics(run, thr, dm, wl.defs, st.north, st.south, is_south)
    return t_thr, t_met, thr, met


SAMPLE_SEED = 1234           # measure 0 of member 0 of the GPU arm: both arms draw their CPU sample from this field


def sample_field(wl, sel, device):
    """Cells `sel` of measure 0 / member 0 of the workload's synthetic field - the very values the GPU arm processes when
    `device` is the GPU (torch's CPU and CUDA generators produce different streams, so without a GPU the sample is drawn
    from the CPU generator's field of the same statistics)."""
    from hdp_b200 import synth
    lat, _ = synth.grid_latitudes(wl.n_lat, wl.n_lon)
    cols = (int(sel.min()), int(sel.max()) + 1)
    idx = sel - cols[0]
    base = synth.gridded_field(lat, wl.base_axis().dayofyr, seed=SAMPLE_SEED, offset=5.0, device=device, cols=cols)[:, idx].cpu().numpy()
    run = None
    if wl.run_years:
        run = synth.gridded_field(lat, wl.run_axis().dayofyr, seed=SAMPLE_SEED + 1, offset=5.0, trend=4.0, device=device,
                                  cols=cols)[:, idx].cpu().numpy()
    return base, run, (lat[sel] < 0).astype(np.uint8)


def base_config(wl, world, scaling):
    """`config` of the JSON line - identical for both arms (what differs, e.g. the CPU sample, lives in `cpu_baseline`)."""
    return {"workload": wl.name, "description": wl.description, "grid_cells": wl.cells, "base_days": len(wl.base_axis()),
            "run_days": len(wl.run_axis()) if wl.run_years else 0, "measures": wl.measures, "percentiles": len(wl.percentiles),
            "definitions": len(wl.defs), "window_radius": wl.radius, "n_gpus": world, "scaling": scaling}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (its Numba kernels from oracle/_ref under a
    process pool, one worker per host core; the oracle port only if that is absent) on a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from hdp_b200 import workloads
    wl = workloads.get(args.workload)
    cores = host_cores()
    n = args.cells or max(8 * cores, 64)
    sel = np.linspace(0, wl.cells - 1, n).astype(np.int64)
    try:
        import torch
        device = "cuda" if torch.cuda.is_available() else "cpu"
    except Exception:                                      # noqa: BLE001
        device = "cpu"
    base, run, south = sample_field(wl, sel, device)
    pool = reference_pool()
    kind = "reference" if pool else "port"
    one = (lambda b, r, s: reference_pass(pool, wl, b, r, s)) if pool else (lambda b, r, s: port_pass(wl, b, r, s))
    k = min(n, cores)
    for _ in range(max(args.warmup, 1)):
        one(base[:, :k], None if run is None else run[:, :k], south[:k])
    t_thr = t_met = 0.0
    for _ in range(args.steps):
        a, b, _, _ = one(base, run, south)
        t_thr += a; t_met += b
    if pool:
        pool.close()
    total = t_thr + t_met
    cy = n * (wl.base_years + wl.run_years) * args.steps          # one measure per sampled cell
    value = cy / total
    how = ("the reference's Numba kernels (oracle/_ref, hdp/threshold.py:52-93 + hdp/metric.py:304-369) under a process pool"
           if pool else "oracle/hdp_oracle.c with OpenMP")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": base_config(wl, args.gpus, args.scaling),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{n} cells of measure 0 of {wl.name} (evenly spaced over the grid, seed {SAMPLE_SEED}, generated on {device}) "
                                   f"per step, thresholds + metric sweep, {how}",
                         "thresholds_cell_years_per_s": n * wl.base_years * args.steps / max(t_thr, 1e-9),
                         "metrics_cell_years_per_s": (n * wl.run_years * args.steps / t_met) if t_met > 0 else None},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was diverted to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


THR_KERNELS = ("k_thr_generic", "k_thr_net", "k_thr_cand", "k_thr_seg", "k_thr_ranked", "normalize")
MET_KERNELS = ("k_hot_words", "k_scan", "k_met_fused")


class Job:
    """This rank's shard of one sharded job: `members` copies of the workload's grid, flattened (member, cell), cut into
    contiguous ranges by hdp_b200.shard.cell_range.  With `wl.members > 1` (lens50) the members share one member-free
    baseline: thresholds are computed on a shard of the GRID and all-gathered once (the only exchange on that path);
    otherwise every (member, cell) has its own baseline and nothing is exchanged."""

    def __init__(self, wl, dev, rank, world, members, cells_override=0):
        import torch
        from hdp_b200 import _tables as tb, shard, synth
        self.torch, self.shard, self.wl, self.dev, self.rank, self.world = torch, shard, wl, dev, rank, world
        self.shared_thr = wl.members > 1
        self.members = wl.members if self.shared_thr else members
        lat, _ = synth.grid_latitudes(wl.n_lat, wl.n_lon)
        if cells_override:
            lat = lat[np.linspace(0, wl.cells - 1, cells_override).astype(np.int64)]
        self.lat, self.grid = lat, lat.size
        self.C_global = self.grid * self.members
        self.c0, self.c1 = shard.cell_range(self.C_global, rank, world)
        self.pieces = shard.member_pieces(self.c0, self.c1, self.grid)
        self.C = self.c1 - self.c0
        self.wt = wl.window_tables()
        self.st = wl.seasons() if wl.run_years else None
        self.dm = tb.doy_map(wl.run_axis().dayofyr) if wl.run_years else None
        self.q, self.defs = wl.percentiles, wl.defs
        self.P, self.D, self.Y, self.n_doy = len(self.q), len(self.defs), (self.st.n_years if self.st else 0), self.wt.n_doy
        offsets = [5.0, -5.0, 0.0][: wl.measures]                       # tmax / tmin / tavg
        self.M = len(offsets)
        lat_local = np.concatenate([lat[g0:g1] for _, g0, g1 in self.pieces]) if self.pieces else lat[:0]
        self.south = torch.as_tensor((lat_local < 0).astype(np.uint8), device=dev)
        self.south_np = (lat_local < 0).astype(np.uint8)

        def field(axis, seed_of, off, trend, pieces):
            full = torch.empty((len(axis), sum(g1 - g0 for _, g0, g1 in pieces)), dtype=torch.float32, device=dev)
            a = 0
            for m, g0, g1 in pieces:                                    # every piece straight into its column block
                synth.gridded_field(lat, axis.dayofyr, seed=seed_of(m), offset=off, trend=trend, device=dev, cols=(g0, g1),
                                    out=full[:, a:a + g1 - g0])
                a += g1 - g0
            return full

        self.base, self.run = [], []
        for i, off in enumerate(offsets):
            seed = lambda m, i=i: SAMPLE_SEED + 10 * i + 1000 * m                       # noqa: E731
            if self.shared_thr:
                self.g0, self.g1 = shard.cell_range(self.grid, rank, world)             # this rank's part of the member-free baseline
                self.base.append(field(wl.base_axis(), lambda m, i=i: SAMPLE_SEED + 10 * i, off, 0.0, [(0, self.g0, self.g1)]))
            else:
                self.base.append(field(wl.base_axis(), seed, off, 0.0, self.pieces))
            self.run.append(field(wl.run_axis(), lambda m, i=i: SAMPLE_SEED + 10 * i + 1000 * m + 1, off, 4.0, self.pieces)
                            if wl.run_years else None)
        n_thr = (self.g1 - self.g0) if self.shared_thr else self.C
        self.thr = [torch.empty((n_thr, self.n_doy, self.P), dtype=torch.float64, device=dev) for _ in offsets]
        self.thr_full = [None] * self.M
        self.out = [torch.empty((4, self.P, self.D, self.Y, self.C), dtype=torch.uint16, device=dev) if wl.run_years else None
                    for _ in offsets]

    # ---- one step: every measure's thresholds, then its full percentile x definition sweep, on this rank's cells
    def step(self):
        from hdp_b200 import _core
        sh = self.shard
        for m in range(self.M):
            if not self.shared_thr:
                if self.run[m] is None:
                    _core.thresholds_array(self.base[m], self.wt, self.q, out=self.thr[m])
                else:
                    sh.run_sharded(self.base[m], self.run[m], self.wt, self.q, self.dm, self.defs, self.st.north, self.st.south,
                                   self.south, gather=False, local_of=self.C_global, out=(self.thr[m], self.out[m]))
                continue
            # member-free thresholds: a shard of the grid each, one all_gather, then this rank's (member, cell) pieces
            _core.thresholds_array(self.base[m], self.wt, self.q, out=self.thr[m])
            full = sh.gather_cells(self.thr[m], self.grid, dim=0)
            self.thr_full[m] = full
            a = 0
            for _, g0, g1 in self.pieces:
                n = g1 - g0
                piece = _core.metrics_array(self.run[m][:, a:a + n], full[g0:g1], self.dm, self.defs, self.st.north, self.st.south,
                                            self.south[a:a + n])
                self.out[m][..., a:a + n].copy_(piece)
                a += n

    def cell_years(self):
        wl = self.wl
        if self.shared_thr:
            return (self.grid * wl.base_years + self.C_global * wl.run_years) * self.M
        return self.C_global * (wl.base_years + wl.run_years) * self.M

    def bytes_per_step_global(self):
        wl = self.wl
        if self.shared_thr:      # SURVEY 8d, config 3: thresholds written once, read once per GPU
            met = self.C_global * (4 * len(wl.run_axis()) + 2 * 4 * self.Y * self.P * self.D) + self.world * self.grid * 8 * self.n_doy * self.P
            return self.M * (wl.bytes_thresholds(self.grid) + met)
        return self.M * (wl.bytes_thresholds(self.C_global) + (wl.bytes_metrics(self.C_global) if wl.run_years else 0))

    # ---- the output gather: every measure's thresholds and metrics of all ranks, over NCCL (NVLink / NVSwitch)
    def gather_once(self):
        """Every rank's outputs side by side on every rank (rank-major shards: what a consumer that assembles the arrays on the
        host needs; shard.gather_cells would add a device repacking pass for the cell-minor metrics)."""
        sh = self.shard
        got = 0
        for m in range(self.M):
            if not self.shared_thr:
                t, _ = sh.gather_shards(self.thr[m], self.C_global, dim=0)
                got += t.numel() * t.element_size()
                del t
            if self.out[m] is not None:
                o, _ = sh.gather_shards(self.out[m], self.C_global, dim=-1)
                got += o.numel() * o.element_size()
                del o
        return got

    def free(self):
        self.base = self.run = self.thr = self.out = self.thr_full = None
        self.torch.cuda.empty_cache()


def timed_steps(job, steps, warmup, world, dev, with_kernels=False):
    """`warmup` untimed steps, then `steps` timed ones between barrier + synchronize, CUDA events, max over ranks."""
    import torch
    import torch.distributed as dist
    from hdp_b200 import _core

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(warmup):
        job.step()
    sync_all()
    if with_kernels:
        _core.timing_enable(True)
        _core.timing_read()
    launches0 = _core.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        job.step()
    e1.record()
    sync_all()
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = _core.launch_count() - launches0
    kern = _core.timing_read() if with_kernels else []
    if with_kernels:
        _core.timing_enable(False)
    local_ms = ms
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {"ms": ms, "local_ms": local_ms, "launches": launches, "kern": kern, "t0": t0, "t1": t1}


def timed_gather(job, reps, world, dev):
    """The output gather alone (after the steps): all ranks' thresholds + metrics to every rank, CUDA events, max over ranks.
    NVLink figure: bytes a rank RECEIVES from its peers / time (with NVSwitch every rank's ingress is the limit)."""
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    job.gather_once()                                                   # warm-up (NCCL channel setup, allocator)
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    total = 0
    for _ in range(reps):
        total = job.gather_once()
    e1.record()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    received = total * (world - 1) / world
    return {"ms_per_step": ms, "bytes_gathered_per_step": int(total), "bytes_received_per_rank": int(received),
            "nvlink_ingress_gbs_per_gpu": received / (ms / 1e3) / 1e9, "collective": "all_gather (NCCL) of thresholds f64 + metrics u16 (shard.gather_shards: rank-major shards, no repacking pass)",
            "reps": reps}


def kernel_breakdown(kern, passes):
    by = {}
    for name, ms in kern:
        by.setdefault(name, []).append(ms)
    total = max(sum(np.sum(v) for v in by.values()), 1e-9)
    return ({k: float(np.sum(v)) / passes for k, v in by.items()}, {k: len(v) / passes for k, v in by.items()},
            {k: float(np.sum(v)) / total for k, v in by.items()})


def roofline_of(job, kernel_ms, kernel_share, kernel_launches, peak, peak_src):
    """Dominant kernel by summed CUDA-event time; its path's algorithmic bytes (SURVEY 8d) over the time of the kernels of that
    path (path 1: the threshold kernels incl. the transposing copy; path 2: the metric kernels, one pass split in launches)."""
    if not kernel_share:
        return None
    wl, C = job.wl, job.C
    dominant = max(kernel_share, key=kernel_share.get)
    if dominant in MET_KERNELS:
        names = [k for k in MET_KERNELS if k in kernel_ms]
        alg = wl.bytes_metrics(C)
    else:
        names = [k for k in THR_KERNELS if k in kernel_ms]
        alg = wl.bytes_thresholds(C)
    dur = sum(kernel_ms[k] for k in names)
    label = "+".join(names)
    achieved = alg / (dur / 1e3) / 1e9
    return {"bound": "hbm", "kernel": label, "dominant": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": measured_traffic(label, C), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
            "kernel_ms": kernel_ms, "kernel_share": kernel_share, "kernel_launches_per_measure": kernel_launches,
            "unit_of_launch": f"all launches of the kernel(s) for one measure ({C} cells)"}


def parity_on_sample(job, n, threads):
    """Oracle port on `n` of this rank's cells of measure 0 against what the GPU produced in the last step."""
    import torch
    if job.shared_thr:
        return None
    sel = np.linspace(0, job.C - 1, min(n, job.C)).astype(np.int64)
    sel_t = torch.as_tensor(sel, device=job.dev)
    b = job.base[0][:, sel_t].cpu().numpy()
    r = job.run[0][:, sel_t].cpu().numpy() if job.run[0] is not None else None
    _, _, thr_cpu, met_cpu = port_pass(job.wl, b, r, job.south_np[sel], threads)
    thr_gpu = job.thr[0][sel_t].cpu().numpy()
    res = {"cells": int(sel.size), "thresholds_bit_exact": bool(np.array_equal((thr_gpu + 0.0).view(np.uint64), (thr_cpu + 0.0).view(np.uint64)))}
    if met_cpu is not None:
        got = job.out[0].view(torch.int16)[..., sel_t].cpu().numpy().view(np.uint16).astype(np.int64).transpose(1, 2, 4, 0, 3)
        res["metrics_bit_exact"] = bool(np.array_equal(got, met_cpu))
    return res


DUMP_BYTES = 63_000_000      # under 64 MB with the .npy headers and cells.npy
DUMP_SEED = 2026


def dump_outputs(job, out_dir):
    """What the timed path handed back in its last step, so that two builds can be compared output for output: on a fixed,
    seeded sample of this rank's cells, every measure's thresholds (float64 [cells, n_doy, P]) and metrics (uint16
    [4, P, D, Y, cells], stored as float32, which holds them exactly), plus the sampled cell indices."""
    import torch
    per_cell = job.M * (job.n_doy * job.P * 8 + (4 * job.P * job.D * job.Y * 4 if job.wl.run_years else 0))
    n = max(1, min(job.C, DUMP_BYTES // per_cell))
    sel = np.sort(np.random.default_rng(DUMP_SEED).choice(job.C, n, replace=False))
    if job.shared_thr:           # thresholds are per grid cell: the grid cell of every sampled (member, cell)
        thr_rows, thr = np.concatenate([np.arange(g0, g1) for _, g0, g1 in job.pieces])[sel], job.thr_full
    else:
        thr_rows, thr = sel, job.thr
    sel_t, rows_t = torch.as_tensor(sel, device=job.dev), torch.as_tensor(thr_rows, device=job.dev)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "cells.npy"), (job.c0 + sel).astype(np.float64))
    for m in range(job.M):
        np.save(os.path.join(out_dir, f"thresholds_m{m}.npy"), thr[m][rows_t].cpu().numpy())
        if job.out[m] is not None:
            met = job.out[m].view(torch.int16)[..., sel_t].cpu().numpy().view(np.uint16)
            np.save(os.path.join(out_dir, f"metrics_m{m}.npy"), met.astype(np.float32))


def sub_record(job, res, steps, peak):
    bytes_step = job.bytes_per_step_global()
    ms = res["ms"] / steps
    gbs = bytes_step / (ms / 1e3) / 1e9 / job.world
    return {"value": job.cell_years() * steps / (res["ms"] / 1e3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
            "cells_global": int(job.C_global), "cells_per_gpu": int(job.C),
            "step_roofline_frac_per_gpu": gbs / peak, "achieved_gbs_per_gpu": gbs, "gpu_launches": int(res["launches"])}


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)            # libraries that print to fd 1 (NCCL's version banner) must not pollute the JSON line
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from hdp_b200 import _core, workloads

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: hdp_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    gpu_id = str(getattr(torch.cuda.get_device_properties(dev), "uuid", local_rank))
    if not gpu_id.startswith("GPU-") and len(gpu_id) > 8:
        gpu_id = "GPU-" + gpu_id
    full_affinity = bind_to_gpu_numa_node(gpu_id) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    peak, peak_src = peaks()
    wl = workloads.get(args.workload)
    scaling = args.scaling if world > 1 else "weak"
    members = world if scaling == "weak" else 1
    job = Job(wl, dev, rank, world, members, args.cells)

    sampler = ClockSampler(gpu_id) if rank == 0 else None
    res = timed_steps(job, args.steps, args.warmup, world, dev, with_kernels=True)
    clocks = sampler.stop(res["t0"], res["t1"]) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(job, args.dump_outputs)
    elapsed_ms = res["ms"]
    value = job.cell_years() * args.steps / (elapsed_ms / 1e3)

    kernel_ms, kernel_launches, kernel_share = kernel_breakdown(res["kern"], args.steps * job.M)
    roofline = roofline_of(job, kernel_ms, kernel_share, kernel_launches, peak, peak_src)
    step_bytes = job.bytes_per_step_global()
    step_gbs = step_bytes / (elapsed_ms / args.steps / 1e3) / 1e9 / world

    if world == 1:
        sharding = "one GPU: the whole grid"
    elif job.shared_thr:
        sharding = (f"{job.members} members x {job.grid} cells flattened, contiguous ranges over {world} ranks (shard.cell_range); "
                    "member-free thresholds computed on 1/N of the grid each and all-gathered once")
    elif scaling == "weak":
        sharding = (f"one job of {world} ensemble members x {job.grid} cells, flattened (member, cell) index cut into {world} contiguous "
                    "ranges (shard.cell_range -> one member per rank); thresholds stay on the GPU that computed them; no collective on the path")
    else:
        sharding = f"one grid of {job.grid} cells cut into {world} contiguous 32-aligned ranges (shard.cell_range); no collective on the path"
    config = base_config(wl, world, scaling)
    config.update({"cells_per_gpu": int(job.C), "cells_global": int(job.C_global), "sharding": sharding,
                   "l2": "inputs per step far larger than L2 (no flush needed)", "host_numa_binding": bool(full_affinity)})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32+f64", "data": "synthetic", "config": config,
        "gpu_launches": int(res["launches"]),
        "step_roofline": {"algorithmic_bytes_per_step_per_gpu": int(step_bytes // world), "achieved_gbs_per_gpu": step_gbs, "frac": step_gbs / peak},
        "roofline": roofline,
        "clocks": clocks,
    }

    # ---- the output gather over NVLink, timed on its own (SURVEY 8d: "outputs left on device, gather timed separately")
    if world > 1 and not args.no_gather:
        g = timed_gather(job, 2, world, dev)
        g["value_with_gather"] = job.cell_years() / ((elapsed_ms / args.steps + g["ms_per_step"]) / 1e3)
        line["gather"] = g

    # ---- e2e: the same step through the host-buffer C ABI (hdp_b200_*_host), H2D and D2H inside the timed region
    if not args.no_e2e and wl.run_years and not job.shared_thr:
        base0, run0, thr0, out0 = job.base[0], job.run[0], job.thr[0], job.out[0]
        h_base = torch.empty(base0.shape, dtype=torch.float32, pin_memory=True)
        h_run = torch.empty(run0.shape, dtype=torch.float32, pin_memory=True)
        h_thr = torch.empty(thr0.shape, dtype=torch.float64, pin_memory=True)
        h_out = torch.empty(out0.shape, dtype=torch.uint16, pin_memory=True)
        h_base.copy_(base0); h_run.copy_(run0)
        d_keep = torch.empty_like(thr0)
        torch.cuda.synchronize()

        def e2e_step():
            # host measures are reused for the M measures (same bytes moved as M distinct measures); the thresholds go to the
            # caller's host array AND stay on the device for the metric pass (hdp_b200_thresholds_host d_keep -> metrics_host d_thr)
            for _ in range(job.M):
                _core.thresholds_host(h_base.numpy(), job.wt, job.q, out=h_thr.numpy(), keep=d_keep)
                _core.metrics_host(h_run.numpy(), d_keep, job.dm, job.defs, job.st.north, job.st.south, job.south_np, out=h_out.numpy())

        def sync_all():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()

        e2e_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        sync_all()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        thr_bytes = job.C * job.n_doy * job.P * 8
        h2d = job.M * (h_base.numel() * 4 + h_run.numel() * 4 + job.C)
        d2h = job.M * (thr_bytes + h_out.numel() * 2)
        line["e2e"] = {"value": job.cell_years() * args.e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                       "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps, "ms_per_step": 1e3 * dt / args.e2e_steps,
                       "api": "hdp_b200_thresholds_host (d_keep) + hdp_b200_metrics_host (d_thr): pinned host buffers per rank, "
                              "thresholds returned to the host once and kept on the device for the metric pass"}
        # parity of the two arms on this run's data: host pipeline vs device-resident results of measure 0
        line["e2e"]["matches_device_path"] = bool(torch.equal(h_out.view(torch.int16).to(dev), out0.view(torch.int16)) and
                                                  torch.equal(h_thr.to(dev).view(torch.int64), thr0.view(torch.int64)))
        del h_base, h_run, h_thr, h_out, d_keep
        _core.host_release()

    # ---- cpu_baseline (rank 0): the reference's Numba kernels under a process pool on a bounded sample of measure 0 / member 0
    #      (the oracle port beside it; the port also checks this run's GPU results bit for bit)
    if rank == 0 and not args.no_cpu:
        if full_affinity:
            os.sched_setaffinity(0, full_affinity)         # the CPU baseline uses every host core
        cores = host_cores()
        n_probe = min(job.C, max(cores, 8))
        sel = np.linspace(0, job.C - 1, n_probe).astype(np.int64)

        def fetch(sel):
            sel_t = torch.as_tensor(sel, device=dev)
            b = job.base[0][:, sel_t].cpu().numpy()
            r = job.run[0][:, sel_t].cpu().numpy() if wl.run_years else None
            return b, r, job.south_np[sel]

        line["parity_on_sample"] = parity_on_sample(job, max(64, 4 * cores), cores)
        b_h, r_h, s_h = fetch(sel)
        a, b, _, _ = port_pass(wl, b_h, r_h, s_h)                                   # calibration of the port
        n = int(min(job.C, max(n_probe, 2 * args.cpu_seconds / max((a + b) / n_probe, 1e-6))))
        b_h, r_h, s_h = fetch(np.linspace(0, job.C - 1, n).astype(np.int64))
        t_thr, t_met, thr_port, met_port = port_pass(wl, b_h, r_h, s_h)
        port = {"value": n * (wl.base_years + wl.run_years) / (t_thr + t_met), "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{n} cells of measure 0 (rank 0's shard), oracle/hdp_oracle.c with OpenMP", "seconds": t_thr + t_met}
        pool = reference_pool() if not job.shared_thr else None
        if pool:
            k = min(job.C, 4 * cores)
            kb, kr, ks = fetch(np.linspace(0, job.C - 1, k).astype(np.int64))
            a, b, _, _ = reference_pass(pool, wl, kb, kr, ks)                       # calibration (JIT is already warm)
            n_ref = int(min(job.C, max(k, 2 * args.cpu_seconds / max((a + b) / k, 1e-6))))
            rb, rr, rs = fetch(np.linspace(0, job.C - 1, n_ref).astype(np.int64))
            t_thr, t_met, thr_ref, met_ref = reference_pass(pool, wl, rb, rr, rs)
            pool.close()
            line["cpu_baseline"] = {
                "value": n_ref * (wl.base_years + wl.run_years) / (t_thr + t_met), "unit": UNIT, "cores": cores, "kind": "reference",
                "sample": f"{n_ref} cells of measure 0 of {wl.name} (evenly spaced over rank 0's shard: the GPU arm's own inputs), thresholds + full "
                          "metric sweep through the reference's Numba kernels (oracle/_ref: hdp/threshold.py:52-93, hdp/metric.py:304-369), one "
                          "worker process per core, JIT warm-up excluded",
                "thresholds_cell_years_per_s": n_ref * wl.base_years / max(t_thr, 1e-9),
                "metrics_cell_years_per_s": (n_ref * wl.run_years / t_met) if t_met > 0 else None,
                "seconds": t_thr + t_met, "port": port,
            }
        else:
            line["cpu_baseline"] = port
        if r_h is not None:
            line["config"]["hot_day_fraction_lowest_percentile"] = float(np.mean(r_h > thr_port[np.arange(n)[None, :], job.dm[:, None], 0]))

    # ---- extra records: the other named workloads / partitions, each to the same timing rules (fewer steps)
    if not args.no_extra and not args.cells:
        job.free()
        k_steps, k_warm = max(2, args.steps // 3), 3
        def guarded(fn):
            """An extra record must never cost the headline: a failure (e.g. out of memory) is reported in its place.  Failures
            here are symmetric across ranks (same shapes everywhere), so no rank is left waiting in a collective."""
            try:
                return fn()
            except Exception as e:                         # noqa: BLE001
                torch.cuda.empty_cache()
                return {"error": f"{type(e).__name__}: {str(e)[:300]}"}

        def strong_record():
            sj = Job(wl, dev, rank, world, 1)
            try:
                r = timed_steps(sj, k_steps, k_warm, world, dev)
                rec = sub_record(sj, r, k_steps, peak)
                rec["sharding"] = f"one grid of {sj.grid} cells cut into {world} contiguous 32-aligned ranges; no collective on the path"
                if not args.no_gather:
                    rec["gather"] = guarded(lambda: timed_gather(sj, 2, world, dev))
                return rec
            finally:
                sj.free()

        def lens50_record():
            lw = workloads.get("lens50")
            lj = Job(lw, dev, rank, world, 1)
            try:
                r = timed_steps(lj, 2, 2, world, dev)
                rec = sub_record(lj, r, 2, peak)
                rec["sharding"] = (f"{lj.members} members x {lj.grid} cells flattened, {world} contiguous ranges ({len(lj.pieces)} member pieces "
                                   "on rank 0); thresholds: 1/N of the grid per rank + one all_gather inside the timed step")
                rec["imbalance"] = {"cells_per_gpu_max": int(max(b - a for a, b in lj.shard.all_ranges(lj.C_global, world))),
                                    "cells_per_gpu_mean": lj.C_global / world}
                # no output gather here: the metrics of all 50 members are 114 GB as uint16 - they stay sharded (each GPU hands its
                # own cells to the host); the one exchange of this workload, the threshold all_gather, is inside the timed step
                rec["gather"] = None
                return rec
            finally:
                lj.free()

        def config_record(name):
            xw = workloads.get(name)
            xj = Job(xw, dev, rank, world, 1)
            try:
                r = timed_steps(xj, k_steps, k_warm, world, dev, with_kernels=True)
                rec = sub_record(xj, r, k_steps, peak)
                kms, _, _ = kernel_breakdown(r["kern"], k_steps * xj.M)
                rec["kernel_ms_per_measure"] = kms
                rec["description"] = xw.description
                rec["parity_on_sample"] = parity_on_sample(xj, 16, host_cores())
                return rec
            finally:
                xj.free()

        if world > 1 and scaling == "weak" and not wl.members > 1:
            line["strong"] = guarded(strong_record)
        if world >= 4 and wl.name == "cmip6_1deg":
            line["lens50"] = guarded(lens50_record)
        if world == 1 and wl.name == "cmip6_1deg":
            line["configs"] = {name: guarded(lambda name=name: config_record(name)) for name in ("lens_member", "wide_sweep", "era5_025deg")}

    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
