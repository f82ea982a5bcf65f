#!/usr/bin/env python
"""bench.py — grid-cells/s for Grid.diff + Grid.interp on a C-grid field (BASELINE.json metric).

A *step* = one pass of the hot path over one synthetic (75, 2400, 3600) fp32 field
(BASELINE configs[2], "C3"): ``Grid.diff`` and ``Grid.interp`` along X (periodic),
Y (fill) and Z (extend) — six fused ``xg_stencil2`` launches, 6 x 648 M output cells.

  value   whole-job cells/s with the field already resident in HBM (device-backed DataArray),
          timed with CUDA events, barrier + synchronize on both sides, max over ranks.
  e2e     the same six Grid calls on a HOST (page-locked numpy) DataArray: every call streams
          H2D -> kernel -> D2H inside the C-ABI (xg_stencil2_host); copies are in the timed region.
  roofline  algorithmic bytes (8 B/cell fp32, SURVEY 8d) / mean per-launch duration measured live
          with CUDA events on the launching stream, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline  the oracle (numpy restatement of the reference's calls: np.pad + ufunc on a
          moveaxis view) timed single-threaded on the host, rank 0, N=1, on a bounded sample.

``--dump-outputs DIR`` writes what the last timed step returned, one ``DIR/<op>_<axis>.npy`` (fp32) per Grid call:
a seeded sub-block (DUMP_SAMPLE levels x rows x columns, both edges of every axis included) of each output, the
same cells on every run with the same arguments, so two builds can be compared output for output.

``--impl reference`` times the reference's own CPU path (the oracle port; xarray/dask are not
installable, see DESIGN.md) with a thread pool over all host cores on broadcast-dim chunks —
the dask="parallelized" analogue (xgcm/grid.py:786-789).

Multi-GPU (torchrun): every rank owns the time steps of its shard (one field per step, no
data-path collective, SURVEY 8e) => weak scaling.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (75, 2400, 3600)  # (Z, Y, X), C3
DTYPE = np.float32
SEED = 0xC0FFEE
# (axis name, padding, fill) — SURVEY 8d: periodic X, fill Y, extend Z
AXES = (("X", "periodic", None), ("Y", "fill", 0.0), ("Z", "extend", None))
OPS = ("diff", "interp")
METRIC = "grid-cells/s for diff+interp on C-grid field; achieved HBM GB/s vs peak"
DUMP_SAMPLE = (16, 128, 1024)  # (Z, Y, X) indices kept per output by --dump-outputs: 8 MiB fp32 each, 48 MiB for six
WORKLOAD = ("C3 (BASELINE configs[2]): Grid.diff + Grid.interp along X(periodic), Y(fill), Z(extend) of one "
            "75x2400x3600 fp32 C-grid field per step")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", type=int, nargs=3, default=list(SHAPE))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the per-config records (C1, C2, C3 integrate, C4 loop, C5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of each output of the last timed step to DIR/<op>_<axis>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_sample_index(shape):
    """Sorted indices along (Z, Y, X) for --dump-outputs: the first and last two of every axis, where the
    boundary conditions act, plus seeded random interior ones; the whole axis when it is short."""
    rng = np.random.default_rng(SEED)
    idx = []
    for n, k in zip(shape, DUMP_SAMPLE):
        if n <= k:
            idx.append(np.arange(n))
        else:
            inner = rng.choice(np.arange(2, n - 2), k - 4, replace=False)
            idx.append(np.sort(np.concatenate([[0, 1, n - 2, n - 1], inner])))
    return idx


def make_dataset(shape, field):
    import xgcm_b200 as xg

    nz, ny, nx = shape
    coords = {
        "Z": np.arange(nz) + 0.5, "Zl": np.arange(nz) + 0.0,
        "YC": np.arange(ny) + 0.5, "YG": np.arange(ny) + 0.0,
        "XC": np.arange(nx) + 0.5, "XG": np.arange(nx) + 0.0,
    }
    ds = xg.Dataset(coords=coords)
    grid = xg.Grid(
        ds,
        coords={"X": {"center": "XC", "left": "XG"}, "Y": {"center": "YC", "left": "YG"},
                "Z": {"center": "Z", "left": "Zl"}},
        padding={"X": "periodic", "Y": "fill", "Z": "extend"},
        autoparse_metadata=False,
    )
    da = xg.DataArray(field, dims=("Z", "YC", "XC"), name="theta")
    return grid, da


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = f"/tmp/xgcm_b200_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=self.out, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    smax.append(float(parts[2]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        busy = [s for s in sm if s > 0]
        return {
            "sm_mhz": statistics.median(busy) if busy else None,
            "sm_max_mhz": max(smax) if smax else None,
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# --------------------------------------------------------------------------- the oracle legs (CPU)
def oracle_step(a, pool=None, nchunks=1, out_buf=None):
    """The reference's numpy calls for the six ops (np.pad copy + kernel on a moveaxis view).
    out_buf: a preallocated result array re-used by every op (no first-touch page faults per call) —
    kinder than the reference, which returns a fresh array per op."""
    from oracle import stencil as oracle

    def one(op, axis_i, bc, fill):
        lo, hi = 1, 0  # center -> left
        if pool is None:
            return oracle.stencil2(op, a, axis_i, lo, hi, bc, 0.0 if fill is None else fill)
        # dask="parallelized" analogue: chunk a broadcast (non-operated) dim, one task per chunk
        chunk_axis = 0 if axis_i != 0 else 1
        nch = max(1, min(nchunks, a.shape[chunk_axis]))
        bounds = np.linspace(0, a.shape[chunk_axis], nch + 1).astype(int)
        out = np.empty(a.shape, a.dtype) if out_buf is None else out_buf

        def task(i):
            sl = [slice(None)] * a.ndim
            sl[chunk_axis] = slice(bounds[i], bounds[i + 1])
            out[tuple(sl)] = oracle.stencil2(op, a[tuple(sl)], axis_i, lo, hi, bc, 0.0 if fill is None else fill)

        list(pool.map(task, range(nch)))
        return out

    axis_index = {"Z": 0, "Y": 1, "X": 2}
    cells = 0
    for ax, bc, fill in AXES:
        for op in OPS:
            r = one(op, axis_index[ax], bc, fill)
            cells += r.size
            del r
    return cells


def run_reference(args):
    """--impl reference: the reference's CPU path on the host cores (rank 0 only).  Nothing of the product
    is imported here: inputs come from oracle/synth.py (same bits as the device generator)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor

    from oracle import synth

    cores = os.cpu_count() or 1
    shape = tuple(args.shape)
    a = np.empty(shape, DTYPE)
    with ThreadPoolExecutor(max_workers=min(cores, 32)) as gen:  # numpy releases the GIL: generate planes in parallel
        plane = int(np.prod(shape[1:]))
        list(gen.map(lambda k: synth.fill_uniform(a[k], SEED, k * plane), range(shape[0])))

    out_buf = np.empty(shape, DTYPE)
    out_buf.fill(0)  # touch the pages once

    def timed_step(workers, buf=out_buf):
        with ThreadPoolExecutor(max_workers=workers) as pool:
            t0 = time.perf_counter()
            oracle_step(a, pool, workers, buf)
            return time.perf_counter() - t0

    t_alloc = timed_step(cores, None)  # the untuned figure: every hardware thread, a fresh result per op

    # pool calibration, one full step each: every hardware thread (dask's default) and one worker per
    # physical core (SMT siblings share the load/store ports this path saturates)
    candidates = sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True)
    calib = {w: timed_step(w) for w in candidates}
    workers = min(calib, key=calib.get)
    t_full = calib[workers]
    steps_total = args.steps + max(args.warmup - 1, 0)
    budget_s = 240.0  # the whole --steps K --warmup W run should end within a few minutes
    nz = shape[0]
    nz_s = nz if t_full * steps_total <= budget_s else max(2, int(nz * budget_s / (t_full * steps_total)))
    sub = a if nz_s == nz else np.ascontiguousarray(a[:nz_s])
    sub_out = out_buf[:nz_s]
    with ThreadPoolExecutor(max_workers=workers) as pool:
        for _ in range(max(args.warmup - 1, 0)):
            oracle_step(sub, pool, workers, sub_out)
        t0 = time.perf_counter()
        cells = 0
        for _ in range(args.steps):
            cells += oracle_step(sub, pool, workers, sub_out)
        dt = time.perf_counter() - t0
    value = cells / dt
    cells_full = 6 * int(np.prod(shape))
    sample = (f"{'the full workload' if nz_s == nz else f'first {nz_s} of {nz} Z levels of the field'} per step, "
              f"{args.steps} steps; thread pool of {workers} workers over broadcast-dim chunks (dask='parallelized' "
              f"analogue, xgcm/grid.py:786-789) writing into ONE preallocated result array; one-step calibration, "
              f"workers -> cells/s: " + ", ".join(f"{w}: {cells_full / t:.3g}" for w, t in sorted(calib.items())) +
              f"; untuned ({cores} workers, fresh result array per op as the reference returns): "
              f"{cells_full / t_alloc:.3g} cells/s; np.pad still copies the field per call, so the path scales poorly")
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "shape": list(shape), "cells_per_step": cells // args.steps,
                   "same_config": nz_s == nz},
        "cpu_baseline": {"value": value, "unit": "cells/s", "cores": workers, "kind": "port", "sample": sample,
                         "host_cores": cores,
                         "calibration_cells_per_s": {str(w): cells_full / t for w, t in sorted(calib.items())},
                         "untuned_cells_per_s": cells_full / t_alloc},
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "numpy": np.__version__,
    }
    print(json.dumps(line), flush=True)



# --------------------------------------------------------------------------- every BASELINE config, one record each
def run_extras(torch, dist, ops, _capi, x, rank, world, peak):
    """`extra`: ms, cells/s, algorithmic bytes and fraction of the measured HBM peak for the BASELINE configs
    the headline does not cover (configs[0], [1], the integrate('Z') half of [2], [3] as a 32-step loop with
    device-generated steps, [4]).  Device-resident, CUDA events, median of the timed repeats, max over ranks;
    a buffer larger than L2 is rewritten between the repeats of the L2-sized configs (C1, C2)."""
    import xgcm_b200 as xg

    dev = x.device
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, iters, flush_l2=False, warmup=2, reps=1):
        """median over `iters` of (time of `reps` back-to-back calls) / reps.  reps > 1 is used for the
        bandwidth-bound configs (every call streams >= 2.6 GB, far beyond L2): the host-side bookkeeping of
        call k+1 overlaps the kernel of call k, as in any real sequence of Grid calls."""
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(iters):
            if flush_l2:
                flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(reps):
                fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) / reps)
        ms = torch.tensor([statistics.median(ts)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def rec(name, ms, cells, nbytes, launches, note):
        return {"config": name, "ms": ms, "cells_per_s": cells * world / (ms * 1e-3),
                "algorithmic_bytes": nbytes, "GBps_per_gpu": nbytes / (ms * 1e-3) / 1e9,
                "frac_of_peak": nbytes / (ms * 1e-3) / 1e9 / peak, "launches_per_call": launches, "note": note}

    out = []

    def count(fn):
        n0 = _capi.load().xg_launch_count()
        fn()
        return int(_capi.load().xg_launch_count() - n0)

    # ---- C1: 1-D periodic, 1e6 fp64, Grid.diff('X') + Grid.interp('X') -------------------------------------
    n1 = 1_000_000
    a1 = torch.empty(n1, dtype=torch.float64, device=dev)
    ops.fill_uniform(a1, SEED + 1)
    ds1 = xg.Dataset(coords={"XC": np.arange(n1) + 0.5, "XG": np.arange(n1) + 0.0})
    g1 = xg.Grid(ds1, coords={"X": {"center": "XC", "left": "XG"}}, padding="periodic", autoparse_metadata=False)
    d1 = xg.DataArray(a1, dims=("XC",))

    def c1():
        g1.diff(d1, "X")
        g1.interp(d1, "X")

    out.append(rec("C1 (configs[0]): 1e6 fp64 periodic, Grid.diff('X') + Grid.interp('X')", timed(c1, 20, True), 2 * n1,
                   2 * 16 * n1, count(c1), "16 MB per launch: launch/latency bound, L2 flushed between repeats"))

    # ---- C2: 360x240x50 fp32, derivative('X') with dx(Y,X); metric-weighted interp('Z') ---------------------
    nz2, ny2, nx2 = 50, 240, 360
    a2 = torch.empty((nz2, ny2, nx2), dtype=torch.float32, device=dev)
    ops.fill_uniform(a2, SEED + 2)
    jj = np.arange(ny2, dtype=np.float64)[:, None]
    dx2 = (1e3 * (1 + 0.1 * np.cos(2 * np.pi * jj / ny2)) * np.ones((1, nx2))).astype(np.float32)
    dz2 = (10 * 1.05 ** np.arange(nz2)).astype(np.float32)
    ds2 = xg.Dataset(coords={"Z": np.arange(nz2) + 0.5, "Zl": np.arange(nz2) + 0.0, "YC": np.arange(ny2) + 0.5,
                             "YG": np.arange(ny2) + 0.0, "XC": np.arange(nx2) + 0.5, "XG": np.arange(nx2) + 0.0})
    for nm, dims, arr in (("dxC", ("YC", "XC"), dx2), ("dxG", ("YC", "XG"), dx2), ("drF", ("Z",), dz2), ("drC", ("Zl",), dz2)):
        ds2[nm] = xg.DataArray(torch.from_numpy(arr).to(dev), dims=dims)
    g2 = xg.Grid(ds2, coords={"X": {"center": "XC", "left": "XG"}, "Y": {"center": "YC", "left": "YG"},
                              "Z": {"center": "Z", "left": "Zl"}},
                 metrics={("X",): ["dxC", "dxG"], ("Z",): ["drF", "drC"]},
                 padding={"X": "periodic", "Y": "fill", "Z": "extend"}, autoparse_metadata=False)
    d2 = xg.DataArray(a2, dims=("Z", "YC", "XC"))
    c2 = a2.numel()
    f_der2 = lambda: g2.derivative(d2, "X")
    out.append(rec("C2 (configs[1]): 50x240x360 fp32 Grid.derivative('X'), dx(Y,X) fused", timed(f_der2, 20, True), c2,
                   8 * c2 + 4 * ny2 * nx2, count(f_der2), "17 MB per launch: launch/latency bound, L2 flushed"))
    f_mw2 = lambda: g2.interp(d2, "Z", metric_weighted="X")
    out.append(rec("C2: Grid.interp('Z', metric_weighted='X') (x dx, / dx fused)", timed(f_mw2, 20, True), c2,
                   8 * c2 + 8 * ny2 * nx2, count(f_mw2), "launch/latency bound"))
    del a2, d2

    # ---- C3-sized metric-fused stencils and integrate('Z') ----------------------------------------------------
    nz, ny, nx = x.shape
    cells = x.numel()
    jj = np.arange(ny, dtype=np.float64)[:, None]
    dx3 = (1e3 * (1 + 0.1 * np.cos(2 * np.pi * jj / ny)) * np.ones((1, nx))).astype(np.float32)
    dz3 = (10 * 1.05 ** np.arange(nz)).astype(np.float32)
    ds3 = xg.Dataset(coords={"Z": np.arange(nz) + 0.5, "Zl": np.arange(nz) + 0.0, "YC": np.arange(ny) + 0.5,
                             "YG": np.arange(ny) + 0.0, "XC": np.arange(nx) + 0.5, "XG": np.arange(nx) + 0.0})
    for nm, dims, arr in (("dxC", ("YC", "XC"), dx3), ("dxG", ("YC", "XG"), dx3), ("drF", ("Z",), dz3), ("drC", ("Zl",), dz3)):
        ds3[nm] = xg.DataArray(torch.from_numpy(arr).to(dev), dims=dims)
    g3 = xg.Grid(ds3, coords={"X": {"center": "XC", "left": "XG"}, "Y": {"center": "YC", "left": "YG"},
                              "Z": {"center": "Z", "left": "Zl"}},
                 metrics={("X",): ["dxC", "dxG"], ("Z",): ["drF", "drC"]},
                 padding={"X": "periodic", "Y": "fill", "Z": "extend"}, autoparse_metadata=False)
    d3 = xg.DataArray(x, dims=("Z", "YC", "XC"))
    f_int = lambda: g3.integrate(d3, "Z")
    out.append(rec("C3 (configs[2]): Grid.integrate('Z'), 1-D dz", timed(f_int, 5, reps=4), cells, 4 * cells + 4 * ny * nx + 4 * nz,
                   count(f_int), "cells = input cells; 2.59 GB in, 34.6 MB out"))
    f_der3 = lambda: g3.derivative(d3, "X")
    out.append(rec("C3-sized Grid.derivative('X'), dx(Y,X) fused", timed(f_der3, 5, reps=4), cells, 8 * cells + 4 * ny * nx,
                   count(f_der3), "the C2 operation at a bandwidth-bound size"))
    # two-field composite: (diff(u dy, X) + diff(v dx, Y)) / area in one pass (3 array streams, 12 B/cell)
    v3 = torch.empty_like(x)
    ops.fill_uniform(v3, SEED + 7)
    dx_t = torch.from_numpy(dx3).to(dev)
    area_t = dx_t * dx_t
    spec_a, spec_b = ("diff", 0, 1, "periodic", 0.0), (1, "diff", 0, 1, "periodic", 0.0)
    f_div = lambda: ops.stencil_pair(x, v3, spec_a, spec_b, 0, pre_a=dx_t, pre_b=dx_t, post=area_t)
    out.append(rec("C3-sized divergence (diff(u dy,'X') + diff(v dx,'Y')) / rA, one fused pass (xg_stencil_pair)",
                   timed(f_div, 5, reps=4), cells, 12 * cells + 3 * 4 * ny * nx, count(f_div),
                   "the explicit chain moves ~9 array passes; here read u, read v, write out"))
    del v3
    # the notebook idiom grid.interp(da, ['X', 'Y', 'Z']) (center -> corner): one fused pass (xg_stencil_multi)
    f_multi = lambda: g3.interp(d3, ["X", "Y", "Z"])
    try:
        out.append(rec("C3-sized Grid.interp(['X','Y','Z']) to the cell corner, one fused pass (xg_stencil_multi)",
                       timed(f_multi, 5, reps=4), cells, 8 * cells, count(f_multi),
                       "the reference runs one full pad + ufunc pass per axis"))
    except Exception as exc:
        out.append({"config": "C3-sized Grid.interp(['X','Y','Z'])", "error": repr(exc)})
    f_mwz = lambda: g3.interp(d3, "Z", metric_weighted="Z")
    try:
        out.append(rec("C3-sized Grid.interp('Z', metric_weighted='Z') (x drF, / drC fused)", timed(f_mwz, 5, reps=4), cells,
                       8 * cells, count(f_mwz), ""))
    except Exception as exc:
        out.append({"config": "C3-sized Grid.interp('Z', metric_weighted='Z')", "error": repr(exc)})
    f_cum = lambda: g3.cumsum(d3, "Z", padding="fill")
    try:
        out.append(rec("C3-sized Grid.cumsum('Z')", timed(f_cum, 5, reps=4), cells, 8 * cells, count(f_cum), ""))
    except Exception as exc:  # keep the bench line alive if an optional record fails
        out.append({"config": "C3-sized Grid.cumsum('Z')", "error": repr(exc)})

    # ---- C5: Grid.transform Z -> 100 levels (linear, mask_edges), Y-sharded when N > 1 ------------------------
    m = 100
    y0, y1 = (0, ny) if world == 1 else (ny * rank // world, ny * (rank + 1) // world)
    dzf = 10 * 1.05 ** np.arange(nz)
    depth = (np.cumsum(dzf) - dzf / 2).astype(np.float32)
    levels = np.linspace(depth[0] - 5, depth[-1] + 5, m).astype(np.float32)
    ds5 = xg.Dataset(coords={"Z": depth})
    g5 = xg.Grid(ds5, coords={"Z": {"center": "Z"}}, autoparse_metadata=False)
    xs = x[:, y0:y1, :].contiguous() if world > 1 else x
    d5 = xg.DataArray(xs, dims=("Z", "Y", "X"))
    f_tr = lambda: g5.transform(d5, "Z", levels)
    cols = (y1 - y0) * nx
    ms5 = timed(f_tr, 5, reps=4)
    r5 = rec("C5 (configs[4]): Grid.transform('Z' -> 100 levels, linear, mask_edges)" + (f", Y sharded x{world}" if world > 1 else ""),
             ms5, cols * m, cols * (nz + m) * 4, count(f_tr), "cells = output cells; (n + m) * 4 B per column")
    r5["kernel"] = _capi.last_launch()
    out.append(r5)
    del xs, d5

    # ---- N > 1: the one real exchange step of the path — the operated axis itself sharded across the GPUs -------
    if world > 1:
        from xgcm_b200 import parallel

        comm = parallel.Communicator()
        for ax_name, axn in (("Z", 0), ("X", 2)):
            plane_bytes = cells // x.shape[axn] * 4
            f_fused = lambda: comm.stencil2(x, axn, "diff", 1, 0, "periodic")
            f_torch = lambda: parallel.sharded_stencil2(x, axn, "diff", 1, 0, "periodic")
            f_local = lambda: ops.stencil2(x, axn, "diff", 1, 0, "periodic")
            ms_f, ms_t, ms_l = timed(f_fused, 5, reps=4), timed(f_torch, 5, reps=4), timed(f_local, 5, reps=4)
            r = rec(f"C3 block per GPU, {ax_name} axis sharded x{world} (periodic ring): Grid.diff via xg_stencil2_sharded",
                    ms_f, cells, 8 * cells, count(f_fused),
                    "pack kernel + one NCCL group on a side stream while the local block is computed + edge fix-up")
            r.update({"nvlink_bytes_per_gpu_per_call": 2 * plane_bytes, "ms_same_kernel_unsharded": ms_l,
                      "ms_torch_distributed_path": ms_t,
                      "exchange_hidden_frac": None if ms_t <= ms_l else max(0.0, min(1.0, (ms_t - ms_f) / (ms_t - ms_l)))})
            out.append(r)
        comm.close()

    # ---- C4: >= 32 time steps, each generated on the device, then the six ops of the headline -----------------
    grid, da = make_dataset(tuple(x.shape), x)
    nsteps = 32
    t_first = rank * nsteps  # this rank's block of the time axis
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    gen_ms = []
    if world > 1:
        dist.barrier()
    e[0].record()
    for t in range(nsteps):
        g0, g1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        ops.fill_uniform(x, SEED, offset=(t_first + t) * cells)
        g1_.record()
        gen_ms.append((g0, g1_))
        for ax, bc, fill in AXES:
            for op in OPS:
                r = getattr(grid, op)(da, ax)
                del r
    e[1].record()
    torch.cuda.synchronize()
    tot = torch.tensor([e[0].elapsed_time(e[1])], device=dev, dtype=torch.float64)
    gen = torch.tensor([sum(a.elapsed_time(b) for a, b in gen_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        dist.all_reduce(gen, op=dist.ReduceOp.MAX)
    tot, gen = float(tot.item()), float(gen.item())
    out.append({"config": f"C4 (configs[3]) as a {nsteps}-step loop per GPU: generate the step's 75x2400x3600 field on the device, "
                          f"then the 6 ops (time shards x{world}; the full 365 steps: tools/bench_c4.py)",
                "ms_per_step_incl_generation": tot / nsteps, "ms_per_step_ops_only": (tot - gen) / nsteps,
                "cells_per_s": 6 * cells * nsteps * world / (tot * 1e-3),
                "cells_per_s_ops_only": 6 * cells * nsteps * world / ((tot - gen) * 1e-3),
                "frac_of_peak_ops_only": 6 * 8 * cells * nsteps / ((tot - gen) * 1e-3) / 1e9 / peak})
    ops.fill_uniform(x, SEED, offset=rank * cells)  # restore this rank's headline field
    del flush
    return out

# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from xgcm_b200 import _capi, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    from xgcm_b200 import device as xg_device

    numa = xg_device.bind_to_gpu_numa(torch.cuda.current_device())  # before any page-locked allocation
    lib = _capi.load()
    shape = tuple(args.shape)
    cells_field = int(np.prod(shape))
    es = np.dtype(DTYPE).itemsize

    # this rank's field: time step `rank` of the synthetic series (counter-based RNG => any shard anywhere)
    x = torch.empty(shape, dtype=torch.float32, device=dev)
    ops.fill_uniform(x, SEED, offset=rank * cells_field)
    grid, da_dev = make_dataset(shape, x)
    dumped = None
    if args.dump_outputs and rank == 0:
        iz, iy, ix = (torch.as_tensor(i, device=dev) for i in dump_sample_index(shape))
        sample_at = (iz[:, None, None], iy[None, :, None], ix[None, None, :])
        dumped = {}

    def step_device(timer=None, keep=None):
        n = 0
        for ax, bc, fill in AXES:
            for op in OPS:
                if timer is not None:
                    timer.append((ax, op, torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
                    timer[-1][2].record()
                r = getattr(grid, op)(da_dev, ax)
                if timer is not None:
                    timer[-1][3].record()
                if keep is not None:
                    keep[f"{op}_{ax}"] = r
                n += r.size
                del r
        return n

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        # a warm-up step that keeps its results leaves their memory in the allocator's cache, so keeping the
        # last timed step's results for --dump-outputs allocates nothing inside the timed window
        step_device(keep={} if dumped is not None and i == 0 else None)
    barrier()
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    launches0 = lib.xg_launch_count()
    timers = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    cells = 0
    for i in range(args.steps):
        cells += step_device(timers, dumped if i == args.steps - 1 else None)
    e1.record()
    barrier()
    if dumped:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, r in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), r.data[sample_at].cpu().numpy())
        dumped.clear()
    launches = lib.xg_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = cells * world / (ms_total * 1e-3)

    per_kernel = {}
    for ax, op, s, e in timers:
        per_kernel.setdefault(f"{op}_{ax}", []).append(s.elapsed_time(e))
    launch_ms = [t for v in per_kernel.values() for t in v]
    mean_launch_ms = sum(launch_ms) / len(launch_ms)
    peak, peak_src = measured_peak()
    alg_bytes = 2 * es * cells_field  # read n + write n (SURVEY 8d: 8 B/cell fp32)
    achieved = alg_bytes / (mean_launch_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "peak_source": peak_src,
        "kernel": "xg_stencil2 (k_stencil_row_vec for X, k_stencil_strided for Y/Z)",
        "algorithmic_bytes_per_launch": alg_bytes,
        "mean_launch_ms": mean_launch_ms,
        "per_op_GBps": {k: alg_bytes / (statistics.median(v) * 1e-3) / 1e9 for k, v in per_kernel.items()},
    }

    extra = None
    if not args.no_extra:
        try:
            extra = run_extras(torch, dist, ops, _capi, x, rank, world, peak)
        except Exception as exc:  # never lose the headline line to an optional record
            extra = [{"error": repr(exc)}]

    # ---- e2e: host buffers through the public Grid API -----------------------------------------
    e2e = None
    if not args.no_e2e:
        host = ops.pinned_empty(shape, DTYPE)  # allocated AFTER the NUMA binding above: pages on the GPU's socket
        torch.from_numpy(host).copy_(x)
        torch.cuda.synchronize()
        _, da_host = make_dataset(shape, host)
        reqs = [(op, ax) for ax, bc, fill in AXES for op in OPS]

        def step_host_batched():
            # numpy in -> six numpy results out, one call: the field crosses PCIe once (xg_stencil2_host_multi)
            n = 0
            for r in grid.apply_many(da_host, reqs):
                n += r.size
            return n

        def step_host_per_call():
            n = 0
            for ax, bc, fill in AXES:
                for op in OPS:
                    r = getattr(grid, op)(da_host, ax)  # numpy in -> numpy out, copies inside, one upload per call
                    n += r.size
                    del r
            return n

        def time_host(fn, k):
            for _ in range(2):
                fn()
            barrier()
            t0 = time.perf_counter()
            n = 0
            for _ in range(k):
                n += fn()
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            return n, float(dt.item())

        k = max(1, min(args.steps, 5))
        n, dt = time_host(step_host_batched, k)
        n_pc, dt_pc = time_host(step_host_per_call, max(1, min(k, 3)))
        # the same batched call on a PAGEABLE input (a plain np.empty array): the driver stages it
        pageable = np.empty(shape, DTYPE)
        np.copyto(pageable, host)
        _, da_page = make_dataset(shape, pageable)
        n_pg, dt_pg = time_host(lambda: sum(r.size for r in grid.apply_many(da_page, reqs)), 2)
        nbytes = cells_field * es
        e2e = {"value": n * world / dt, "unit": "cells/s", "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": 6 * nbytes, "steps": k, "ms_per_step": dt / k * 1e3,
               "d2h_GBps_per_gpu": 6 * nbytes * k / dt / 1e9,
               "path": "Grid.apply_many(numpy DataArray, 6 requests) -> xg_stencil2_host_multi: one upload per step, "
                       "six results streamed back (3-stream slab pipeline, page-locked buffers)",
               "per_call": {"value": n_pc * world / dt_pc, "ms_per_step": dt_pc / max(1, min(k, 3)) * 1e3,
                            "h2d_bytes_per_step": 6 * nbytes, "d2h_bytes_per_step": 6 * nbytes,
                            "path": "six separate Grid.diff / Grid.interp calls -> xg_stencil2_host (one upload per call)"},
               "pageable_input": {"value": n_pg * world / dt_pg, "ms_per_step": dt_pg / 2 * 1e3,
                                  "note": "same batched call, input in ordinary (not page-locked) numpy memory"}}
        del host, da_host, pageable, da_page

    # ---- cpu_baseline (rank 0, N=1 only): the oracle, single thread, one full step ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        a = x.cpu().numpy()
        t0 = time.perf_counter()
        n = oracle_step(a)  # numpy elementwise ufuncs / np.pad are single-threaded
        dt = time.perf_counter() - t0
        cpu = {"value": n / dt, "unit": "cells/s", "cores": 1, "kind": "port",
               "sample": f"1 full step (6 ops x {cells_field} cells) of the same workload, numpy {np.__version__}, "
                         f"host has {os.cpu_count()} cores; --impl reference uses all of them",
               "seconds": dt}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "shape": list(shape), "cells_per_step_per_gpu": cells // args.steps,
                       "l2": "each field is 2.59 GB in + 2.59 GB out per launch, >> 126 MB L2: no flush needed",
                       "parallelism": f"time-shards x{world} (one field per rank per step, no collective on the data path)",
                       "numa": numa},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
