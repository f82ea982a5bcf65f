"""Generate tests/golden/* by RUNNING the reference's unmodified kernels.

Needs a source checkout of xgcm (the committed vectors come from xgcm 052b033a):

    python -m oracle.make_golden PATH_TO_XGCM_CHECKOUT

Outputs (small, committed):
  tests/golden/gridops_ref.npz      every <op>_<from>_to_<to> GridUFunc of xgcm/gridops.py applied to
                                    np.pad'ed inputs (the exact calls xarray makes), fp32 + fp64
  tests/golden/gridops_table.json   signature + padding_width of each of those GridUFuncs
  tests/golden/interp1d_ref.npz     xgcm.transform.interp_1d_linear (numba gufunc) on random columns
                                    incl. NaN / decreasing theta, all flag combinations
  tests/golden/conservative_ref.npz xgcm.transform.interp_1d_conservative (numba gufunc) incl. NaN bounds,
                                    decreasing / kinked columns, decreasing bins
  tests/golden/transform_cases.json the linear / log / conservative entries of the `cases` dict of
                                    xgcm/test/test_transform.py:41-683 (inputs + expected values)
  tests/golden/live_kernels_ref.npz every diff / interp / min / max GridUFunc on a periodic-padded fp64
                                    field along each axis, and interp_1d_linear on columns (every third
                                    one decreasing), with and without mask_edges

TEST INFRASTRUCTURE ONLY.
"""

from __future__ import annotations

import json
import re
import sys
from pathlib import Path

import numpy as np

from . import ref_loader

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"
PAD_MODE = {"periodic": "wrap", "fill": "constant", "extend": "edge"}


def gridops_vectors(gridops):
    rng = np.random.default_rng(20260924)
    out = {}
    table = {}
    names = [n for n in dir(gridops) if re.match(r"^(diff|interp|min|max)_\w+_to_\w+$", n)]
    for name in sorted(names):
        gu = getattr(gridops, name)
        sig = str(gu.signature)
        table[name] = {"signature": sig, "padding_width": gu.padding_width}
        if gu.padding_width is None:
            continue  # diff_left_to_inner: NotImplementedError
        lo, hi = gu.padding_width["X"]
        for dtype in (np.float32, np.float64):
            a = rng.random((3, 4, 9)).astype(dtype)
            a[0, 1, 3] = np.nan
            for axis in range(3):
                for bc, fill in (("periodic", 0.0), ("fill", 0.0), ("fill", 1.5), ("extend", 0.0)):
                    widths = [(0, 0)] * 3
                    widths[axis] = (lo, hi)
                    if bc == "fill":
                        p = np.pad(a, widths, mode="constant", constant_values=fill)
                    else:
                        p = np.pad(a, widths, mode=PAD_MODE[bc])
                    r = gu.ufunc(np.moveaxis(p, axis, -1))
                    r = np.moveaxis(r, -1, axis)
                    key = f"{name}|{np.dtype(dtype).name}|{axis}|{bc}|{fill}"
                    out[key] = r
            out[f"input|{np.dtype(dtype).name}|{name}"] = a
    return out, table


def interp1d_vectors(transform):
    rng = np.random.default_rng(7)
    out = {}
    for dtype in (np.float32, np.float64):
        ncol, n, m = 24, 13, 9
        phi = rng.random((ncol, n)).astype(dtype)
        theta = np.cumsum(0.2 + rng.random((ncol, n)), axis=-1).astype(dtype)
        theta[5:10] = theta[5:10, ::-1]  # decreasing columns
        theta[3, 4] = np.nan
        theta[7, 0] = np.nan
        theta[12, -1] = np.nan
        phi[2, 6] = np.nan
        target = np.linspace(0.0, float(np.nanmax(theta)) + 0.5, m).astype(dtype)
        target[4] = np.nan
        tag = np.dtype(dtype).name
        out[f"phi|{tag}"] = phi
        out[f"theta|{tag}"] = theta
        out[f"target|{tag}"] = target
        for mask in (False, True):
            for bypass in (False, True):
                with np.errstate(all="ignore"):
                    r = transform.interp_1d_linear(phi, theta, target, mask_edges=mask,
                                                   bypass_checks=bypass)
                out[f"out|{tag}|{int(mask)}|{int(bypass)}|0"] = r
        pos_theta = np.abs(theta) + 1.0
        pos_target = np.abs(np.nan_to_num(target, nan=1.0)) + 1.0
        out[f"log_theta|{tag}"] = pos_theta
        out[f"log_target|{tag}"] = pos_target
        with np.errstate(all="ignore"):
            r = transform.interp_1d_linear(phi, pos_theta, pos_target, mask_edges=True,
                                           logarithmic=True)
        out[f"out|{tag}|1|0|1"] = r
    return out


def conservative_vectors(transform):
    rng = np.random.default_rng(11)
    out = {}
    for dtype in (np.float32, np.float64):
        ncol, n, m = 20, 11, 8
        phi = rng.random((ncol, n)).astype(dtype)
        theta = np.cumsum(0.3 + rng.random((ncol, n + 1)), axis=-1).astype(dtype)
        theta[3:6] = theta[3:6, ::-1]            # decreasing columns
        theta[7, 4:6] = theta[7, 4:6][::-1]      # a non-monotonic kink
        theta[8, 0] = np.nan
        theta[9, -1] = np.nan
        theta[10, 3:5] = np.nan
        theta[11, 5] = theta[11, 6]              # zero-thickness cell
        phi[2, 4] = np.nan
        bins = np.linspace(0.0, float(np.nanmax(theta)) + 0.5, m).astype(dtype)
        tag = np.dtype(dtype).name
        out[f"phi|{tag}"] = phi
        out[f"theta|{tag}"] = theta
        out[f"bins|{tag}"] = bins
        with np.errstate(all="ignore"):
            out[f"out|{tag}|up"] = np.stack([transform.interp_1d_conservative(phi[c], theta[c], bins) for c in range(ncol)])
            out[f"out|{tag}|down"] = np.stack([transform.interp_1d_conservative(phi[c], theta[c], bins[::-1].copy()) for c in range(ncol)])
    return out


def live_kernel_vectors(gridops, transform):
    rng = np.random.default_rng(0)
    a = rng.random((3, 4, 7))
    out = {"a": a}
    names = [n for n in dir(gridops) if re.match(r"^(diff|interp|min|max)_\w+_to_\w+$", n)]
    for name in sorted(names):
        gu = getattr(gridops, name)
        if gu.padding_width is None:
            continue
        lo, hi = gu.padding_width["X"]
        for axis in range(3):
            widths = [(0, 0)] * 3
            widths[axis] = (lo, hi)
            p = np.pad(a, widths, mode="wrap")
            out[f"{name}|{axis}"] = np.moveaxis(gu.ufunc(np.moveaxis(p, axis, -1)), -1, axis)
    phi = rng.random((40, 30))
    theta = np.cumsum(rng.random((40, 30)) + 0.1, axis=-1)
    theta[::3] = theta[::3, ::-1]
    target = np.linspace(-1, theta.max() + 1, 25)
    out.update({"phi": phi, "theta": theta, "target": target})
    for mask in (False, True):
        out[f"interp_1d_linear|{int(mask)}"] = transform.interp_1d_linear(phi, theta, target, mask_edges=mask)
    return out


def transform_cases(root):
    src = (Path(root) / "xgcm" / "test" / "test_transform.py").read_text()
    start = src.index("cases = {")
    end = src.index("def construct_test_source_data")
    ns = {"np": np}
    exec(compile(src[start:end], "test_transform_cases", "exec"), ns)  # data literal only
    cases = ns["cases"]

    def conv(v):
        if isinstance(v, np.ndarray):
            return conv(v.tolist())
        if isinstance(v, (list, tuple)):
            return [conv(x) for x in v]
        if isinstance(v, dict):
            return {k: conv(x) for k, x in v.items()}
        if isinstance(v, (np.floating, float)):
            return None if np.isnan(v) else float(v)
        if isinstance(v, (np.integer,)):
            return int(v)
        return v

    keep = {}
    for name, case in cases.items():
        method = case["transform_kwargs"].get("method", "linear")
        if method not in ("linear", "log", "conservative"):
            continue
        keep[name] = conv(case)
    return keep


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python -m oracle.make_golden PATH_TO_XGCM_CHECKOUT")
    root = sys.argv[1]
    gridops, transform = ref_loader.load(root)
    GOLDEN.mkdir(parents=True, exist_ok=True)
    vec, table = gridops_vectors(gridops)
    np.savez_compressed(GOLDEN / "gridops_ref.npz", **vec)
    (GOLDEN / "gridops_table.json").write_text(json.dumps(table, indent=1, sort_keys=True))
    np.savez_compressed(GOLDEN / "interp1d_ref.npz", **interp1d_vectors(transform))
    np.savez_compressed(GOLDEN / "conservative_ref.npz", **conservative_vectors(transform))
    (GOLDEN / "transform_cases.json").write_text(json.dumps(transform_cases(root), indent=1, sort_keys=True))
    np.savez_compressed(GOLDEN / "live_kernels_ref.npz", **live_kernel_vectors(gridops, transform))
    for p in sorted(GOLDEN.iterdir()):
        print(p.name, p.stat().st_size)


if __name__ == "__main__":
    main()
