"""BASELINE.json's full sizes (config 3: 75 x 2400 x 3600 fp32, 648 M cells) and a > 2^31-element
field: the oracle cannot hold these in seconds, so parity is checked through size-independent
properties — any sub-block of the full-size result must equal the oracle applied to the matching
input sub-block (plus its halo), bit for bit."""

import itertools

import numpy as np
import pytest
import torch

from oracle import stencil as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
C3 = (75, 2400, 3600)
# Output windows per dim of a C3 field, placed on the seams of the TMA kernels' tile schedule (fp32: 224-cell x
# tiles, 4-row tile rows in row blocks of 128 rows, batches of 4 levels; fp64: 240 x 2, the same 128-row blocks):
# the first and last two levels, rows and columns, the last, 3-level batch (72-74), both sides of the first two
# row-block boundaries (127 / 128, 255 / 256), both sides of the last x tile's start (3584, 16 columns wide in
# fp32) and one window in the middle of each dim.
C3_WINDOWS = ([(0, 2), (37, 41), (70, 75)],
              [(0, 2), (125, 131), (253, 258), (1200, 1204), (2398, 2400)],
              [(0, 3), (1790, 1796), (3580, 3588), (3594, 3600)])


def _field(shape, seed, dtype=torch.float32):
    from xgcm_b200 import ops

    x = torch.empty(shape, dtype=dtype, device=DEV)
    return ops.fill_uniform(x, seed)


def _label():
    from xgcm_b200 import _capi

    return _capi.last_launch()


def _check_windows(x, out, specs, windows=C3_WINDOWS, pre=None, post=None):
    """Windows of `out` against the oracle chain `specs` = [(axis, op, lo, hi, padding, fill), ...] applied to the
    matching input windows, bit for bit.  Along an operated axis the input window reaches one cell further on each
    side, clipped at the array edge, so every kept output sees the same neighbours as in the full array, and one at
    a real edge sees the real boundary rule; a periodic or length-changing axis is taken whole.  `pre` / `post`:
    device metrics broadcasting against the field / the output (pre x field before the chain, / post after it)."""
    shape = x.shape
    whole = {ax for ax, _, lo, hi, bc, _ in specs if bc == "periodic" or lo + hi != 1}
    operated = {ax for ax, *_ in specs}
    per_dim = [[None] if d in whole else windows[d] for d in range(x.dim())]
    for wins in itertools.product(*per_dim):
        isl, osl, keep = [], [], []
        for d, w in enumerate(wins):
            if w is None:
                isl.append(slice(None)), osl.append(slice(None)), keep.append(slice(None))
                continue
            s, e = w
            s_in, e_in = (max(0, s - 1), min(shape[d], e + 1)) if d in operated else (s, e)
            isl.append(slice(s_in, e_in)), osl.append(slice(s, e)), keep.append(slice(s - s_in, e - s_in))

        def part(m, sl):
            return m[tuple(t if m.shape[d] > 1 else slice(None) for d, t in enumerate(sl))].cpu().numpy()

        want = x[tuple(isl)].cpu().numpy()
        if pre is not None:
            want = want * part(pre, isl)
        for ax, op, lo, hi, bc, fill in specs:
            want = oracle.stencil2(op, want, ax, lo, hi, bc if (lo or hi) else None, fill)
        want = want[tuple(keep)]
        if post is not None:
            want = want / part(post, osl)
        np.testing.assert_array_equal(out[tuple(osl)].cpu().numpy(), want, err_msg=f"{specs} at {wins}")


def _check_axis_blocks(x, out, axis, op, lo, hi, bc, fill, rng, nblocks=12):
    """Compare random full lines along `axis` (all cells of the operated axis, a small window of the
    other dims) against the oracle."""
    shape = x.shape
    for _ in range(nblocks):
        sl = []
        for d, n in enumerate(shape):
            if d == axis:
                sl.append(slice(None))
            else:
                w = min(n, 5)
                s0 = int(rng.integers(0, n - w + 1))
                sl.append(slice(s0, s0 + w))
        a = x[tuple(sl)].cpu().numpy()
        want = oracle.stencil2(op, a, axis, lo, hi, bc if (lo or hi) else None, fill)
        np.testing.assert_array_equal(out[tuple(sl)].cpu().numpy(), want)


def test_config3_full_size_stencils():
    from xgcm_b200 import ops

    shape = (75, 2400, 3600)
    x = _field(shape, 0xC0FFEE)
    rng = np.random.default_rng(0)
    for axis, (lo, hi), bc, fill in [(2, (1, 0), "periodic", 0.0), (1, (0, 1), "fill", 1.5), (0, (1, 0), "extend", 0.0),
                                     (0, (1, 1), "fill", 0.0), (2, (0, 0), None, 0.0), (1, (1, 1), "periodic", 0.0)]:
        for op in ("diff", "interp"):
            out = ops.stencil2(x, axis, op, lo, hi, bc, fill)
            _check_axis_blocks(x, out, axis, op, lo, hi, bc, fill, rng)
            del out


def test_config3_full_size_integrate_cumsum_transform():
    from xgcm_b200 import ops

    shape = (75, 2400, 3600)
    x = _field(shape, 7)
    rng = np.random.default_rng(1)
    dz = torch.from_numpy((10 * 1.05 ** np.arange(75)).astype(np.float32)).to(DEV).reshape(75, 1, 1)
    got = ops.wreduce(x, 0, dz, "sum")
    for _ in range(8):
        j, i = int(rng.integers(0, 2396)), int(rng.integers(0, 3596))
        a = x[:, j:j + 4, i:i + 4].cpu().numpy()
        np.testing.assert_array_equal(got[j:j + 4, i:i + 4].cpu().numpy(), oracle.wreduce(a, dz.cpu().numpy(), 0))
    for axis in (0, 1, 2):
        c = ops.cumscan(x, axis, False, "drop_last", 1, 0, "fill", 0.0)
        for _ in range(6):
            sl = [slice(int(s0), int(s0) + 3) for s0 in (rng.integers(0, n - 3) for n in shape)]
            sl[axis] = slice(None)
            a = x[tuple(sl)].cpu().numpy()
            np.testing.assert_array_equal(c[tuple(sl)].cpu().numpy(), oracle.cumscan(a, axis, False, "drop_last", 1, 0, "fill", 0.0))
        del c
    depth = torch.cumsum(dz.reshape(-1), 0)
    levels = torch.linspace(float(depth[0]) - 5, float(depth[-1]) + 5, 100, device=DEV)
    t = ops.vinterp_linear(x, depth.reshape(-1, 1, 1), levels, 0, True)
    assert t.shape == (2400, 3600, 100)
    for _ in range(6):
        j, i = int(rng.integers(0, 2396)), int(rng.integers(0, 3596))
        a = x[:, j:j + 4, i:i + 4].cpu().numpy()
        want = oracle.vinterp_linear(a, depth.cpu().numpy().reshape(-1, 1, 1) * np.ones((1, 4, 4), np.float32), levels.cpu().numpy(), 0, True)
        np.testing.assert_array_equal(t[j:j + 4, i:i + 4].cpu().numpy(), want)


def test_more_than_2_31_elements():
    """64-bit indexing: 2.42 G cells (9.7 GB) per field."""
    from xgcm_b200 import ops

    shape = (9, 16384, 16400)
    assert np.prod(shape) > 2**31
    x = _field(shape, 3)
    rng = np.random.default_rng(2)
    for axis, (lo, hi), bc in [(2, (1, 0), "periodic"), (1, (0, 1), "extend"), (0, (1, 0), "fill")]:
        out = ops.stencil2(x, axis, "diff", lo, hi, bc, 2.0)
        _check_axis_blocks(x, out, axis, "diff", lo, hi, bc, 2.0, rng, nblocks=6)
        # the far corner of the array (flat offsets beyond 2^31)
        sl = [slice(n - 3, n) for n in shape]
        sl[axis] = slice(None)
        a = x[tuple(sl)].cpu().numpy()
        np.testing.assert_array_equal(out[tuple(sl)].cpu().numpy(), oracle.stencil2("diff", a, axis, lo, hi, bc, 2.0))
        del out
    s = ops.wreduce(x, 0, None, "sum")
    np.testing.assert_array_equal(s[-2:, -5:].cpu().numpy(), x[:, -2:, -5:].cpu().numpy().sum(axis=0))
    del s
    c = ops.cumscan(x, 2)
    np.testing.assert_array_equal(c[-1, -1, :].cpu().numpy(), np.cumsum(x[-1, -1, :].cpu().numpy()))


def test_cubed_sphere_full_size_operators():
    """A cubed sphere at production size (50 levels x 6 faces x 1020^2 fp32, 1.25 GB, device
    resident): every operator result on sampled levels must equal the oracle's face-connection
    padding + pairwise kernel on those levels — seams, rotations and all — bit for bit."""
    import xgcm_b200 as xg
    from oracle import faces as oracle_faces
    from test_faces_gpu import AXES, COORDS, CUBED_SPHERE

    nz, nf, n = 50, 6, 1020
    f = _field((nz, nf, n, n), 11)
    ds = xg.Dataset(coords={"z": np.arange(nz), "face": np.arange(nf), "y": np.arange(n) + 0.0,
                            "yl": np.arange(n) - 0.5, "x": np.arange(n) + 0.0, "xl": np.arange(n) - 0.5})
    grid = xg.Grid(ds, coords=COORDS, face_connections=CUBED_SPHERE, autoparse_metadata=False)
    da = xg.DataArray(f, dims=("z", "face", "y", "x"))
    levels = [0, 17, nz - 1]
    host = f[levels].cpu().numpy()
    for op, ax in (("diff", "X"), ("interp", "Y"), ("max", "X")):
        out = getattr(grid, op)(da, ax)
        assert out.is_device and out.shape == (nz, nf, n, n)
        padded = oracle_faces.pad_face_connections(
            host, ("z", "face", "y", "x"), AXES, "face", CUBED_SPHERE["face"], {ax: (1, 0)},
            {"X": None, "Y": None}, {"X": 0.0, "Y": 0.0})
        k = 3 if ax == "X" else 2
        want = np.moveaxis(oracle.KERNELS[op](np.moveaxis(padded, k, -1)), -1, k)
        np.testing.assert_array_equal(out.data[levels].cpu().numpy(), want.astype(np.float32))


def test_config4_sampled_steps():
    """BASELINE configs[3] (x365 time steps, time-sharded): the field of ANY global step is
    regenerated on the device from the step index (tools/bench_c4.py uses the same generator), so
    parity is checked on sampled steps — first, middle, last of the year — exactly as a rank that
    owns them would compute them: Grid.diff / Grid.interp on X (periodic), Y (fill), Z (extend),
    random full lines of every result against the oracle, bit for bit."""
    import xgcm_b200 as xg
    from xgcm_b200 import ops

    shape = (75, 2400, 3600)
    nz, ny, nx = shape
    ds = xg.Dataset(coords={"Z": np.arange(nz) + 0.5, "Zl": np.arange(nz) + 0.0, "YC": np.arange(ny) + 0.5,
                            "YG": np.arange(ny) + 0.0, "XC": np.arange(nx) + 0.5, "XG": np.arange(nx) + 0.0})
    grid = xg.Grid(ds, coords={"X": {"center": "XC", "left": "XG"}, "Y": {"center": "YC", "left": "YG"},
                               "Z": {"center": "Z", "left": "Zl"}},
                   padding={"X": "periodic", "Y": "fill", "Z": "extend"}, autoparse_metadata=False)
    x = torch.empty(shape, dtype=torch.float32, device=DEV)
    da = xg.DataArray(x, dims=("Z", "YC", "XC"))
    rng = np.random.default_rng(4)
    for t in (0, 182, 364):
        ops.fill_uniform(x, 0xC0FFEE, offset=t * x.numel())
        for ax, k, bc in (("X", 2, "periodic"), ("Y", 1, "fill"), ("Z", 0, "extend")):
            for op in ("diff", "interp"):
                out = getattr(grid, op)(da, ax)
                _check_axis_blocks(x, out.data, k, op, 1, 0, bc, 0.0, rng, nblocks=4)


def _c3_grid(dev=DEV):
    """The C3 dataset of bench.py's `extra` records (dxC / dxG (Y, X), drF / drC (Z), periodic X, fill Y,
    extend Z) plus dyC / dyG (Y, X) metrics for derivative('Y')."""
    import xgcm_b200 as xg

    nz, ny, nx = C3
    jj = np.arange(ny, dtype=np.float64)[:, None]
    dx = (1e3 * (1 + 0.1 * np.cos(2 * np.pi * jj / ny)) * np.ones((1, nx))).astype(np.float32)
    dy = (1e3 * (1 + 0.1 * np.sin(2 * np.pi * jj / ny)) * np.ones((1, nx))).astype(np.float32)
    dz = (10 * 1.05 ** np.arange(nz)).astype(np.float32)
    ds = xg.Dataset(coords={"Z": np.arange(nz) + 0.5, "Zl": np.arange(nz) + 0.0, "YC": np.arange(ny) + 0.5,
                            "YG": np.arange(ny) + 0.0, "XC": np.arange(nx) + 0.5, "XG": np.arange(nx) + 0.0})
    for nm, dims, arr in (("dxC", ("YC", "XC"), dx), ("dxG", ("YC", "XG"), dx), ("dyC", ("YG", "XC"), dy),
                          ("dyG", ("YC", "XG"), dy), ("drF", ("Z",), dz), ("drC", ("Zl",), dz)):
        ds[nm] = xg.DataArray(torch.from_numpy(arr).to(dev), dims=dims)
    grid = xg.Grid(ds, coords={"X": {"center": "XC", "left": "XG"}, "Y": {"center": "YC", "left": "YG"},
                               "Z": {"center": "Z", "left": "Zl"}},
                   metrics={("X",): ["dxC", "dxG"], ("Y",): ["dyC", "dyG"], ("Z",): ["drF", "drC"]},
                   padding={"X": "periodic", "Y": "fill", "Z": "extend"}, autoparse_metadata=False)
    metrics = {"dx": torch.from_numpy(dx[None]).to(dev), "dy": torch.from_numpy(dy[None]).to(dev),
               "dz": torch.from_numpy(dz.reshape(nz, 1, 1)).to(dev)}
    return grid, metrics


def test_config3_tma_kernels_full_size():
    """The persistent TMA-staged kernels at the size they were timed at (C3 fp32: ~440 tiles per CTA, 19 row
    blocks with 8 padding tile rows, a 16-column last x tile, a 3-level last batch), called like bench.py's
    `extra` records; windows on every seam of the schedule against the oracle, and the kernel that served each call."""
    import xgcm_b200 as xg
    from xgcm_b200 import ops

    grid, m = _c3_grid()
    x = _field(C3, 0xC0FFEE)
    d = xg.DataArray(x, dims=("Z", "YC", "XC"))
    P, F, E = ("periodic", 0.0), ("fill", 0.0), ("extend", 0.0)
    calls = [
        (lambda: grid.derivative(d, "X"), "xg_stencil2(row_tma)", [(2, "diff", 1, 0) + P], None, m["dx"]),
        (lambda: grid.derivative(d, "Y"), "xg_stencil2(tile_tma)", [(1, "diff", 1, 0) + F], None, m["dy"]),
        (lambda: grid.interp(d, "Z", metric_weighted="Z"), "xg_stencil2(tile_tma)", [(0, "interp", 1, 0) + E], m["dz"], m["dz"]),
        (lambda: grid.interp(d, ["X", "Y"]), "xg_stencil_multi(tile_tma)", [(2, "interp", 1, 0) + P, (1, "interp", 1, 0) + F],
         None, None),
        (lambda: grid.interp(d, ["Y", "Z"]), "xg_stencil_multi(tile_tma)", [(1, "interp", 1, 0) + F, (0, "interp", 1, 0) + E],
         None, None),
        (lambda: grid.interp(d, ["X", "Y", "Z"]), "xg_stencil_multi(tile_tma)",
         [(2, "interp", 1, 0) + P, (1, "interp", 1, 0) + F, (0, "interp", 1, 0) + E], None, None),
    ]
    for fn, label, specs, pre, post in calls:
        out = fn().data
        assert _label() == label, (specs, _label())
        _check_windows(x, out, specs, pre=pre, post=post)
        del out
    # diff('Y') x hFac(Z, Y, X) / dx(Y, X): a full pre-metric next to a level-shared divisor
    hfac = _field(C3, 5) + 0.5
    out = ops.stencil2(x, 1, "diff", 1, 0, "fill", 0.0, pre=hfac, post=m["dx"])
    assert _label() == "xg_stencil2(tile_tma)", _label()
    _check_windows(x, out, [(1, "diff", 1, 0) + F], pre=hfac, post=m["dx"])


def test_config3_vorticity_full_size():
    """C3-sized vorticity (diff(v dy, 'X') - diff(u dx, 'Y')) / rA, both signs, through the two-field tile kernel:
    the first and last two levels (the last, 3-level batch) and one in the middle, whole planes."""
    from xgcm_b200 import ops

    grid, m = _c3_grid()
    u, v = _field(C3, 21), _field(C3, 22)
    area = m["dx"] * m["dy"]
    hp = [t.cpu().numpy()[0] for t in (m["dx"], m["dy"], area)]
    for sub in (1, 2):
        out = ops.stencil_pair(v, u, ("diff", 1, 0, "periodic", 0.0), (1, "diff", 1, 0, "fill", 0.0), sub,
                               pre_a=m["dy"], pre_b=m["dx"], post=area)
        assert _label() == "xg_stencil_pair(tile_tma)", _label()
        for k in (0, 1, 37, 73, 74):
            va, ua = v[k].cpu().numpy(), u[k].cpu().numpy()
            want = oracle.stencil_pair("diff", va, 1, 1, 0, "periodic", 0.0, hp[1], "diff", ua, 0, 1, 0, "fill", 0.0,
                                       hp[0], sub, hp[2])
            np.testing.assert_array_equal(out[k].cpu().numpy(), want, err_msg=f"sub={sub} level {k}")
        del out


def test_config3_fp64_derivatives_full_size():
    """derivative('X') (row kernel) and derivative('Y') (tile kernel) on a C3-sized fp64 field, 5.2 GB: the fp64
    instantiations with their ring wrapping ~900 times per CTA."""
    from xgcm_b200 import ops

    _, m = _c3_grid()
    x = _field(C3, 31, torch.float64)
    for axis, bc, metric, label in ((2, "periodic", "dx", "xg_stencil2(row_tma)"), (1, "fill", "dy", "xg_stencil2(tile_tma)")):
        post = m[metric].double()
        out = ops.stencil2(x, axis, "diff", 1, 0, bc, 0.0, post=post)
        assert _label() == label, _label()
        _check_windows(x, out, [(axis, "diff", 1, 0, bc, 0.0)], post=post)
        del out


def test_fallback_stencils_full_size():
    """The kernels that serve what the vector paths cannot: length-changing shifts along X (the scalar row
    kernel, whose grid-stride loop only iterates at this size) and a 3601-wide (`outer`-position) field along
    X, Y and Z (scalar row kernel, strided kernel)."""
    from xgcm_b200 import ops

    x = _field(C3, 41)
    for (lo, hi), bc, fill in (((0, 0), None, 0.0), ((1, 1), "periodic", 0.0), ((1, 1), "fill", 2.5), ((1, 1), "extend", 0.0)):
        for op in ("diff", "interp"):
            out = ops.stencil2(x, 2, op, lo, hi, bc, fill)
            assert _label() == "xg_stencil2(row_scalar)", _label()
            _check_windows(x, out, [(2, op, lo, hi, bc, fill)])
            del out
    del x
    shape = (75, 2400, 3601)
    x = _field(shape, 42)
    windows = C3_WINDOWS[:2] + ([(0, 3), (1790, 1796), (3596, 3601)],)
    for axis, (lo, hi), bc, label in ((2, (1, 0), "extend", "row_scalar"), (2, (0, 1), "fill", "row_scalar"),
                                      (1, (1, 0), "periodic", "strided"), (1, (0, 1), "extend", "strided"),
                                      (0, (1, 0), "fill", "strided"), (0, (1, 1), "extend", "strided")):
        for op in ("diff", "max"):
            out = ops.stencil2(x, axis, op, lo, hi, bc, 1.5)
            assert _label() == f"xg_stencil2({label})", (axis, _label())
            _check_windows(x, out, [(axis, op, lo, hi, bc, 1.5)], windows=windows)
            del out
