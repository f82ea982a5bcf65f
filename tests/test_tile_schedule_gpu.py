"""The persistent TMA-staged stencil kernels on fields large enough that every CTA runs many tiles.

k_stencil_row_tma (xg_stencil2.cu), k_tile_stencil (xg_stencil_tile.cu) and k_tile_multi
(xg_stencil_multi_tma.cu) share one schedule: a CTA walks the virtual tiles i * gridDim.x + blockIdx.x,
ordered row block (~128 rows) by row block with level batches of U = 4 inside each, skips the padding tile
rows of the last row block, and cycles a ring of NST stages (2, or 1 for k_tile_multi without an x op)
guarded by full / empty mbarriers.  On the small shapes of the other suites each CTA runs one tile, so the
ring never wraps.  Here every case first checks, from the launchers' own geometry, that it does: more than
two tiles per CTA at the largest grid a launcher can pick, at least two row blocks, ragged x tiles and a
ragged last level batch.  Then the whole output is compared with the oracle bit for bit and the label of
the kernel that served the call is asserted.
"""

import itertools
import math

import numpy as np
import pytest
import torch

from oracle import stencil as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Launcher geometry, the same for the three kernels: TXE cells x TY rows per tile (RowTmaGeo, xg_stencil2.cu:491-500;
# TileGeo, xg_stencil_tile.cu:32-41; MultiGeo, xg_stencil_multi_tma.cu:34-43), U = 4 levels per tile
# (xg_stencil2.cu:838, kU xg_stencil_tile.cu:30, kUM xg_stencil_multi_tma.cu:32), row blocks of
# ceil(128 / TY) tile rows evened out to nrb blocks of rbq (xg_stencil2.cu:902-913, xg_stencil_tile.cu:480-491,
# xg_stencil_multi_tma.cu:342-353), grid = min(ctas * SMs, ntiles) with at most 4 CTAs per SM
# (xg_stencil2.cu:890-891,935-936, xg_stencil_tile.cu:464-465,527-528, xg_stencil_multi_tma.cu:332-333,360-361).
GEO = {np.float32: (224, 4), np.float64: (240, 2)}  # TXE, TY
U, RB, MAX_CTAS_PER_SM = 4, 128, 4
ROW_SHAPES = {np.float32: (18, 258, 1000), np.float64: (18, 260, 1000)}  # (levels, rows, x)
SWAP_SHAPE = (130, 42, 1000)  # stencils along Z: rows = Z, levels = Y
BCS = [("periodic", 0.0), ("fill", 1.5), ("fill", float("nan")), ("extend", 0.0), ("extrapolate", 0.0)]


def schedule(dtype, levels, rows, n):
    """The launchers' tile decomposition of a (levels, rows, n) view (rows = output rows)."""
    txe, ty = GEO[dtype]
    ntx = math.ceil(n / txe)
    npq = math.ceil(rows / ty)
    nrb = math.ceil(npq / math.ceil(RB / ty))
    rbq = math.ceil(npq / nrb)
    nzq = math.ceil(levels / U)
    return {"ntiles": nrb * nzq * rbq * ntx, "nrb": nrb, "rbq": rbq, "npq": npq, "padding": nrb * rbq - npq}


def premise(dtype, levels, rows, n):
    """Fail, saying why, when a shape no longer exercises the many-tiles-per-CTA schedule."""
    s = schedule(dtype, levels, rows, n)
    max_grid = MAX_CTAS_PER_SM * torch.cuda.get_device_properties(0).multi_processor_count
    what = f"{np.dtype(dtype).name} (levels, rows, x) = ({levels}, {rows}, {n}): {s}"
    assert s["ntiles"] > 2 * max_grid, f"{what}: fewer than 2 tiles per CTA at {max_grid} CTAs, the ring never wraps"
    assert s["nrb"] >= 2, f"{what}: a single row block"
    assert n % GEO[dtype][0] != 0, f"{what}: no partial last x tile"
    assert levels % U != 0, f"{what}: no partial last level batch"
    return s


def _field(shape, dtype, seed, nan_frac=0.01):
    rng = np.random.default_rng(seed)
    a = rng.random(shape).astype(dtype)
    if nan_frac:
        a[rng.random(shape) < nan_frac] = np.nan
    return a


def _metric(rng, shape, dtype):
    return (0.5 + rng.random(shape)).astype(dtype)


def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _label():
    from xgcm_b200 import _capi

    return _capi.last_launch()


def _check(got, want, label, expected, msg):
    assert label == expected, f"{msg}: served by {label}"
    assert got.shape == want.shape and got.dtype == want.dtype, msg
    np.testing.assert_array_equal(got, want, err_msg=msg)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_row_tma_ring_wraps(dtype):
    """Metric-fused diff / interp along x with a level-shared divisor dx(Y, X): every halo side and boundary,
    pre-metric absent, full (Z, Y, X), shared (Y, X), row-less (X) and one scalar per row (Y) or level (Z)."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    s = premise(dtype, Z, Y, X)
    assert s["padding"] > 0, s
    rng = np.random.default_rng(100)
    a = _field(shape, dtype, 101)
    x = _t(a)
    post = _metric(rng, (1, Y, X), dtype)
    pres = {"none": None, "full": _metric(rng, shape, dtype), "yx": _metric(rng, (1, Y, X), dtype),
            "x": _metric(rng, (1, 1, X), dtype), "y": _metric(rng, (1, Y, 1), dtype), "z": _metric(rng, (Z, 1, 1), dtype)}
    tp = {k: _t(v) for k, v in pres.items()}
    tq = _t(post)
    for lo, (bc, fill) in itertools.product((0, 1), BCS):
        for op, names in (("diff", list(pres)), ("interp", ["yx", "y"])):
            for name in names:
                got = ops.stencil2(x, 2, op, lo, 1 - lo, bc, fill, pre=tp[name], post=tq).cpu().numpy()
                want = oracle.stencil2(op, a, 2, lo, 1 - lo, bc, fill, pres[name], post)
                _check(got, want, _label(), "xg_stencil2(row_tma)", f"{op} lo={lo} {bc} {fill} pre={name}")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_row_tma_halo_planes(dtype):
    """Explicit halo planes replace the boundary rule on their side; the spare rows of the last tile row read
    their halo cell too."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    premise(dtype, Z, Y, X)
    rng = np.random.default_rng(110)
    a = _field(shape, dtype, 111)
    pre, post = _metric(rng, (1, Y, X), dtype), _metric(rng, (1, Y, X), dtype)
    hl, hh = rng.random((Z, Y)).astype(dtype), rng.random((Z, Y)).astype(dtype)
    for lo, op in itertools.product((0, 1), ("diff", "interp")):
        halo = hl if lo else hh
        parts = [halo[..., None], a * pre] if lo else [a * pre, halo[..., None]]
        want = oracle.KERNELS[op](np.concatenate(parts, axis=2)) / post
        got = ops.stencil2(_t(a), 2, op, lo, 1 - lo, "extend", 0.0, pre=_t(pre), post=_t(post),
                           halo_lo=_t(hl) if lo else None, halo_hi=None if lo else _t(hh)).cpu().numpy()
        _check(got, want.astype(dtype), _label(), "xg_stencil2(row_tma)", f"{op} lo={lo}")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tile_stencil_along_rows(dtype):
    """Metric-fused stencils along Y of a (Z, Y, X) field: n_out = n - 1, n, n + 1, the row boundaries that
    read their partner rows from global memory (periodic, extrapolate) and the ones that do not, level-shared
    (Y, X), full (Z, Y, X), per-row and per-level scalar metrics, min / max with a divisor."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    rng = np.random.default_rng(120)
    a = _field(shape, dtype, 121)
    x = _t(a)
    pre_full, pre_yx = _metric(rng, shape, dtype), _metric(rng, (1, Y, X), dtype)
    saw_padding = False
    for lo, hi in ((1, 0), (0, 1), (0, 0), (1, 1)):
        Yo = Y + lo + hi - 1
        s = premise(dtype, Z, Yo, X)
        saw_padding |= s["padding"] > 0
        q_yx, q_y, q_z = _metric(rng, (1, Yo, X), dtype), _metric(rng, (1, Yo, 1), dtype), _metric(rng, (Z, 1, 1), dtype)
        for i, (bc, fill) in enumerate((("periodic", 0.0), ("extrapolate", 0.0), ("fill", 1.5), ("extend", 0.0))):
            cases = [("diff", None, q_yx, "post yx"), ("diff", pre_full, q_yx, "pre full, post yx"),
                     ("interp", pre_yx, q_y, "pre yx, post y"),
                     ("max", None, q_yx, "post yx") if i % 2 else ("min", pre_yx, q_yx, "pre yx, post yx")]
            if bc in ("periodic", "extrapolate"):
                cases.append(("diff", pre_yx, q_z, "pre yx, post z"))
            for op, pre, post, name in cases:
                got = ops.stencil2(x, 1, op, lo, hi, bc, fill, pre=_t(pre), post=_t(post)).cpu().numpy()
                want = oracle.stencil2(op, a, 1, lo, hi, bc, fill, pre, post)
                _check(got, want, _label(), "xg_stencil2(tile_tma)", f"{op} lo={lo} hi={hi} {bc} {name}")
    assert saw_padding


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tile_stencil_along_rows_halo_planes(dtype):
    """Halo planes on the row term: lanes of the last, partial x tile read the plane at a clamped column."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    premise(dtype, Z, Y, X)
    rng = np.random.default_rng(130)
    a = _field(shape, dtype, 131)
    pre, post = _metric(rng, (1, Y, X), dtype), _metric(rng, (1, Y, X), dtype)
    hl, hh = rng.random((Z, X)).astype(dtype), rng.random((Z, X)).astype(dtype)
    for lo, op in itertools.product((0, 1), ("diff", "interp")):
        parts = [hl[:, None], a * pre] if lo else [a * pre, hh[:, None]]
        want = np.moveaxis(oracle.KERNELS[op](np.moveaxis(np.concatenate(parts, axis=1), 1, -1)), -1, 1) / post
        got = ops.stencil2(_t(a), 1, op, lo, 1 - lo, "periodic", 0.0, pre=_t(pre), post=_t(post),
                           halo_lo=_t(hl) if lo else None, halo_hi=None if lo else _t(hh)).cpu().numpy()
        _check(got, want.astype(dtype), _label(), "xg_stencil2(tile_tma)", f"{op} lo={lo}")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tile_stencil_swap_layout(dtype):
    """Metric-weighted interp and derivative along Z of a (Z, Y, X) field: the tile kernel runs rows = Z,
    levels = Y, with dz(Z) scalars per row (and a full pre-metric)."""
    from xgcm_b200 import ops

    Z, Y, X = SWAP_SHAPE
    rng = np.random.default_rng(140)
    a = _field(SWAP_SHAPE, dtype, 141)
    x = _t(a)
    dz, full = _metric(rng, (Z, 1, 1), dtype), _metric(rng, SWAP_SHAPE, dtype)
    saw_padding = False
    for lo, hi in ((1, 0), (0, 1), (0, 0), (1, 1)):
        Zo = Z + lo + hi - 1
        s = premise(dtype, Y, Zo, X)
        saw_padding |= s["padding"] > 0
        dzo = _metric(rng, (Zo, 1, 1), dtype)
        for bc, fill in (("extend", 0.0), ("periodic", 0.0), ("fill", float("nan")), ("extrapolate", 0.0)):
            for op, pre, name in (("interp", dz, "interp x dz / dz"), ("diff", None, "diff / dz"),
                                  ("interp", full, "interp x full / dz")):
                got = ops.stencil2(x, 0, op, lo, hi, bc, fill, pre=_t(pre), post=_t(dzo)).cpu().numpy()
                want = oracle.stencil2(op, a, 0, lo, hi, bc, fill, pre, dzo)
                _check(got, want, _label(), "xg_stencil2(tile_tma)", f"{name} lo={lo} hi={hi} {bc}")
    assert saw_padding


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_pair_tile_ring_wraps(dtype):
    """Divergence (a + b) and vorticity (a - b, b - a) with (Y, X) metrics on both terms and the divisor:
    diff / diff and interp / diff, every halo side pair, boundary pairs that include periodic on both axes."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    s = premise(dtype, Z, Y, X)
    assert s["padding"] > 0, s
    rng = np.random.default_rng(150)
    a, b = _field(shape, dtype, 151), _field(shape, dtype, 152)
    ta, tb = _t(a), _t(b)
    ma, mb, q = (_metric(rng, (1, Y, X), dtype) for _ in range(3))
    tma, tmb, tq = _t(ma), _t(mb), _t(q)
    bc_pairs = [(("periodic", 0.0), ("periodic", 0.0)), (("periodic", 0.0), ("fill", 1.5)), (("extend", 0.0), ("periodic", 0.0)),
                (("fill", 2.5), ("extend", 0.0))]
    for i, ((op_a, op_b), sub, (lo_a, lo_b)) in enumerate(itertools.product(
            (("diff", "diff"), ("interp", "diff")), (0, 1, 2), ((1, 0), (0, 1), (1, 1), (0, 0)))):
        (bc_a, fa), (bc_b, fb) = bc_pairs[i % len(bc_pairs)]
        got = ops.stencil_pair(ta, tb, (op_a, lo_a, 1 - lo_a, bc_a, fa), (1, op_b, lo_b, 1 - lo_b, bc_b, fb), sub,
                               pre_a=tma, pre_b=tmb, post=tq).cpu().numpy()
        want = oracle.stencil_pair(op_a, a, 2, lo_a, 1 - lo_a, bc_a, fa, ma, op_b, b, 1, lo_b, 1 - lo_b, bc_b, fb, mb, sub, q)
        _check(got, want, _label(), "xg_stencil_pair(tile_tma)", f"{op_a}/{op_b} sub={sub} lo=({lo_a},{lo_b}) {bc_a}/{bc_b}")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_multi_tile_ring_wraps(dtype):
    """Fused interp / diff / min / max along XY, YZ (one-stage ring), XZ and XYZ, every lo choice; all-periodic
    and all-extend boundaries (boundary tiles materialise wrapped / clamped cells into stages the TMA unit
    refills later), periodic / extend mixes, and a fill axis (the chain with operand overrides)."""
    from xgcm_b200 import ops

    shape = ROW_SHAPES[dtype]
    Z, Y, X = shape
    s = premise(dtype, Z, Y, X)
    assert s["padding"] > 0, s
    a = _field(shape, dtype, 161)
    x = _t(a)
    P, E, F = ("periodic", 0.0), ("extend", 0.0), ("fill", 1.5)
    patterns = [lambda k: [P] * k, lambda k: [E] * k, lambda k: [P, E, P][:k], lambda k: [F] + [E, P][: k - 1]]
    ops_ = ("interp", "diff", "min", "max")
    for j, axes in enumerate(((2, 1), (1, 0), (2, 0), (2, 1, 0))):
        for i, los in enumerate(itertools.product((0, 1), repeat=len(axes))):
            bcs = patterns[i % 4](len(axes))
            op = ops_[(i + j) % 4]
            specs = [(ax, op, lo, 1 - lo, bc, fill) for ax, lo, (bc, fill) in zip(axes, los, bcs)]
            got = ops.stencil_multi(x, specs).cpu().numpy()
            want = a
            for ax, o, lo, hi, bc, fill in specs:
                want = oracle.stencil2(o, want, ax, lo, hi, bc, fill)
            _check(got, want, _label(), "xg_stencil_multi(tile_tma)", str(specs))
