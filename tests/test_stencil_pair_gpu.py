"""xg_stencil_pair (two-field composites: divergence, vorticity) against the explicit chain of single-axis
stencils and numpy arithmetic (oracle.stencil_pair <- docs/ufunc_examples.md:105-153, grid.py:796-832)."""

import itertools

import numpy as np
import pytest
import torch

from oracle import stencil as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", [(6, 40, 64), (3, 5, 24, 132), (17, 36), (4, 9, 50), (2, 300, 8)])
def test_pair_matches_chain(dtype, shape):
    from xgcm_b200 import ops

    rng = np.random.default_rng(31)
    a = rng.standard_normal(shape).astype(dtype)
    b = rng.standard_normal(shape).astype(dtype)
    a[rng.random(shape) < 0.01] = np.nan
    nd = len(shape)
    bcs = [("periodic", 0.0), ("fill", 1.5), ("extend", 0.0)]
    for axis_b in range(nd - 1):
        for (op_a, op_b), (lo_a, lo_b), ((bc_a, fa), (bc_b, fb)), sub in itertools.product(
                [("diff", "diff"), ("interp", "diff"), ("min", "max")], [(1, 0), (0, 1), (1, 1), (0, 0)],
                [(bcs[0], bcs[1]), (bcs[1], bcs[2]), (bcs[2], bcs[0])], [0, 1, 2]):
            hi_a, hi_b = 1 - lo_a, 1 - lo_b
            want = oracle.stencil_pair(op_a, a, nd - 1, lo_a, hi_a, bc_a, fa, None, op_b, b, axis_b, lo_b, hi_b, bc_b,
                                       fb, None, sub, None)
            got = ops.stencil_pair(_t(a), _t(b), (op_a, lo_a, hi_a, bc_a, fa), (axis_b, op_b, lo_b, hi_b, bc_b, fb),
                                   sub).cpu().numpy()
            np.testing.assert_array_equal(got, want, err_msg=f"{op_a}/{op_b} b={axis_b} lo=({lo_a},{lo_b}) {bc_a}/{bc_b} sub={sub}")
    # metrics: 2-D horizontal (broadcast over the leading dims), full-shape, and 1-D along axis b
    if nd >= 3:
        m2 = (1 + rng.random(shape[-2:])).astype(dtype)
        mfull = (1 + rng.random(shape)).astype(dtype)
        m1 = (1 + rng.random((shape[0],) + (1,) * (nd - 1))).astype(dtype)
        for pre_a, pre_b, post in [(m2, m2, m2), (mfull, m2, mfull), (m1, mfull, m2), (None, m2, None)]:
            for sub in (0, 1):
                want = oracle.stencil_pair("diff", a, nd - 1, 0, 1, "periodic", 0.0, pre_a, "diff", b, nd - 2, 0, 1,
                                           "periodic", 0.0, pre_b, sub, post)
                got = ops.stencil_pair(_t(a), _t(b), ("diff", 0, 1, "periodic", 0.0), (nd - 2, "diff", 0, 1, "periodic", 0.0),
                                       sub, pre_a=_t(pre_a), pre_b=_t(pre_b), post=_t(post)).cpu().numpy()
                np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", [(5, 9, 452), (3, 6, 904), (2, 3, 5, 676), (6, 2, 1000)])
def test_pair_tile_kernel_matches_chain(dtype, shape):
    """Rows long enough for the TMA-staged tile kernel (axis b next to x, metrics shared between levels):
    every boundary / shift / sign combination and every metric layout it stages (2-D shared, full 3-D,
    x-only, per-row and per-level scalars), ragged tiles in x, rows and levels."""
    from xgcm_b200 import _capi, ops

    rng = np.random.default_rng(33)
    a = rng.standard_normal(shape).astype(dtype)
    b = rng.standard_normal(shape).astype(dtype)
    a[rng.random(shape) < 0.01] = np.nan
    nd = len(shape)
    axis_b = nd - 2

    def metric(dims):
        return (0.5 + rng.random([shape[d] if d in dims else 1 for d in range(nd)])).astype(dtype)

    m2, mfull, mz, mx, my = metric((nd - 2, nd - 1)), metric(range(nd)), metric((0,)), metric((nd - 1,)), metric((nd - 2,))
    bcs = [("periodic", 0.0), ("fill", 1.5), ("extend", 0.0)]
    for (op_a, op_b), (lo_a, lo_b), ((bc_a, fa), (bc_b, fb)), sub in itertools.product(
            [("diff", "diff"), ("interp", "diff"), ("min", "max")], [(1, 0), (0, 1), (1, 1), (0, 0)],
            [(bcs[0], bcs[1]), (bcs[1], bcs[2]), (bcs[2], bcs[0])], [0, 1, 2]):
        hi_a, hi_b = 1 - lo_a, 1 - lo_b
        want = oracle.stencil_pair(op_a, a, nd - 1, lo_a, hi_a, bc_a, fa, m2, op_b, b, axis_b, lo_b, hi_b, bc_b, fb, m2, sub, m2)
        got = ops.stencil_pair(_t(a), _t(b), (op_a, lo_a, hi_a, bc_a, fa), (axis_b, op_b, lo_b, hi_b, bc_b, fb), sub,
                               pre_a=_t(m2), pre_b=_t(m2), post=_t(m2)).cpu().numpy()
        if shape[-1] >= (448 if dtype == np.float32 else 480) and op_a != "min":  # two tiles per row; diff / interp
            assert _capi.last_launch() == "xg_stencil_pair(tile_tma)"
        np.testing.assert_array_equal(got, want, err_msg=f"{op_a}/{op_b} lo=({lo_a},{lo_b}) {bc_a}/{bc_b} sub={sub}")
    combos = [(mfull, m2, m2), (mz, mfull, m2), (None, m2, None), (m2, None, m2), (mx, my, m2), (my, mx, mx), (None, None, m2),
              (m2, m2, mz), (m2, m2, my), (mfull, mfull, mfull), (m2, mfull, mfull)]
    for pre_a, pre_b, post in combos:
        for (lo_a, lo_b), sub, (bc, f) in itertools.product([(0, 1), (1, 0)], (0, 1), bcs):
            want = oracle.stencil_pair("diff", a, nd - 1, lo_a, 1 - lo_a, bc, f, pre_a, "interp", b, axis_b, lo_b, 1 - lo_b,
                                       bc, f, pre_b, sub, post)
            got = ops.stencil_pair(_t(a), _t(b), ("diff", lo_a, 1 - lo_a, bc, f), (axis_b, "interp", lo_b, 1 - lo_b, bc, f),
                                   sub, pre_a=_t(pre_a), pre_b=_t(pre_b), post=_t(post)).cpu().numpy()
            np.testing.assert_array_equal(got, want)


def test_pair_argument_validation():
    from xgcm_b200 import ops

    a = torch.zeros((4, 8, 16), device=DEV)
    with pytest.raises(NotImplementedError):
        ops.stencil_pair(a, a.clone(), ("diff", 1, 1, "fill", 0.0), (0, "diff", 1, 0, "fill", 0.0))
    with pytest.raises(ValueError):
        ops.stencil_pair(a, a.clone(), ("diff", 1, 0, "fill", 0.0), (2, "diff", 1, 0, "fill", 0.0))  # axis_b innermost
    with pytest.raises(ValueError):
        ops.stencil_pair(a, torch.zeros((4, 8, 17), device=DEV), ("diff", 1, 0, "fill", 0.0), (0, "diff", 1, 0, "fill", 0.0))


def test_divergence_full_size_samples():
    """C3-sized divergence: sampled blocks against the chain."""
    from xgcm_b200 import _capi, ops

    nz, ny, nx = 75, 2400, 3600
    u = torch.empty((nz, ny, nx), dtype=torch.float32, device=DEV)
    v = torch.empty((nz, ny, nx), dtype=torch.float32, device=DEV)
    ops.fill_uniform(u, 11)
    ops.fill_uniform(v, 12)
    jj = np.arange(ny, dtype=np.float64)[:, None]
    dy = (1e3 * (1 + 0.1 * np.cos(2 * np.pi * jj / ny)) * np.ones((1, nx))).astype(np.float32)
    dx = (1e3 * (1 + 0.1 * np.sin(2 * np.pi * jj / ny)) * np.ones((1, nx))).astype(np.float32)
    ra = (dx * dy).astype(np.float32)
    out = ops.stencil_pair(u, v, ("diff", 0, 1, "periodic", 0.0), (1, "diff", 0, 1, "periodic", 0.0), 0,
                           pre_a=_t(dy), pre_b=_t(dx), post=_t(ra))
    assert _capi.last_launch() == "xg_stencil_pair(tile_tma)"
    rng = np.random.default_rng(5)
    for _ in range(4):
        k = int(rng.integers(0, nz))
        ua, va = u[k].cpu().numpy(), v[k].cpu().numpy()
        want = oracle.stencil_pair("diff", ua, 1, 0, 1, "periodic", 0.0, dy, "diff", va, 0, 0, 1, "periodic", 0.0, dx, 0, ra)
        np.testing.assert_array_equal(out[k].cpu().numpy(), want)
