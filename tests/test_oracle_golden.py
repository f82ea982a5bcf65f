"""Pin the oracle: golden vectors produced by the reference's own kernels + the known answers
transcribed from the reference's tests and docs.  CPU only."""

import json
import os

import numpy as np
import pytest

from oracle import stencil as oracle

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_gridops_table_matches_oracle_table():
    """Signatures / halo widths of xgcm/gridops.py:27-215."""
    table = json.load(open(os.path.join(GOLDEN, "gridops_table.json")))
    for name, entry in table.items():
        op, src, _, dst = name.split("_")
        if entry["padding_width"] is None:
            assert name == "diff_left_to_inner"  # gridops.py:68-70
            continue
        assert entry["signature"] == f"(X:{src})->(X:{dst})"
        assert tuple(entry["padding_width"]["X"]) == oracle.PADDING_WIDTH[(src, dst)]


def test_oracle_equals_reference_gridops_golden():
    g = np.load(os.path.join(GOLDEN, "gridops_ref.npz"))
    n = 0
    for key in g.files:
        if key.startswith("input|"):
            continue
        name, dt, axis, bc, fill = key.split("|")
        op, src, _, dst = name.split("_")
        lo, hi = oracle.PADDING_WIDTH[(src, dst)]
        a = g[f"input|{dt}|{name}"]
        got = oracle.stencil2(op, a, int(axis), lo, hi, bc if (lo or hi) else None, float(fill))
        assert got.dtype == g[key].dtype
        np.testing.assert_array_equal(got, g[key])
        n += 1
    assert n == 32 * 2 * 3 * 4


def test_oracle_equals_reference_interp1d_golden():
    g = np.load(os.path.join(GOLDEN, "interp1d_ref.npz"))
    for tag in ("float32", "float64"):
        phi, theta, target = g[f"phi|{tag}"], g[f"theta|{tag}"], g[f"target|{tag}"]
        for mask in (0, 1):
            for bypass in (0, 1):
                want = g[f"out|{tag}|{mask}|{bypass}|0"]
                got = oracle.vinterp_linear(phi, theta, target, -1, bool(mask), bool(bypass))
                assert got.dtype == want.dtype
                np.testing.assert_array_equal(got, want)
        want = g[f"out|{tag}|1|0|1"]
        got = oracle.vinterp_linear(phi, g[f"log_theta|{tag}"], g[f"log_target|{tag}"], -1, True, False, True)
        np.testing.assert_array_equal(got, want)


def test_oracle_equals_reference_conservative_golden():
    g = np.load(os.path.join(GOLDEN, "conservative_ref.npz"))
    for tag in ("float32", "float64"):
        phi, theta, bins = g[f"phi|{tag}"], g[f"theta|{tag}"], g[f"bins|{tag}"]
        for d, b in (("up", bins), ("down", bins[::-1].copy())):
            got = oracle.vinterp_conservative(phi, theta, b, -1)
            assert got.dtype == g[f"out|{tag}|{d}"].dtype
            np.testing.assert_array_equal(got, g[f"out|{tag}|{d}"])


def test_oracle_equals_live_reference_kernels():
    """tests/golden/live_kernels_ref.npz: what the reference's own kernels return, recorded by
    oracle/make_golden.py — every GridUFunc along every axis of a periodic fp64 field, and
    interp_1d_linear on columns with every third one decreasing."""
    table = json.load(open(os.path.join(GOLDEN, "gridops_table.json")))
    g = np.load(os.path.join(GOLDEN, "live_kernels_ref.npz"))
    a = g["a"]
    for op in ("diff", "interp", "min", "max"):
        for (src, dst), (lo, hi) in oracle.PADDING_WIDTH.items():
            name = f"{op}_{src}_to_{dst}"
            assert table[name]["padding_width"] == {"X": [lo, hi]}
            for axis in range(3):
                got = oracle.stencil2(op, a, axis, lo, hi, "periodic" if (lo or hi) else None)
                want = g[f"{name}|{axis}"]
                assert got.dtype == want.dtype
                np.testing.assert_array_equal(got, want)
    phi, theta, tg = g["phi"], g["theta"], g["target"]
    for mask in (False, True):
        want = g[f"interp_1d_linear|{int(mask)}"]
        np.testing.assert_array_equal(oracle.vinterp_linear(phi, theta, tg, -1, mask), want)


# ---- known answers of the reference's tests / docs -------------------------------------------
def test_doc_boundary_conditions_known_answers():
    """docs/boundary_conditions.md:61,110-113: last diff is 0 / -2 / -3 / +2."""
    x_g = np.arange(0.5, 9.0, 1.0)  # wait: x_g = 0.5 ... 8.5 (9 points)
    g = np.sqrt(x_g + 0.5) + np.sin((x_g - 0.5) * 2 * np.pi / 8)
    # left -> center needs one halo cell above
    assert oracle.stencil2("diff", g, 0, 0, 1, "extend")[-1] == 0.0
    np.testing.assert_allclose(oracle.stencil2("diff", g, 0, 0, 1, "periodic")[-1], -2.0, atol=1e-12)
    np.testing.assert_allclose(oracle.stencil2("diff", g, 0, 0, 1, "fill", 0.0)[-1], -3.0, atol=1e-12)
    np.testing.assert_allclose(oracle.stencil2("diff", g, 0, 0, 1, "fill", 5.0)[-1], 2.0, atol=1e-12)


def test_center_to_outer_extend_linspace():
    """xgcm/test/test_grid_ufunc.py:1326-1338."""
    a = np.linspace(1, 10, 10)
    got = oracle.stencil2("interp", a, 0, 1, 1, "extend")
    np.testing.assert_array_equal(got, np.concatenate([[1.0], np.arange(1.5, 10, 1.0), [10.0]]))


def test_center_to_left_fill_arange():
    """xgcm/test/test_grid_ufunc.py:1227-1273: fill 0 / 1 / 10 on arange(9), center -> left."""
    a = np.arange(9.0)
    for fill in (0.0, 1.0, 10.0):
        want_diff = np.diff(np.concatenate([[fill], a]))
        np.testing.assert_array_equal(oracle.stencil2("diff", a, 0, 1, 0, "fill", fill), want_diff)
        want_interp = 0.5 * (np.concatenate([[fill], a])[:-1] + np.concatenate([[fill], a])[1:])
        np.testing.assert_array_equal(oracle.stencil2("interp", a, 0, 1, 0, "fill", fill), want_interp)


def test_cumsum_center_to_outer_fill():
    """xgcm/test/test_grid.py:549-552: [0, 1, 3, 6, ...]."""
    a = np.arange(1.0, 15.0)
    trim, (plo, phi) = oracle.CUMSUM_TABLE_FWD[("center", "outer")]
    got = oracle.cumscan(a, 0, False, trim, plo, phi, "fill", 0.0)
    np.testing.assert_array_equal(got, np.concatenate([[0.0], np.cumsum(a)]))


def test_cumsum_extend_replicates_cumsummed_edge():
    """grid.py:1385-1391: the halo is taken from the cumsum'd data."""
    a = np.arange(1.0, 6.0)
    trim, (plo, phi) = oracle.CUMSUM_TABLE_FWD[("center", "left")]
    got = oracle.cumscan(a, 0, False, trim, plo, phi, "extend")
    np.testing.assert_array_equal(got, [1.0, 1.0, 3.0, 6.0, 10.0])
    trim, (plo, phi) = oracle.CUMSUM_TABLE_REV[("center", "right")]
    got = oracle.cumscan(a, 0, True, trim, plo, phi, "fill", 0.0)
    np.testing.assert_array_equal(got, [14.0, 12.0, 9.0, 5.0, 0.0])


def test_transform_cases_golden():
    """The linear / log entries of the `cases` dict of xgcm/test/test_transform.py:41-683."""
    cases = json.load(open(os.path.join(GOLDEN, "transform_cases.json")))

    def arr(v):
        return np.array([np.nan if x is None else x for x in v], dtype=float)

    checked = 0
    for name, c in cases.items():
        if "multidim_target" in name or c["transform_kwargs"]["method"] == "conservative":
            continue
        kw = c["transform_kwargs"]
        phi = arr(c["source_data"][1])
        if kw.get("target_data"):
            assert c["source_additional_data"][0] == kw["target_data"]
            theta = arr(c["source_additional_data"][1])
        else:
            theta = arr(c["source_coord"][1])
        target = arr(c["target_data"][1])
        want = arr(c["expected_data"][1])
        for ii in c.get("expected_data_mask_index", []):
            want[ii] = np.nan
        got = oracle.vinterp_linear(phi, theta, target, 0, kw.get("mask_edges", True),
                                    False, kw["method"] == "log")
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6, equal_nan=True, err_msg=name)
        checked += 1
    assert checked >= 10


def _numpy_simd_log():
    """np.log(float32) runs numpy's SIMD algorithm only on x86 with AVX2+FMA3 / AVX512F (elsewhere: libm)."""
    try:
        from numpy._core._multiarray_umath import __cpu_features__ as f
    except Exception:
        return False
    return bool(f.get("AVX512F") or (f.get("AVX2") and f.get("FMA3")))


def test_log32_port_is_numpys():
    """The float32 log the device uses for method="log" (oracle.log32_port restates it in numpy) is numpy's own:
    bit-identical on every exponent, denormals, the reduction threshold and the neighbourhood of 1."""
    if not _numpy_simd_log():
        pytest.skip("np.log(float32) does not take numpy's SIMD path on this CPU")
    rng = np.random.default_rng(3)
    man = np.concatenate([np.arange(0x3504F3 - 64, 0x3504F3 + 64), np.arange(0, 64),
                          np.arange(0x7FFFFF - 64, 0x7FFFFF + 1)]).astype(np.uint32)
    exp = np.arange(0, 255, dtype=np.uint32)
    bits = ((exp[:, None] << 23) | man[None, :]).reshape(-1)
    bits = np.concatenate([bits[bits != 0], rng.integers(1, 0x7F800000, size=3_000_000, dtype=np.int64).astype(np.uint32)])
    x = bits.view(np.float32)
    with np.errstate(all="ignore"):
        want = np.log(x)
    got = oracle.log32_port(x)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    special = np.array([0.0, -0.0, -1.0, np.inf, np.nan], np.float32)
    with np.errstate(all="ignore"):
        np.testing.assert_array_equal(oracle.log32_port(special), np.log(special))
