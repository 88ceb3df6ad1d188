"""Known-answer test of the hot kernel: one Jacobi sweep on linear systems captured from INSIDE the
reference (tests/golden/jacobi_kat.npz: the compact-row matrix, b, x that Water::JacobiWaterCPU saw, and
the x it produced), and on seeded synthetic systems whose answer is a numpy restatement of the row
(sf3d_row_jacobi, water.cpp:570-596).  The row arithmetic has no libm call, so x must be bit-identical
everywhere (the product is compiled with -fmad=false; numpy multiplies and subtracts without contraction);
the norm differs only by summation order.

The synthetic sizes sit at the edges of the product's sweep grid (256 threads a block, at most 148 x 8 = 1184
blocks): one partial block, exactly one block, one row into a second block, one row short of / exactly at /
one past one row per thread of the full grid, and 2 000 003 rows (6-7 rows per thread, ragged last pass, a
fold of 1184 partials by 256 threads)."""
import math
from pathlib import Path

import numpy as np
import pytest

from criteria3d_b200 import SoilFluxes3D
from oracle import ORACLE_LIB, REFERENCE_LIB

KAT = Path(__file__).parent / "golden" / "jacobi_kat.npz"
SIZES = (1, 255, 256, 257, 303_103, 303_104, 303_105, 2_000_003)
NORM_REL_SYNTHETIC = 1e-13      # the device sums non-negative terms in a tree of depth <= ~30: several times its rounding


def _captured():
    with np.load(KAT) as z:
        d = {k: z[k] for k in z.files}
    for k in (0, 1):
        norm = float(d[f"norm{k}"])
        yield (int(d[f"ns{k}"]), d[f"ncols{k}"], d[f"col{k}"], d[f"val{k}"], d[f"b{k}"], d[f"z{k}"], d[f"x_in{k}"],
               d[f"x_out{k}"], norm, norm)


def _restated_sweep(ns, ncols, col, val, b, z, x):
    """sf3d_row_jacobi on every row, same column order; returns (x_new, the rows' norm terms)"""
    n = len(b)
    rows = np.arange(n)
    xnew = b.copy()
    for c in range(1, 11):
        has = c < ncols
        xnew = np.where(has, xnew - val[:, c] * x[np.where(has, col[:, c], rows)], xnew)
    surface = rows < ns
    xnew = np.where(surface & (xnew < z), z, xnew)
    term = np.abs(xnew - x)
    psi = np.abs(xnew - z)
    term = np.where(psi > 1.0, term * (1.0 / np.where(psi > 1.0, psi, 1.0)), term)
    return xnew, term


def _synthetic(n, seed=20261020):
    """A seeded system of n rows: a surface prefix on which the clamp to z binds on some rows and not on others,
    rows on both sides of |x_new - z| = 1, 1 to 11 columns per row, column indices spread over the whole vector
    (0 and n-1 included), weakly diagonally dominant values."""
    rng = np.random.default_rng(seed + n)
    rows = np.arange(n, dtype=np.int64)
    ns = (n + 2) // 3
    ncols = rng.integers(1, 12, n).astype(np.uint8)
    ncols[0], ncols[-1] = 11, 1
    if n > 2:
        ncols[1] = 11
    col = rng.integers(0, n, (n, 11), dtype=np.uint32)
    col[:, 0] = rows
    near = rng.random((n, 11)) < 0.3                      # some index neighbours too, as a catchment's links are
    near[:, 0] = False
    col[near] = ((rows[:, None] + rng.integers(-2, 3, (n, 11), dtype=np.int8)) % n)[near]
    col[::7, 1] = 0
    col[3::7, 2] = n - 1
    val = rng.uniform(-0.1, 0.08, (n, 11))
    val[:, 0] = 1.0
    absent = np.arange(11)[None, :] >= ncols[:, None]
    col[absent] = 0xFFFFFFFF                              # absent entries must never be read
    val[absent] = np.nan
    x = 100.0 + rng.uniform(-3.0, 3.0, n)
    b = x + rng.uniform(-2.5, 2.5, n)
    xfree, _ = _restated_sweep(0, ncols, col, val, b, np.zeros(n), x)
    # z relative to the unclamped update: above it (the clamp binds on surface rows), or 0.5 / 3 below it
    z = xfree + rng.choice([2.0, 0.5, -0.5, -3.0], n)
    xnew, term = _restated_sweep(ns, ncols, col, val, b, z, x)
    if n >= 255:
        clamped = xnew[:ns] != xfree[:ns]
        psi = np.abs(xnew - z)
        assert clamped.any() and not clamped.all() and (psi > 1.0).any() and ((psi > 0.0) & (psi < 1.0)).any()
        read = col[:, 1:][~absent[:, 1:]]
        assert (read == 0).any() and (read == n - 1).any()
    seq = float(np.cumsum(term)[-1]) / n                   # row order, one accumulator (the CPU implementations)
    return ns, ncols, col, val, b, z, x, xnew, math.fsum(term) / n, seq


def _check(sf, norm_rel, synthetic_norm_rel=None):
    """norm_rel: against the captured norms.  synthetic_norm_rel: against the exact sum of the synthetic terms;
    None = the implementation sums in row order with one accumulator, so its norm is that sequential sum exactly."""
    cases = [(c, norm_rel) for c in _captured()] + [(_synthetic(n), synthetic_norm_rel) for n in SIZES]
    for (ns, ncols, col, val, b, z, x_in, x_ref, norm_exact, norm_seq), rel in cases:
        n = len(b)
        x, norm = sf.jacobi_sweep(ns, ncols, col, val, b, z, x_in)
        assert np.array_equal(x, x_ref), f"n={n}: max diff {np.max(np.abs(x - x_ref))}"
        if rel is None:
            assert norm == norm_seq, f"n={n}: norm {norm!r} != {norm_seq!r}"
        else:
            assert abs(norm - norm_exact) <= rel * abs(norm_exact), f"n={n}: norm {norm!r} vs {norm_exact!r}"
        assert n == 1 or ((ncols < 11).any() and (ncols == 11).any())   # ragged rows and full rows are both present


def test_restatement_sweep_is_bit_exact():
    if not ORACLE_LIB.exists():
        pytest.skip("oracle library not built")
    _check(SoilFluxes3D(ORACLE_LIB), 0.0)


def test_reference_reproduces_its_own_capture():
    if not REFERENCE_LIB.exists():
        pytest.skip("oracle/_ref not built here")
    from criteria3d_b200.synth import Catchment, setup
    ref = SoilFluxes3D(REFERENCE_LIB)
    setup(ref, Catchment(4, 4, 2), threads=1)                   # the real sweep needs an initialised solver object
    _check(ref, 0.0)


@pytest.mark.gpu
def test_product_sweep_is_bit_exact_on_x(product):
    _check(product, 1e-12, NORM_REL_SYNTHETIC)
