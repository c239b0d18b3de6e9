"""ΔU of single-monomer moves on adversarial chain states against an extended-precision (long double) restatement of
the changed pair terms.

The rectangle heads×tails forms the moved separation's square from projections on the move,
|r'|² = (r² − 2p_L) + (|D|² + 2p_B) with p_k = (x_k − x_idx)·D (cta_kernels.cuh).  Its rounding grows with the
distance of a pair from the rotated monomer and with |D|, so the states here put close pairs far from the pivot
(hairpins), make |D| large, stretch a chain to n = 700 and run the n = 4096 shape of the two-SM kernel.
The bound is 1e-13 of Σ|changed terms|, ten times tighter than the oracle gate of the other tests, except at n = 4096:
there the staged positions (a block scan on the device, a sequential sum in the reference) already differ enough that
r' formed and squared (the form before the projections) measures 2.2e-13 on this state, as the projections do.
"""
import math

import numpy as np
import pytest

from conftest import both_cases

pytestmark = pytest.mark.gpu

TOL = 1e-13
LD = np.longdouble


def changed_pairs(x, m, idx):
    """(i, j) index arrays of the pairs a move of monomer idx changes: row {idx}×rest and heads×tails."""
    n = len(x)
    heads = np.arange(idx + 1)
    tails = np.arange(idx + 1, n)
    i = np.repeat(heads, len(tails))
    j = np.tile(tails, len(heads))
    lo = np.arange(idx)
    return np.concatenate([i, lo]), np.concatenate([j, np.full(idx, idx)])


def terms(x, m, i, j):
    """4π × dipole-dipole energy of the pairs (i, j) in long double: y³(μi·μj − 3(μi·r)(μj·r) y²), y = 1/|r|."""
    x, m = x.astype(LD), m.astype(LD)
    r = x[i] - x[j]
    r2 = (r * r).sum(axis=1)
    mm = (m[i] * m[j]).sum(axis=1)
    a = (m[i] * r).sum(axis=1)
    b = (m[j] * r).sum(axis=1)
    y2 = 1 / r2
    y3 = y2 / np.sqrt(r2)
    return y3 * (mm - 3 * a * b * y2)


def check_moves(pm, O, n, phi, theta, moves, tol=TOL, **kw):
    pc, oc = both_cases(pm, O, n=n, energy_type="interacting", **kw)
    worst = 0.0
    with pm.Ensemble(pc, replicas=1, seed=5) as ens:
        ens.set_state(0, phi, theta)
        och = O.Chain(oc, phi, theta)
        x0, m0 = och.xs(), och.mus()
        for idx, dphi, dth in moves:
            do = och.delta_u(idx, dphi, dth)
            moved = och.copy()
            moved.move(idx, dphi, dth)
            x1, m1 = moved.xs(), moved.mus()
            i, j = changed_pairs(x0, m0, idx)
            t0, t1 = terms(x0, m0, i, j), terms(x1, m1, i, j)
            dpair = float((t1 - t0).sum() / (4 * LD(math.pi)))
            scale = float((np.abs(t0) + np.abs(t1)).sum() / (4 * LD(math.pi))) + abs(do["du"]) + abs(do["drF"])
            ref = do["du"] + do["drF"] + dpair
            dg = ens.delta_u(0, idx, dphi, dth)
            err = abs(dg["dU"] - ref) / scale
            worst = max(worst, err)
            assert err <= tol, (n, idx, dphi, dth, dg["dU"], ref, err)
    return worst


def hairpin(n, jitter=1e-3, seed=0):
    """Up the z axis, one step along x, back down: monomers i and n−1−i sit about b apart."""
    rng = np.random.default_rng(seed)
    half = n // 2
    theta = np.where(np.arange(n) < half, 0.02, math.pi - 0.02) + rng.uniform(-jitter, jitter, n)
    phi = rng.uniform(-jitter, jitter, n)
    theta[half] = math.pi / 2
    phi[half] = 0.0
    return phi, theta


@pytest.mark.parametrize("n", [256, 512, 1000])
def test_hairpin_near_pairs_far_from_pivot(pm, O, n):
    phi, theta = hairpin(n, seed=n)
    rng = np.random.default_rng(n + 1)
    # pivots near the ends: the close pairs (i, n−1−i) of the middle are far from them; large angle changes → |D| ≈ 2b
    idxs = [1, 2, 5, 17, 40, n - 2, n - 3, n - 18, n // 2 - 3, n // 2 + 2]
    moves = [(int(k), float(rng.uniform(2.0, 3.0)), float(rng.uniform(1.2, 1.5)) * (1 if k < n // 2 else -1))
             for k in idxs]
    check_moves(pm, O, n, phi, theta, moves, E0=1.5, K1=1.0, K2=0.2, Fz=0.4, b=1.0)


def test_near_contact_large_d(pm, O):
    """A tight hairpin (strands 0.6 b apart) and moves that swing a tail by nearly 2b."""
    n = 400
    phi, theta = hairpin(n, jitter=1e-4, seed=3)
    theta[n // 2] = 0.6435   # the turn monomer steps 0.6 b along x
    rng = np.random.default_rng(4)
    moves = [(int(k), math.pi - 0.05, float(rng.uniform(-0.3, 0.3))) for k in (3, 50, 120, 190, 210, 280, 350, 396)]
    check_moves(pm, O, n, phi, theta, moves, E0=2.0, K1=1.0, K2=0.0, Fz=0.0, b=1.0)


def test_stretched_n700(pm, O):
    n = 700
    rng = np.random.default_rng(7)
    phi = rng.uniform(-math.pi, math.pi, n)
    theta = rng.uniform(0.01, 0.15, n)
    moves = [(int(k), float(rng.uniform(-3.0, 3.0)), float(rng.uniform(0.5, 1.5)))
             for k in [0, 1, 63, 64, 200, 349, 350, 351, 500, 636, 698, 699]]
    check_moves(pm, O, n, phi, theta, moves, E0=1.0, K1=1.0, K2=0.1, Fz=2.0, b=0.9)


def test_pair_kernel_shape_n4096(pm, O):
    n = 4096
    rng = np.random.default_rng(11)
    phi = rng.uniform(-math.pi, math.pi, n)
    theta = np.arccos(rng.uniform(-1.0, 1.0, n))
    moves = [(int(k), float(rng.uniform(-2.0, 2.0)), float(rng.uniform(-1.0, 1.0))) for k in [5, 1500, 2047, 2048, 3900]]
    check_moves(pm, O, n, phi, theta, moves, tol=5e-13, E0=1.0, K1=1.0, K2=0.1, Fz=0.5, b=1.0)
