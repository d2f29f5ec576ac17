"""CPU checks of the TemporalSmoothnessPenalty restatement (tests/temporal_oracle.py) and of the penalty's host logic.

The reference has no temporal smoothness penalty, so the NumPy oracle is pinned here: its prox satisfies the KKT
conditions, agrees with the reference-pinned GeneralizedL2 penalty applied to the stacked slices, and the partition
solve the CUDA kernel implements gives the direct solution."""
import os
import sys

import numpy as np
import pytest

from oracle import aoadmm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import temporal_oracle as T  # noqa: E402


@pytest.mark.parametrize("I", [1, 2, 3, 7, 40])
@pytest.mark.parametrize("ratio", [1e-6, 1e-2, 1.0, 1e3, 1e6])
def test_prox_satisfies_the_kkt_conditions(I, ratio):
    rs = np.random.RandomState(I)
    rho = 10 ** rs.uniform(-2, 2, size=I)
    lam = ratio * float(np.median(rho))
    V = rs.standard_normal((I, 13))
    z = T.prox_stacked(V, rho, lam)
    resid = 2 * lam * T.laplacian(I) @ z + rho[:, None] * (z - V)
    scale = np.abs(rho[:, None] * V).max() + 2 * lam * 4 * np.abs(z).max()
    assert np.abs(resid).max() <= 1e-12 * scale


def test_constant_rho_equals_the_generalized_l2_penalty_on_the_stacked_slices():
    """x^T (lam L) x per column of the stacked (I, J*R) matrix: the reference's own GL2 prox and value."""
    rs = np.random.RandomState(0)
    I, J, R, lam, rho = 9, 5, 3, 0.7, 2.3
    Bs = [rs.standard_normal((J, R)) for _ in range(I)]
    stacked = np.stack([b.reshape(-1) for b in Bs])
    gl2 = O.GeneralizedL2P(lam * T.laplacian(I))
    pen = T.TemporalSmoothnessP(lam)
    got = np.stack([z.reshape(-1) for z in pen.prox_list(Bs, [rho] * I, None)])
    assert np.allclose(got, gl2.prox(stacked, rho, None), rtol=1e-12, atol=1e-12)
    assert np.isclose(pen.value(Bs), gl2.value(stacked), rtol=1e-12)


@pytest.mark.parametrize("bounds", [
    "chunks1",      # one slice per block
    "chunks4",      # blocks of 4, last one shorter
    "single",       # one block: the direct solve
    "ranks",        # uneven per-rank blocks, as in a sharded run
])
def test_partition_solve_equals_the_direct_solve(bounds):
    rs = np.random.RandomState(3)
    I = 23
    rho = 10 ** rs.uniform(-2, 2, size=I)
    V = rs.standard_normal((I, 11))
    cut = dict(chunks1=list(range(I + 1)), chunks4=list(range(0, I, 4)) + [I], single=[0, I],
               ranks=[0, 1, 1, 9, 10, 23])[bounds]
    for lam in (1e-4, 0.3, 50.0):
        want = T.prox_stacked(V, rho, lam)
        got = T.partition_solve(V, rho, lam, cut)
        assert np.allclose(got, want, rtol=1e-11, atol=1e-11 * np.abs(want).max()), (bounds, lam)


def test_single_slice_is_the_identity_and_has_no_value():
    V = np.arange(6.0).reshape(1, 6)
    assert np.array_equal(T.prox_stacked(V, [3.0], 5.0), V)
    assert T.value_stacked(V, 5.0) == 0.0


def test_constructor_validation_and_single_matrix_refusal():
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    for bad in (0, -1.0):
        with pytest.raises(ValueError, match="must be positive"):
            TemporalSmoothnessPenalty(bad)
    pen = TemporalSmoothnessPenalty(0.5)
    assert "smoothness_reg=0.5" in repr(pen)
    with pytest.raises(TypeError):
        pen.penalty(np.ones((3, 2)))
    with pytest.raises(ValueError, match=r"found heights \[3, 4\]"):
        pen._check_heights([3, 4, 3])
    assert pen._check_heights([5, 5]) == 5
