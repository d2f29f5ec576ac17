"""Masked fitting without a GPU: the NumPy restatement of the EM semantics (tests/masked_oracle.py) and the host-side
mask packing."""
import os
import sys

import numpy as np
import pytest

from oracle import aoadmm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from masked_oracle import ao_admm_masked  # noqa: E402


def _ragged_problem(seed, I=6, K=20, R=3, frac=0.2, noise=0.0, Js=None):
    rs = np.random.RandomState(seed)
    Js = rs.randint(10, 30, size=I) if Js is None else Js
    A, C = rs.uniform(0.5, 1.5, (len(Js), R)), rs.standard_normal((K, R))
    X = [(rs.standard_normal((J, R)) * A[i]) @ C.T for i, J in enumerate(Js)]
    X = [x + noise * rs.standard_normal(x.shape) for x in X]
    M = [rs.uniform(size=x.shape) >= frac for x in X]
    return X, M


def test_oracle_all_ones_mask_is_the_unmasked_run():
    X, _ = _ragged_problem(0, noise=0.1)
    kw = dict(non_negative=True, n_iter_max=15, random_state=3, tol=None, absolute_tol=None)
    ref = O.ao_admm(X, 3, **kw)
    got = ao_admm_masked(X, 3, [np.ones(x.shape, dtype=int) for x in X], **kw)
    assert np.array_equal(ref["A"], got["A"]) and np.array_equal(ref["C"], got["C"])
    assert all(np.array_equal(a, b) for a, b in zip(ref["B_is"], got["B_is"]))
    assert ref["rec_errors"] == got["rec_errors"] and ref["regularized_loss"] == got["regularized_loss"]


def test_oracle_observed_error_is_non_increasing_without_penalties():
    """Without penalties and ridge every mode update is an exact least-squares step on F: EM never increases the
    observed error."""
    X, M = _ragged_problem(0, noise=0.1)
    X = [np.where(m, x, np.nan) for x, m in zip(X, M)]  # missing values are never read
    o = ao_admm_masked(X, 3, M, n_iter_max=50, tol=None, absolute_tol=None, random_state=1, l2_penalty=0)
    e = np.asarray(o["rec_errors"])
    assert len(e) == 51 and np.all(np.isfinite(e))
    assert np.all(e[1:] <= e[:-1] * (1 + 1e-12)), np.max(np.diff(e) / e[:-1])
    assert e[-1] < 0.5 * e[0]


def test_oracle_planted_recovery_with_missing_entries():
    """Exact rank-3 ragged data, 20 % missing: the held-out entries come back.  Measured with this seed: observed
    relative error 1.4e-5 after 30 iterations (absolute loss criterion), held-out relative error 5.3e-5."""
    X, M = _ragged_problem(10)
    Xn = [np.where(m, x, np.nan) for x, m in zip(X, M)]
    o = ao_admm_masked(Xn, 3, M, n_iter_max=2000, tol=1e-12, random_state=0)
    assert o["rec_errors"][-1] < 1e-4
    Xh = [(B * o["A"][i]) @ o["C"].T for i, B in enumerate(o["B_is"])]
    held = np.sqrt(sum(np.sum(np.where(m, 0, x - xh) ** 2) for x, xh, m in zip(X, Xh, M)))
    held /= np.sqrt(sum(np.sum(np.where(m, 0, x) ** 2) for x, m in zip(X, M)))
    assert held < 1e-3


def test_mask_packing_to_csr():
    from matcouply_b200._engine import pack_mask

    K = 5
    m0 = np.ones((3, K), dtype=bool)
    m0[1, [4, 0, 2]] = False          # some columns missing (given out of order)
    m1 = np.zeros((0, K), dtype=bool)  # empty slice
    m2 = np.ones((4, K), dtype=np.int64)
    m2[0] = 0                         # a fully missing row
    m2[3, 1] = 0
    p = pack_mask([m0, m1, m2], [(3, K), (0, K), (4, K)])
    assert p.row_ptr.dtype == np.int64 and p.col.dtype == np.int32
    assert p.row_ptr.tolist() == [0, 0, 3, 3, 8, 8, 8, 9]
    assert p.col.tolist() == [0, 2, 4, 0, 1, 2, 3, 4, 1]
    assert p.n_missing == 9 and p.n_observed == 7 * K - 9
    full = pack_mask([np.ones((2, 3))], [(2, 3)])  # torch-free 0/1 floats, nothing missing
    assert full.n_missing == 0 and full.row_ptr.tolist() == [0, 0, 0]


def test_mask_packing_accepts_torch_slices():
    import torch

    from matcouply_b200._engine import pack_mask

    m = torch.tensor([[1, 0, 1], [0, 0, 1]], dtype=torch.bool)
    p = pack_mask([m], [(2, 3)])
    assert p.row_ptr.tolist() == [0, 1, 3] and p.col.tolist() == [1, 0, 1]


def test_mask_validation_messages():
    from matcouply_b200 import cmf_aoadmm, parafac2_aoadmm
    from matcouply_b200._engine import pack_mask

    X = [np.ones((4, 3)), np.ones((2, 3))]
    with pytest.raises(ValueError, match="shape"):
        cmf_aoadmm(X, 2, mask=[np.ones((4, 3)), np.ones((3, 3))])
    with pytest.raises(ValueError, match="slices"):
        cmf_aoadmm(X, 2, mask=[np.ones((4, 3))])
    with pytest.raises(ValueError, match="no observed entry"):
        cmf_aoadmm(X, 2, mask=[np.zeros((4, 3)), np.zeros((2, 3))])
    with pytest.raises(ValueError, match="other than 0 and 1"):
        pack_mask([np.full((4, 3), 0.5)], [(4, 3)])
    for init in ("svd", "threshold_svd", "cp_als"):
        with pytest.raises(ValueError, match="complete data"):
            cmf_aoadmm(X, 2, init=init, mask=[np.ones((4, 3)), np.ones((2, 3))])
        with pytest.raises(ValueError, match="complete data"):
            parafac2_aoadmm(X, 2, init=init, mask=[np.ones((4, 3)), np.ones((2, 3))])
    with pytest.raises(ValueError, match="complete data"):
        ao_admm_masked(X, 2, [np.ones((4, 3)), np.ones((2, 3))], init="svd")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_refill_reference_agrees_with_the_oracle_semantics(dtype):
    """The NumPy statement of one refill launch (``refill_reference``, the yardstick of the kernel tests) against the
    dense formulas of the trajectory oracle: the refilled data is ``masked_fill``; ``‖F_old − X̂‖² − out[0]`` is the
    ``observed_error`` squared (the engine's loss identity); ``out[1]`` is the change of ``‖F‖²``; and a ``Y = F_old C``
    corrected by the refill is ``F_new C``.  Slices of 0 and 1 rows, a fully missing row and a complete row included."""
    from masked_oracle import masked_fill, observed_error, refill_reference

    rs = np.random.RandomState(5)
    Js, K, R = [7, 0, 12, 1, 9], 37, 4
    X, M = _ragged_problem(2, K=K, R=R, Js=Js, frac=0.3)
    M[2][3], M[2][4] = False, True  # a fully missing row and a complete one
    X = [x.astype(dtype).astype(np.float64) for x in X]
    A, C = rs.uniform(size=(len(Js), R)), rs.standard_normal((K, R))
    Bs = [rs.standard_normal((J, R)) for J in Js]
    F_old = [np.where(m, x, rs.standard_normal(x.shape).astype(dtype)) for x, m in zip(X, M)]  # any previous fill
    miss = ~np.concatenate(M, 0)
    row_ptr = np.concatenate([[0], np.cumsum(miss.sum(axis=1))])
    rows, col = np.nonzero(miss)
    gor = np.repeat(np.arange(len(Js)), Js)
    Fo, B = np.concatenate(F_old, 0), np.concatenate(Bs, 0)
    Y_old = Fo @ C
    ref = refill_reference(Fo[rows, col], row_ptr, col, gor, A, B, C, Y=Y_old, dtype=dtype)

    Fn = Fo.copy()
    Fn[rows, col] = ref["new"]
    want = np.concatenate(masked_fill([np.where(m, x, 0.0) for x, m in zip(X, M)], M, A, Bs, C), 0)
    tol = 1e-13 if dtype == np.float64 else 1e-6
    np.testing.assert_allclose(Fn, want, rtol=tol, atol=tol)
    np.testing.assert_array_equal(Fn[~miss], Fo[~miss])
    Xh = np.concatenate([(b * A[i]) @ C.T for i, b in enumerate(Bs)], 0)
    sse_obs = np.sum((Fo - Xh) ** 2) - ref["sums"][0]
    # fp32: d is taken against the stored (rounded) x̂, as the kernel does
    floor = 1e-12 if dtype == np.float64 else 1e-6
    assert abs(sse_obs - observed_error(X, M, A, Bs, C) ** 2) <= floor * np.sum(Fo ** 2 + Xh ** 2)
    assert abs(ref["sums"][1] - (np.sum(Fn ** 2) - np.sum(Fo ** 2))) <= 1e-13 * ref["sums_scale"]
    assert np.all(np.abs(ref["Y"] - Fn @ C) <= (1e-12 if dtype == np.float64 else 1e-6) * (np.abs(Fn) @ np.abs(C)))
