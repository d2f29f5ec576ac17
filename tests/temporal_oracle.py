"""NumPy fp64 restatement of ``TemporalSmoothnessPenalty``, the yardstick of tests/test_temporal_cpu.py and
tests/test_gpu_temporal.py.

The reference has no such penalty.  ``TemporalSmoothnessP`` plugs into the unchanged oracle drivers
(``oracle.aoadmm_oracle.ao_admm(..., regs=...)`` and ``masked_oracle.ao_admm_masked``) as one more ``OraclePenalty``:

    value(B_0..B_{I-1}) = lam * sum_{i>=1} ||B_i - B_{i-1}||_F^2
    prox_list(V, rho)   = z with (diag(rho) + 2 lam L) z = rho o v for every entry (j, r), L the path-graph Laplacian

solved directly with ``scipy.linalg.solve_banded`` on the stacked (I, J*R) array.  ``partition_solve`` restates the
chunked (and per-rank) partition solve of csrc/prox_temporal.cu in NumPy, so that its algebra is pinned on the CPU.
"""
import numpy as np
from scipy.linalg import solve_banded

from oracle import aoadmm_oracle as O


def system_bands(rho, lam):
    """The tridiagonal T = diag(rho) + 2 lam L in ``solve_banded``'s (1, 1) layout."""
    rho = np.asarray(rho, dtype=np.float64)
    I = rho.shape[0]
    deg = np.zeros(I)
    deg[1:] += 1
    deg[:-1] += 1
    ab = np.zeros((3, I))
    ab[0, 1:] = -2 * lam
    ab[1] = rho + 2 * lam * deg
    ab[2, :-1] = -2 * lam
    return ab


def laplacian(I):
    """Path-graph Laplacian of I nodes (dense)."""
    L = np.zeros((I, I))
    for i in range(1, I):
        L[i, i] += 1
        L[i - 1, i - 1] += 1
        L[i, i - 1] = L[i - 1, i] = -1
    return L


def prox_stacked(V, rho, lam):
    """V: (I, n) stacked slices (row i = B_i flattened); rho: I values.  Returns z."""
    V = np.asarray(V, dtype=np.float64)
    rho = np.broadcast_to(np.asarray(rho, dtype=np.float64), (V.shape[0],))
    if V.shape[0] == 1:
        return V.copy()
    return solve_banded((1, 1), system_bands(rho, lam), rho[:, None] * V)


def value_stacked(X, lam):
    X = np.asarray(X, dtype=np.float64)
    return lam * float(np.sum((X[1:] - X[:-1]) ** 2)) if X.shape[0] > 1 else 0.0


def cond_bound(rho, lam):
    """Upper bound on the 2-norm condition number of T (Gershgorin): (max rho + 8 lam) / min rho."""
    rho = np.asarray(rho, dtype=np.float64)
    return (rho.max() + 8 * lam) / rho.min()


def _block_solve(rho, lam, rhs, has_left, has_right):
    """T_block^-1 rhs for a block of consecutive slices whose diagonal keeps the degree in the whole graph."""
    I = rho.shape[0]
    deg = np.zeros(I)
    deg[1:] += 1
    deg[:-1] += 1
    deg[0] += 1 if has_left else 0
    deg[-1] += 1 if has_right else 0
    ab = np.zeros((3, I))
    ab[0, 1:] = -2 * lam
    ab[1] = rho + 2 * lam * deg
    ab[2, :-1] = -2 * lam
    return solve_banded((1, 1), ab, rhs)


def partition_solve(V, rho, lam, bounds):
    """The partition (spike) solve of (diag(rho) + 2 lam L) z = rho o v with blocks [bounds[k], bounds[k+1]): every
    block is solved with zero outer boundaries, its spike vectors alpha = T_q^-1 (2 lam e_first) and beta = T_q^-1
    (2 lam e_last) give the 2 x (#blocks) reduced system in the block ends, and z_q = y_q + alpha_q z_left +
    beta_q z_right.  This is the algebra of the chunks and of the ranks of a sharded run alike."""
    V = np.asarray(V, dtype=np.float64)
    I, n = V.shape
    rho = np.broadcast_to(np.asarray(rho, dtype=np.float64), (I,)).copy()
    blocks = [(a, b) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
    Qn = len(blocks)
    ys, alphas, betas = [], [], []
    for a, b in blocks:
        m = b - a
        e0, e1 = np.zeros((m, 1)), np.zeros((m, 1))
        e0[0], e1[-1] = 2 * lam, 2 * lam
        hl, hr = a > 0, b < I
        ys.append(_block_solve(rho[a:b], lam, rho[a:b, None] * V[a:b], hl, hr))
        alphas.append(_block_solve(rho[a:b], lam, e0, hl, hr)[:, 0])
        betas.append(_block_solve(rho[a:b], lam, e1, hl, hr)[:, 0])
    # reduced system in w_q = (first_q, last_q):  w_q - a_q last_{q-1} - b_q first_{q+1} = (y_q[0], y_q[-1])
    S = np.eye(2 * Qn)
    rhs = np.zeros((2 * Qn, n))
    for q in range(Qn):
        rhs[2 * q], rhs[2 * q + 1] = ys[q][0], ys[q][-1]
        if q > 0:
            S[2 * q, 2 * q - 1] -= alphas[q][0]
            S[2 * q + 1, 2 * q - 1] -= alphas[q][-1]
        if q < Qn - 1:
            S[2 * q, 2 * q + 2] -= betas[q][0]
            S[2 * q + 1, 2 * q + 2] -= betas[q][-1]
    w = np.linalg.solve(S, rhs)
    z = np.empty_like(V)
    for q, (a, b) in enumerate(blocks):
        left = w[2 * q - 1] if q > 0 else np.zeros(n)
        right = w[2 * q + 2] if q < Qn - 1 else np.zeros(n)
        z[a:b] = ys[q] + alphas[q][:, None] * left + betas[q][:, None] * right
    return z


class TemporalSmoothnessP(O.OraclePenalty):
    """lam * sum_i ||B_i - B_{i-1}||_F^2 over the slice order (mode 1)."""

    name = "temporal_smoothness"
    matrixwise = True

    def __init__(self, smoothness_reg, **kw):
        super().__init__(**kw)
        self.smoothness_reg = float(smoothness_reg)

    def prox_list(self, Ms, rhos, auxes):
        shapes = [np.shape(M) for M in Ms]
        V = np.stack([np.asarray(M, dtype=np.float64).reshape(-1) for M in Ms])
        z = prox_stacked(V, np.asarray(rhos, dtype=np.float64), self.smoothness_reg)
        return [zi.reshape(s) for zi, s in zip(z, shapes)]

    def prox(self, M, rho, aux):
        raise AttributeError("TemporalSmoothnessPenalty acts on the list of mode-1 factor matrices only")

    def value(self, x):
        if isinstance(x, np.ndarray):
            raise TypeError("the temporal smoothness penalty needs the list of factor matrices")
        return value_stacked(np.stack([np.asarray(b, dtype=np.float64).reshape(-1) for b in x]), self.smoothness_reg)
