"""NumPy fp64 restatement of masked fitting (EM with one refill per outer iteration), the yardstick of
tests/test_masked_cpu.py, tests/test_gpu_masked.py and tests/test_gpu_masked_width.py.

It drives the oracle's own mode solvers, penalties and diagnostics (oracle/aoadmm_oracle.py, unchanged) with the
masked semantics of ``cmf_aoadmm(..., mask=...)``:

1. F⁽⁰⁾ = M∘X + (1−M)∘X̂(A₀, B₀, C₀) from the start factors (values of X at missing positions are never read);
2. outer iteration t: the unchanged B-, C- and A-updates on F⁽ᵗ⁻¹⁾, then F⁽ᵗ⁾ = M∘X + (1−M)∘X̂(Aₜ, Bₜ, Cₜ);
3. rec_errors[t] = ‖M∘(X − X̂ₜ)‖ / ‖M∘X‖, evaluated densely (not through the expanded identity the engine uses), and
   the reference's loss, gaps and stopping rule with that error.

A mask without a missing entry is the unmasked oracle run itself.
"""
import numpy as np

from oracle import aoadmm_oracle as O


def _model(A, Bs, C):
    return [(B * A[i]) @ C.T for i, B in enumerate(Bs)]


def masked_fill(X_obs, obs, A, Bs, C):
    """F = M∘X + (1−M)∘X̂(A, B, C)."""
    return [np.where(M, X, Xh) for X, M, Xh in zip(X_obs, obs, _model(A, Bs, C))]


def observed_error(X_obs, obs, A, Bs, C):
    """‖M∘(X − X̂)‖, evaluated densely."""
    return np.sqrt(sum(np.sum(np.where(M, X - Xh, 0.0) ** 2) for X, M, Xh in zip(X_obs, obs, _model(A, Bs, C))))


def refill_reference(x_old, row_ptr, col, gor, A, B, C, Y=None, dtype=np.float64, chunk=1 << 20):
    """The contract of one ``b2_mask_refill`` launch (``_ops.mask_refill``) in float64, over the CSR list
    ``(row_ptr, col)`` of the missing entries and their current values ``x_old`` (in CSR order):

    - the missing entry (n, k) becomes x̂ = (B[n] ∘ A[gor[n]]) · C[k], rounded to ``dtype``; d = x̂ − x_old;
    - Y[n] += Σ_k d·C[k] (rounded to ``dtype``);
    - out[0] += Σ d², out[1] += Σ (x̂² − x_old²).

    Returns dict(xhat = x̂ before the rounding, new = x̂ as stored, scale = |B∘A[gor]|·|C| per entry,
    Y = the updated Y or None, yscale = |Y| + Σ_k |d|·|C[k]| per row, sums = (Σ d², Σ (x̂² − x_old²)),
    sums_scale = Σ (x̂² + x_old²))."""
    import scipy.sparse as sp

    row_ptr, col = np.asarray(row_ptr, dtype=np.int64), np.asarray(col, dtype=np.int64)
    N = len(row_ptr) - 1
    rows = np.repeat(np.arange(N), np.diff(row_ptr))
    W = np.asarray(B, dtype=np.float64) * np.asarray(A, dtype=np.float64)[np.asarray(gor)[:N]]
    C = np.asarray(C, dtype=np.float64)
    xhat, scale = np.empty(len(col)), np.empty(len(col))
    for p in range(0, len(col), chunk):  # bounded temporaries at millions of entries
        r, k = rows[p:p + chunk], col[p:p + chunk]
        xhat[p:p + chunk] = np.einsum("er,er->e", W[r], C[k])
        scale[p:p + chunk] = np.einsum("er,er->e", np.abs(W[r]), np.abs(C[k]))
    new = xhat.astype(dtype).astype(np.float64)
    x_old = np.asarray(x_old, dtype=np.float64)
    d = new - x_old
    res = dict(xhat=xhat, new=new, scale=scale, Y=None, yscale=None,
               sums=(float(np.sum(d * d)), float(np.sum(new * new - x_old * x_old))),
               sums_scale=float(np.sum(new * new + x_old * x_old)))
    if Y is not None:
        K = C.shape[0]
        D = sp.csr_matrix((d, col, row_ptr), shape=(N, K))  # Σ_k d·C[k] per row as one sparse product
        Y = np.asarray(Y, dtype=np.float64)
        res["Y"] = (Y + D @ C).astype(dtype).astype(np.float64)
        res["yscale"] = np.abs(Y) + abs(D) @ np.abs(C)
    return res


def ao_admm_masked(matrices, rank, mask, n_iter_max=1000, l2_penalty=None, l1_penalty=None, non_negative=None,
                   unimodal=None, l2_norm_bound=None, lower_bound=None, upper_bound=None, parafac2=None, regs=None,
                   feasibility_penalty_scale=1, constant_feasibility_penalty=False, aux_init="random_uniform",
                   dual_init="random_uniform", random_state=None, tol=1e-8, absolute_tol=1e-10, feasibility_tol=1e-4,
                   inner_n_iter_max=5, update_A=True, update_B_is=True, update_C=True, return_errors=True, init=None,
                   trajectory=None, inner_tol=None, generalized_l2_penalty=None, tv_penalty=None):
    """``oracle.aoadmm_oracle.ao_admm`` with a mask (list of per-slice 0/1 or bool arrays, 1 = observed); same
    arguments and result dict."""
    kw = dict(n_iter_max=n_iter_max, l2_penalty=l2_penalty, l1_penalty=l1_penalty, non_negative=non_negative,
              unimodal=unimodal, l2_norm_bound=l2_norm_bound, lower_bound=lower_bound, upper_bound=upper_bound,
              parafac2=parafac2, regs=regs, feasibility_penalty_scale=feasibility_penalty_scale,
              constant_feasibility_penalty=constant_feasibility_penalty, aux_init=aux_init, dual_init=dual_init,
              random_state=random_state, tol=tol, absolute_tol=absolute_tol, feasibility_tol=feasibility_tol,
              inner_n_iter_max=inner_n_iter_max, update_A=update_A, update_B_is=update_B_is, update_C=update_C,
              return_errors=return_errors, init=init, trajectory=trajectory, inner_tol=inner_tol,
              generalized_l2_penalty=generalized_l2_penalty, tv_penalty=tv_penalty)
    if isinstance(init, str) and init != "random":
        raise ValueError(f'init="{init}" needs complete data and cannot be combined with a mask')
    obs = [np.asarray(M) != 0 for M in mask]
    if all(M.all() for M in obs):
        return O.ao_admm(matrices, rank, **kw)  # no missing entry: exactly the unmasked run

    rs = random_state if isinstance(random_state, np.random.RandomState) else (
        np.random.mtrand._rand if random_state is None else np.random.RandomState(random_state))
    X_obs = [np.where(M, np.asarray(X, dtype=np.float64), 0.0) for X, M in zip(matrices, obs)]  # M∘X
    I, K = len(X_obs), X_obs[0].shape[1]
    if init is None or init == "random":  # decomposition.py:31-39 — draw order A, C, B_i
        A = rs.uniform(size=(I, rank))
        C = rs.uniform(size=(K, rank))
        Bs = [rs.uniform(size=(M.shape[0], rank)) for M in X_obs]
    else:
        A, Bs, C = np.array(init[0]), [np.array(b) for b in init[1]], np.array(init[2])

    l2 = [v if v is not None else 0 for v in O._listify(l2_penalty, "l2_penalty")]
    parsed = O.build_penalties(non_negative, lower_bound, upper_bound, l2_norm_bound, unimodal, parafac2, l1_penalty,
                               aux_init, dual_init, generalized_l2_penalty, tv_penalty)
    extra = regs if regs is not None else [[], [], []]
    regs = [parsed[m] + list(extra[m]) for m in range(3)]
    if not update_A:
        regs[0] = []
    if not update_B_is:
        regs[1] = []
    if not update_C:
        regs[2] = []

    aux = [[r.init_aux(X_obs, rank, m, rs) for r in regs[m]] for m in range(3)]
    dual = [[r.init_dual(X_obs, rank, m, rs) for r in regs[m]] for m in range(3)]
    norm_X = O._rss(X_obs)  # ‖M∘X‖
    F = masked_fill(X_obs, obs, A, Bs, C)  # F⁽⁰⁾
    rec_errors = [observed_error(X_obs, obs, A, Bs, C) / norm_X]
    losses = [0.5 * rec_errors[0] ** 2 + O._l2_term(A, Bs, C, l2) + O._penalty_sum(regs, A, Bs, C)]
    gaps = [O.feasibility_gaps(A, Bs, C, regs, *aux)]

    satisfied, message = False, "MAXIMUM NUMBER OF ITERATIONS REACHED"
    cfp = constant_feasibility_penalty
    const_A = (cfp and not isinstance(cfp, str)) or cfp == "A"
    const_B = (cfp and not isinstance(cfp, str)) or cfp == "B"
    feasible = None
    it = -1
    for it in range(n_iter_max):
        if update_B_is:
            Bs, aux[1], dual[1] = O.solve_mode_B(F, regs[1], A, Bs, C, aux[1], dual[1], l2[1], inner_n_iter_max,
                                                 feasibility_penalty_scale, const_B, inner_tol)
        if update_C:
            C, aux[2], dual[2] = O.solve_mode_C(F, regs[2], A, Bs, C, aux[2], dual[2], l2[2], inner_n_iter_max,
                                                feasibility_penalty_scale, inner_tol)
        if update_A:
            A, aux[0], dual[0], _ = O.solve_mode_A(F, regs[0], A, Bs, C, aux[0], dual[0], l2[0], inner_n_iter_max,
                                                   feasibility_penalty_scale, const_A, inner_tol)
        F = masked_fill(X_obs, obs, A, Bs, C)  # F⁽ᵗ⁾: the refill runs whether or not diagnostics are evaluated
        if trajectory is not None:
            trajectory.append(O.snapshot(A, Bs, C, aux, dual))
        if not (tol or absolute_tol or return_errors):
            continue
        cur = O.feasibility_gaps(A, Bs, C, regs, *aux)
        gaps.append(cur)
        if tol or absolute_tol:
            feasible = feasibility_tol and O._feasible(cur, feasibility_tol)
            if not feasible and not return_errors:
                continue
        err = observed_error(X_obs, obs, A, Bs, C) / norm_X
        rec_errors.append(err)
        losses.append(0.5 * err ** 2 + O._l2_term(A, Bs, C, l2) + O._penalty_sum(regs, A, Bs, C))
        if tol:
            rel_ok = abs(losses[-2] - losses[-1]) < (tol * losses[-2])
            abs_ok = losses[-1] < absolute_tol
            if feasible and rel_ok:
                satisfied, message = True, "FEASIBILITY GAP CRITERION AND RELATIVE LOSS CRITERION SATISFIED"
                break
            elif feasible and abs_ok:
                satisfied, message = True, "FEASIBILITY GAP CRITERION AND ABSOLUTE LOSS CRITERION SATISFIED"
                break
    if feasibility_tol and return_errors:
        feasible = O._feasible(O.feasibility_gaps(A, Bs, C, regs, *aux), feasibility_tol)
    elif not feasibility_tol:
        feasible = None
    if not satisfied and not (tol or absolute_tol):
        satisfied = None
    return dict(A=A, B_is=Bs, C=C, aux=aux, dual=dual, regs=regs, rec_errors=rec_errors, regularized_loss=losses,
                feasibility_gaps=gaps, n_iter=it + 1, message=message, satisfied_stopping_condition=satisfied,
                satisfied_feasibility_condition=feasible)
