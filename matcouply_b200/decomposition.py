"""AO-ADMM for coupled matrix factorization / PARAFAC2 with the call surface of ``matcouply.decomposition``
(reference src/matcouply/decomposition.py): :func:`cmf_aoadmm` (:662), :func:`parafac2_aoadmm` (:1103),
:func:`compute_feasibility_gaps` (:351), :class:`ADMMVars` (:643), :class:`DiagnosticMetrics` (:648).

The host side keeps what must stay on the host for parity — NumPy ``RandomState`` initialisation in the reference's
draw order (:31-39, :78-89), keyword -> penalty parsing (:455-614) and the stopping rule with all its quirks
(:990-1059) — and drives :class:`matcouply_b200._engine.AOADMMEngine`, which runs every numerical step as CUDA
kernels on the B200.  There is no CPU path: without the compiled library / a CUDA device the call raises.
"""
from copy import copy
from typing import NamedTuple, Optional

import os

import numpy as np

from . import _lib, penalties
from .coupled_matrices import CoupledMatrixFactorization

__all__ = ["compute_feasibility_gaps", "ADMMVars", "DiagnosticMetrics", "cmf_aoadmm", "parafac2_aoadmm"]

_MT_JUMP_DEFAULT = "1"  # sharded initial state: "1" = jump-ahead draws of the local rows only (see _device_rows_uniform)
_ALS_INITS = {"parafac2_als", "cp_als", "parafac_als", "cp_hals", "parafac_hals"}  # need TensorLy (host, one-off)


class ADMMVars(NamedTuple):
    auxes: tuple  #: Length three tuple containing a list of auxiliary factor matrices for each mode
    duals: tuple  #: Length three tuple containing a list of dual variables for each mode


class DiagnosticMetrics(NamedTuple):
    rec_errors: list  #: relative reconstruction errors, one per evaluated iteration plus the initial one
    feasibility_gaps: list  #: feasibility gaps, same length convention
    regularized_loss: list  #: regularized loss, same length convention
    satisfied_stopping_condition: Optional[bool]  #: None if no tolerance is set
    satisfied_feasibility_condition: Optional[bool]  #: None if no feasibility tolerance is set
    n_iter: int  #: Number of iterations ran
    message: str  #: Convergence message


def is_iterable(x):
    try:
        iter(x)
    except TypeError:
        return False
    return True


def _listify(input_value, param_name):  # decomposition.py:455-467
    if hasattr(input_value, "get"):
        return [input_value.get(i, None) for i in range(3)]
    if not is_iterable(input_value):
        return [input_value] * 3
    out = list(input_value)
    if len(out) != 3:
        raise ValueError(
            "All parameters must be a dictionary, non-iterable value or non-dictionary iterable of length 3."
            f" {param_name} is iterable of length {len(out)}."
        )
    return out


def _parse_mode_penalties(non_negative, lower_bound, upper_bound, l2_norm_bound, unimodal, parafac2, l1_penalty,
                          tv_penalty, generalized_l2_penalty, svd, dual_init, aux_init):
    """Fixed per-mode order Parafac2, Unimodality, GeneralizedL2, L2Ball, TV, L1, Box, NonNegativity; non_negative is
    folded into the penalties that support it (decomposition.py:549-614)."""
    init = dict(aux_init=aux_init, dual_init=dual_init)
    l1_penalty = l1_penalty if l1_penalty else 0
    regs, nn_handled = [], False
    if parafac2:
        regs.append(penalties.Parafac2(svd=svd, **init))
    if unimodal:
        regs.append(penalties.Unimodality(non_negativity=non_negative, **init))
        nn_handled = True
    if generalized_l2_penalty is not None and generalized_l2_penalty is not False:
        regs.append(penalties.GeneralizedL2Penalty(generalized_l2_penalty, svd=svd, **init))
    if l2_norm_bound:
        regs.append(penalties.L2Ball(l2_norm_bound, non_negativity=non_negative, **init))
        nn_handled = True
    if tv_penalty:
        regs.append(penalties.TotalVariationPenalty(tv_penalty, l1_strength=l1_penalty, **init))
        l1_penalty = 0
    if l1_penalty:
        regs.append(penalties.L1Penalty(l1_penalty, non_negativity=non_negative, **init))
        nn_handled = True
    if lower_bound is not None or upper_bound is not None:
        if lower_bound is None:
            lower_bound = -float("inf")
        if non_negative:
            lower_bound = max(lower_bound, 0)
        regs.append(penalties.Box(lower_bound, upper_bound, **init))
        nn_handled = True
    if non_negative and not nn_handled:
        regs.append(penalties.NonNegativity(**init))
    return regs


def _parse_all_penalties(non_negative, lower_bound, upper_bound, l2_norm_bound, unimodal, parafac2, l1_penalty,
                         tv_penalty, generalized_l2_penalty, svd, regs, dual_init, aux_init, verbose):
    """decomposition.py:470-546."""
    if regs is None:
        regs = [[], [], []]
    elif is_iterable(regs):
        for modereg in regs:
            if not is_iterable(modereg):
                raise TypeError(
                    "regs should contain an iterable of iterables containting "
                    "matcouply.penalties.ADMMMPenalty instances at least one of the"
                    f"elements in regs were not iterable (regs={regs})"
                )
            for reg in modereg:
                if not isinstance(reg, penalties.ADMMPenalty):
                    raise TypeError(
                        "regs should contain an iterable of iterables containting "
                        "matcouply.penalties.ADMMMPenalty instances at least one of the"
                        f"elements in regs contained something other than an ADMMPenalty (regs={regs})"
                    )
    regs = [copy(reg_list) for reg_list in regs]  # the caller's lists are never modified

    per_mode = dict(
        non_negative=_listify(non_negative, "non_negative"),
        upper_bound=_listify(upper_bound, "upper_bound"),
        lower_bound=_listify(lower_bound, "lower_bound"),
        l2_norm_bound=_listify(l2_norm_bound, "l2_norm_bound"),
        unimodal=_listify(unimodal, "unimodal"),
        parafac2=[False, bool(parafac2), False],
        l1_penalty=_listify(l1_penalty, "l1_penalty"),
        generalized_l2_penalty=_listify(generalized_l2_penalty, "generalized_l2_penalty"),
        tv_penalty=_listify(tv_penalty, "tv_penalty"),
    )
    for mode in range(3):
        parsed = _parse_mode_penalties(svd=svd, dual_init=dual_init, aux_init=aux_init,
                                       **{k: v[mode] for k, v in per_mode.items()})
        regs[mode] = parsed + list(regs[mode])

    if verbose:
        print("All regularization penalties (including regs list):")
        for mode, reg in enumerate(regs):
            print(f"* Mode {mode}:")
            if len(reg) == 0:
                print("   - (no regularization added)")
            for single_reg in reg:
                print(f"   - {single_reg}")
    return regs


class _ShapeOnly:
    """Stand-in for a data matrix when only its shape is needed (random init of device-resident inputs)."""

    def __init__(self, shape):
        self.shape = tuple(shape)


def initialize_cmf(matrices, rank, init, svd_fun=None, random_state=None, init_params=None, _device=None):
    """decomposition.py:18-75: a given factorization is used as is, "random" draws A, C, B_0..B_{I-1} (in this
    order) uniformly from one RandomState.  ``_device`` (internal, used by cmf_aoadmm): draw the B_i block on that
    CUDA device from the same stream and return ``(A, DeviceRows, C)`` instead of a CoupledMatrixFactorization.
    ``svd_fun`` / ``init_params`` are accepted for signature compatibility with the reference (the SVD starts use
    LAPACK's ``gesdd`` like TensorLy's ``truncated_svd``; ``init_params`` only concerns the ALS starts)."""
    random_state = penalties._check_random_state(random_state)
    if _device is not None and init == "random":
        n_slices, n_cols = len(matrices), matrices[0].shape[1]
        A = random_state.uniform(size=(n_slices, rank))
        C = random_state.uniform(size=(n_cols, rank))
        return A, penalties._device_rows_uniform(random_state, matrices, rank, _device), C
    if isinstance(init, (tuple, list, CoupledMatrixFactorization)):
        weights, (A, B_is, C) = init
        if weights is not None:
            return CoupledMatrixFactorization((None, (weights * A, B_is, C)))
        return CoupledMatrixFactorization(init)
    if init == "random":
        n_slices, n_cols = len(matrices), matrices[0].shape[1]
        A = random_state.uniform(size=(n_slices, rank))
        C = random_state.uniform(size=(n_cols, rank))
        B_is = [random_state.uniform(size=(m.shape[0], rank)) for m in matrices]
        return CoupledMatrixFactorization((None, [A, B_is, C]))
    if init in ("svd", "threshold_svd"):
        # decomposition.py:42-53: A = 1, B_i = leading left singular vectors of X_i, C = leading right singular vectors
        # of the stacked data; "threshold_svd" clips both at zero.  Like the random start (SURVEY.md §8 row I) this
        # one-off initialisation runs on the HOST with the reference's own LAPACK call (np.linalg.svd = dgesdd): the
        # signs of singular vectors are LAPACK-implementation-defined, so only the same call gives the same start.
        # It is not part of the iteration; the data must be host arrays (or is downloaded once).
        mats = [np.asarray(m.detach().cpu().numpy() if hasattr(m, "detach") else m, dtype=np.float64)
                for m in matrices]
        if any(m.ndim != 2 for m in mats):
            raise ValueError(f'init="{init}" needs the data matrices themselves, not only their shapes')

        def truncated(M, n):  # tensorly.tenalg.svd.truncated_svd (SURVEY.md §8c)
            U, S, Vh = np.linalg.svd(M, full_matrices=n > min(M.shape))
            return U[:, :n], S[:n], Vh[:n, :]

        A = np.ones((len(mats), rank))
        B_is = [truncated(m, rank)[0] for m in mats]
        C = np.transpose(truncated(np.concatenate(mats, 0), rank)[2])
        if init == "threshold_svd":
            B_is = [np.clip(B_i, 0, float("inf")) for B_i in B_is]
            C = np.clip(C, 0, float("inf"))
        return CoupledMatrixFactorization((None, [A, B_is, C]))
    if init in _ALS_INITS:
        # decomposition.py:55-73: the reference hands these starts to TensorLy's own ALS / HALS algorithms (third-party,
        # un-vendored; SURVEY.md §8f).  They are one-off HOST initialisations like the SVD starts, so the same call is
        # made here when TensorLy is installed; without it there is nothing to restate and the start is refused.
        try:
            import tensorly.decomposition as tl_decomposition
        except ImportError as exc:
            raise NotImplementedError(
                f'init="{init}" needs TensorLy decompositions (parafac / parafac2 / non_negative_parafac_hals, '
                'un-vendored third-party code; SURVEY.md §8f) and TensorLy is not installed; use init="random", "svd", '
                '"threshold_svd" or pass a factorization'
            ) from exc
        mats = [np.asarray(m.detach().cpu().numpy() if hasattr(m, "detach") else m) for m in matrices]
        if any(m.ndim != 2 for m in mats):
            raise ValueError(f'init="{init}" needs the data matrices themselves, not only their shapes')
        if init_params is None:
            init_params = {}
        if "n_iter_max" not in init_params:
            init_params["n_iter_max"] = 50
        if init == "parafac2_als":
            pf2 = tl_decomposition.parafac2(mats, rank, **init_params, random_state=random_state)
            return CoupledMatrixFactorization.from_Parafac2Tensor(pf2)
        # PARAFAC starts work on the zero-padded tensor (_utils.py:49-54)
        shapes = [tuple(m.shape) for m in mats]
        tensor = np.zeros((len(mats), max(j for j, _ in shapes), shapes[0][1]), dtype=mats[0].dtype)
        for i, m in enumerate(mats):
            tensor[i, :m.shape[0]] = m
        if init in ("cp_als", "parafac_als"):
            cp = tl_decomposition.parafac(tensor, rank, **init_params, random_state=random_state)
        else:
            cp = tl_decomposition.non_negative_parafac_hals(tensor, rank, **init_params, random_state=random_state)
        return CoupledMatrixFactorization.from_CPTensor(cp, shapes=shapes)
    raise ValueError('Initialization method "{}" not recognized'.format(init))


_SVD_NAMES = ("truncated_svd", "symeig_svd", "randomized_svd", "numpy_svd")  # tensorly.SVD_FUNS, NumPy backend


def _check_svd_name(svd):
    """_utils.py:15-26 (get_svd): an unknown ``svd`` name is refused up front.  The name does not select a code path
    here — every use of the SVD in the reference is basis-invariant (inverse of an SPD matrix, polar factor) and runs
    as Cholesky / Jacobi kernels (DESIGN.md §3)."""
    if svd not in _SVD_NAMES:
        raise ValueError(f"Got svd={svd}. However, for the current backend (numpy), the possible choices are "
                         f"{list(_SVD_NAMES[:3])}")


def initialize_aux(matrices, rank, reg, random_state):
    """decomposition.py:78-82: the auxiliary variables of every penalty, mode by mode, from ONE RandomState."""
    A_aux_list = [A_reg.init_aux(matrices, rank, 0, random_state=random_state) for A_reg in reg[0]]
    B_aux_list = [B_reg.init_aux(matrices, rank, 1, random_state=random_state) for B_reg in reg[1]]
    C_aux_list = [C_reg.init_aux(matrices, rank, 2, random_state=random_state) for C_reg in reg[2]]
    return A_aux_list, B_aux_list, C_aux_list


def initialize_dual(matrices, rank, reg, random_state):
    """decomposition.py:85-89: the scaled dual variables, same order."""
    A_dual_list = [A_reg.init_dual(matrices, rank, 0, random_state=random_state) for A_reg in reg[0]]
    B_dual_list = [B_reg.init_dual(matrices, rank, 1, random_state=random_state) for B_reg in reg[1]]
    C_dual_list = [C_reg.init_dual(matrices, rank, 2, random_state=random_state) for C_reg in reg[2]]
    return A_dual_list, B_dual_list, C_dual_list


def _check_feasibility(feasibility_gaps, feasibility_tol):  # decomposition.py:630-640
    worst = -float("inf")
    for mode_gaps in feasibility_gaps:
        if len(mode_gaps):
            worst = max(max(mode_gaps), worst)
    return worst < feasibility_tol


def compute_feasibility_gaps(cmf, regs, A_aux_list, B_aux_list, C_aux_list):
    """Relative distance between every factor and each of its auxiliary variables (decomposition.py:351-417),
    evaluated with the fused CUDA reduction ``b2_reduce_stats``."""
    import torch

    from . import _ops

    weights, (A, B_is, C) = cmf

    def dev(x):
        return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64).cuda()

    ws = _ops.Workspace("cuda", 1, 1, torch.float64)
    out = torch.zeros(3, dtype=torch.float64, device="cuda")

    def gap(x, z):
        xd = dev(x)
        _ops.reduce_stats(xd, dev(z), xd.numel(), out, ws)
        d2, x2, _ = out.cpu().numpy()
        return np.sqrt(d2) / np.sqrt(x2)

    B_flat = np.concatenate([np.asarray(b) for b in B_is], 0)
    A_gaps = [gap(A, reg.aux_as_matrix(aux)) for reg, aux in zip(regs[0], A_aux_list)]
    B_gaps = [gap(B_flat, np.concatenate([np.asarray(z) for z in reg.auxes_as_matrices(aux)], 0))
              for reg, aux in zip(regs[1], B_aux_list)]
    C_gaps = [gap(C, reg.aux_as_matrix(aux)) for reg, aux in zip(regs[2], C_aux_list)]
    return A_gaps, B_gaps, C_gaps


def _loss(diag, norm_X_sq, l2_penalty, regs, host_factors=None):
    """0.5*rel_err^2 + 0.5*sum_m lambda_m ||factor_m||^2 + sum penalties (decomposition.py:1013-1023).  With a mask,
    ``norm_X_sq`` is ||M o X||^2 and the error is the one over the observed entries: ||F - X_hat||^2 of the filled data
    F the iteration ran on, less its missing-entry part."""
    inner, quad = diag["fit"]
    if "masked" in diag:
        norm_F_sq, missing_sq = diag["masked"]
        rec_error = np.sqrt(max(0, norm_F_sq - 2 * inner + quad - missing_sq)) / np.sqrt(norm_X_sq)
    else:
        rec_error = np.sqrt(max(0, norm_X_sq - 2 * inner + quad)) / np.sqrt(norm_X_sq)
    l2reg = 0
    for m in range(3):
        if l2_penalty[m]:
            l2reg += 0.5 * l2_penalty[m] * diag["sq"][m]
    reg_penalty = 0
    for m in range(3):
        for p, reg in enumerate(regs[m]):
            if isinstance(reg, penalties.L1Penalty):
                reg_penalty += diag["l1"][m][p] * reg.reg_strength
            elif p in diag.get("extra", ({}, {}, {}))[m]:  # GeneralizedL2 / TV values reduced on the device
                reg_penalty += diag["extra"][m][p]
            elif host_factors is not None and reg._descriptor()[0] == _lib.PEN_HOST:
                reg_penalty += reg.penalty(host_factors[m])  # user-defined penalty: the user's own Python code
    return rec_error, 0.5 * rec_error ** 2 + l2reg + reg_penalty


# ----------------------------------------------------------------------------------------------------------
# the three sub-solvers as stand-alone calls (reference decomposition.py:120-344; the reference's own tests drive
# them directly, tests/test_decomposition.py:1018-1443)
# ----------------------------------------------------------------------------------------------------------
def _single_mode_update(mode, matrices, reg, cmf, aux_list, dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                        feasibility_penalty_scale, constant_feasibility_penalty):
    import torch

    from ._engine import AOADMMEngine, PackedMatrices

    if not torch.cuda.is_available():
        raise RuntimeError("matcouply_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    weights, (A, B_is, C) = cmf
    if weights is not None:
        A = A * weights
    device = torch.device("cuda", torch.cuda.current_device())
    matrices = list(matrices)
    all_f32 = all(str(getattr(m, "dtype", "")).endswith("float32") for m in matrices)
    packed = PackedMatrices.from_list(matrices, torch.float32 if all_f32 else torch.float64, device)
    regs, l2 = [[], [], []], [0, 0, 0]
    regs[mode] = list(reg)
    l2[mode] = l2_penalty if l2_penalty else 0
    engine = AOADMMEngine(packed, int(np.asarray(C).shape[1]), regs, l2_penalty=l2,
                          feasibility_penalty_scale=feasibility_penalty_scale,
                          constant_A=bool(constant_feasibility_penalty) and mode == 0,
                          constant_B=bool(constant_feasibility_penalty) and mode == 1,
                          inner_n_iter_max=inner_n_iter_max, update=(mode == 0, mode == 1, mode == 2),
                          inner_tol=inner_tol)
    auxes, duals = [[], [], []], [[], [], []]
    auxes[mode], duals[mode] = list(aux_list), list(dual_list)
    engine.load_state(np.asarray(A), [np.asarray(b) for b in B_is], np.asarray(C), auxes, duals)
    engine.prepare()  # Y = X C, B_i^T B_i, cross products and right-hand sides for the given factors
    (engine.step_A, engine.step_B, engine.step_C)[mode]()
    A1, B1, C1 = engine.factors()
    aux_out, dual_out = engine.admm_vars()
    extra = None
    if mode == 0:
        f64 = lambda t: t.detach().to(torch.float64).cpu().numpy()  # noqa: E731
        extra = (list(f64(engine.rhsA)), list(f64(engine.cross)))
    return (None, [A1, B1, C1]), aux_out[mode], dual_out[mode], extra


def admm_update_A(matrices, reg, cmf, A_aux_list, A_dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                  feasibility_penalty_scale, constant_feasibility_penalty, svd_fun=None):
    """One A-mode ADMM update (decomposition.py:120-219) on the CUDA path; also returns ``(rhses, cross_products)``
    (:219) that the fit term reuses.  ``svd_fun`` is accepted for signature compatibility (the normal matrices are
    factorised with Cholesky on the device)."""
    return _single_mode_update(0, matrices, reg, cmf, A_aux_list, A_dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                               feasibility_penalty_scale, constant_feasibility_penalty)


def admm_update_B(matrices, reg, cmf, B_is_aux_list, B_is_dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                  feasibility_penalty_scale, constant_feasibility_penalty, svd_fun=None):
    """One B-mode ADMM update (decomposition.py:222-292) on the CUDA path."""
    return _single_mode_update(1, matrices, reg, cmf, B_is_aux_list, B_is_dual_list, l2_penalty, inner_n_iter_max,
                               inner_tol, feasibility_penalty_scale, constant_feasibility_penalty)[:3]


def admm_update_C(matrices, reg, cmf, C_aux_list, C_dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                  feasibility_penalty_scale, svd_fun=None):
    """One C-mode ADMM update (decomposition.py:295-344) on the CUDA path."""
    return _single_mode_update(2, matrices, reg, cmf, C_aux_list, C_dual_list, l2_penalty, inner_n_iter_max, inner_tol,
                               feasibility_penalty_scale, False)[:3]


def _cmf_reconstruction_error(matrices, cmf, norm_matrices=None, intermediate_A_calculations=None):
    """||X - X_hat||_F (decomposition.py:420-452), from the expanded form evaluated on the device: one pass over X
    (Y = X C) plus per-slice R x R products."""
    import torch

    from ._engine import AOADMMEngine, PackedMatrices

    weights, (A, B_is, C) = cmf
    if weights is not None:
        A = A * weights
    device = torch.device("cuda", torch.cuda.current_device())
    packed = PackedMatrices.from_list(list(matrices), torch.float64, device)
    engine = AOADMMEngine(packed, int(np.asarray(C).shape[1]), [[], [], []])
    engine.load_state(np.asarray(A), [np.asarray(b) for b in B_is], np.asarray(C), [[], [], []], [[], [], []])
    engine.prepare()
    inner, quad = engine.diagnostics()["fit"]
    norm_X_sq = engine.normX_sq if norm_matrices is None else norm_matrices ** 2
    return float(np.sqrt(max(0, norm_X_sq - 2 * inner + quad)))


def cmf_aoadmm(
    matrices,
    rank,
    init="random",
    n_iter_max=1000,
    l2_penalty=None,
    tv_penalty=None,
    l1_penalty=None,
    non_negative=None,
    unimodal=None,
    generalized_l2_penalty=None,
    l2_norm_bound=None,
    lower_bound=None,
    upper_bound=None,
    parafac2=None,
    regs=None,
    feasibility_penalty_scale=1,
    constant_feasibility_penalty=False,
    aux_init="random_uniform",
    dual_init="random_uniform",
    svd="truncated_svd",
    init_params=None,
    random_state=None,
    tol=1e-8,
    absolute_tol=1e-10,
    feasibility_tol=1e-4,
    inner_tol=None,
    inner_n_iter_max=5,
    update_A=True,
    update_B_is=True,
    update_C=True,
    return_admm_vars=False,
    return_errors=False,
    verbose=False,
    device=None,
    process_group=None,
    shard=None,
    gather_factors=True,
    use_cuda_graph=None,
    mask=None,
):
    """Fit a regularized coupled matrix factorization with AO-ADMM on a B200 (same signature and semantics as the
    reference ``matcouply.decomposition.cmf_aoadmm``, decomposition.py:662-1100).

    ``matrices`` is a list of ``J_i x K`` arrays (NumPy, or torch tensors), a 3-D array iterated along axis 0, or a
    device-resident :class:`matcouply_b200.PackedMatrices`.  float32 inputs run the fp32 kernels, everything else fp64.
    Extra keywords: ``device`` (CUDA device, default current); ``process_group`` + ``shard``
    (:class:`matcouply_b200.distributed.ShardSpec`): ``matrices`` then holds only this rank's slices ``[lo, hi)`` of
    the global problem, the initial state is drawn for the GLOBAL problem from ``random_state`` (so the run equals the
    unsharded one) and cut to the shard, and a few small all-reduces per outer iteration couple the ranks;
    ``gather_factors`` returns the complete ``A`` / ``B_is`` on every rank instead of the local share.
    ``use_cuda_graph``: replay the steady-state outer iteration as one CUDA graph.  ``None`` (default) = the engine's
    policy: on for single-GPU problems without PARAFAC2 whose penalties are single kernels on the main stream and
    ``n_iter_max >= 16`` (config 1: 2.01 -> 1.91 ms per iteration; with PARAFAC2 the replay does not pay — README
    configuration 0.76 ms eager and replayed alike, config 3 slower); ``True`` = wherever the engine allows it
    (single GPU, data <= 1 GB or no PARAFAC2); ``False`` = never.  Same kernels on the same buffers: bit-identical.

    ``mask``: fit data with missing entries (1 / True = observed, 0 / False = missing), as a list of per-slice arrays
    shaped like ``matrices`` (NumPy or torch, bool or 0/1) or, for :class:`matcouply_b200.PackedMatrices` input, also
    one ``(N, K)`` bool CUDA tensor on the data's device; with ``shard`` it holds this rank's slices, as ``matrices``
    does.  The fit is EM-style with one refill per outer iteration.  The iteration runs on filled data
    ``F = M o X + (1 - M) o X_hat``, built first from the initial factors (``X`` is never read at missing positions:
    NaN or inf there is fine).  Every outer iteration runs the unchanged B-, C- and A-updates on ``F`` and then refills
    the missing entries from the new factors.  ``rec_errors`` is the relative error over the observed entries,
    ``||M o (X - X_hat)|| / ||M o X||``; the loss, the feasibility gaps and the stopping rule are as without a mask.
    Without penalties and ridge terms the observed error does not increase from one iteration to the next.  A mask
    without a missing entry gives exactly the unmasked run.  The SVD and ALS starts need complete data and are refused
    with a mask.  Data passed as ``PackedMatrices`` is filled in place during the fit and restored bit for bit on exit.
    """
    import torch

    from ._engine import PackedMatrices

    _check_svd_name(svd)
    if mask is not None:
        if isinstance(init, str) and (init in ("svd", "threshold_svd") or init in _ALS_INITS):
            raise ValueError(f'init="{init}" needs complete data and cannot be combined with a mask; use init="random" '
                             "or pass a factorization")
        if not isinstance(matrices, PackedMatrices):
            from ._engine import pack_mask

            matrices = list(matrices)
            mask = pack_mask(mask, [m.shape for m in matrices], require_observed=shard is None)
    if not torch.cuda.is_available():
        raise RuntimeError("matcouply_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    if device is not None:
        device = torch.device(device)
        if device.type != "cuda":
            raise ValueError(f"matcouply_b200 runs on CUDA devices only, got device={device}")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
    if isinstance(matrices, PackedMatrices):
        if device is not None and device != matrices.X.device:
            raise ValueError(f"`matrices` is resident on {matrices.X.device}, but device={device} was requested")
        device = matrices.X.device
    elif device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    # every kernel launch, workspace allocation and stream / event of the fit binds to `device`, whatever the caller's
    # current device is (the C ABI launches on torch's current stream, which belongs to the current device)
    with torch.cuda.device(device):
        saved = None
        if mask is not None and isinstance(matrices, PackedMatrices):
            # the caller's buffer is filled in place: keep its values at the missing positions and put them back on exit
            from ._engine import MaskCSR, pack_mask, pack_mask_device

            if isinstance(mask, torch.Tensor):
                mask = pack_mask_device(mask, matrices, require_observed=shard is None)
            elif not isinstance(mask, MaskCSR):
                mask = pack_mask(mask, matrices.shapes, require_observed=shard is None)
            mask = mask.to(device)
            flat = mask.flat_index(matrices.X.shape[1])
            saved = matrices.X.view(-1)[flat]
        try:
            return _cmf_aoadmm_on_device(
                matrices=matrices, rank=rank, init=init, n_iter_max=n_iter_max, l2_penalty=l2_penalty,
                tv_penalty=tv_penalty, l1_penalty=l1_penalty, non_negative=non_negative, unimodal=unimodal,
                generalized_l2_penalty=generalized_l2_penalty, l2_norm_bound=l2_norm_bound,
                lower_bound=lower_bound, upper_bound=upper_bound, parafac2=parafac2, regs=regs,
                feasibility_penalty_scale=feasibility_penalty_scale,
                constant_feasibility_penalty=constant_feasibility_penalty, aux_init=aux_init,
                dual_init=dual_init, svd=svd, init_params=init_params, random_state=random_state, tol=tol,
                absolute_tol=absolute_tol, feasibility_tol=feasibility_tol, inner_tol=inner_tol,
                inner_n_iter_max=inner_n_iter_max, update_A=update_A, update_B_is=update_B_is,
                update_C=update_C, return_admm_vars=return_admm_vars, return_errors=return_errors,
                verbose=verbose, process_group=process_group, shard=shard, gather_factors=gather_factors,
                use_cuda_graph=use_cuda_graph, device=device, mask=mask,
            )
        finally:
            if saved is not None:
                matrices.X.view(-1)[flat] = saved


def _cmf_aoadmm_on_device(
    matrices,
    rank,
    init="random",
    n_iter_max=1000,
    l2_penalty=None,
    tv_penalty=None,
    l1_penalty=None,
    non_negative=None,
    unimodal=None,
    generalized_l2_penalty=None,
    l2_norm_bound=None,
    lower_bound=None,
    upper_bound=None,
    parafac2=None,
    regs=None,
    feasibility_penalty_scale=1,
    constant_feasibility_penalty=False,
    aux_init="random_uniform",
    dual_init="random_uniform",
    svd="truncated_svd",
    init_params=None,
    random_state=None,
    tol=1e-8,
    absolute_tol=1e-10,
    feasibility_tol=1e-4,
    inner_tol=None,
    inner_n_iter_max=5,
    update_A=True,
    update_B_is=True,
    update_C=True,
    return_admm_vars=False,
    return_errors=False,
    verbose=False,
    device=None,
    process_group=None,
    shard=None,
    gather_factors=True,
    use_cuda_graph=None,
    mask=None,
):
    """Body of :func:`cmf_aoadmm`; runs with ``device`` as the current CUDA device.  ``mask``: None or a MaskCSR."""
    import torch

    from ._engine import AOADMMEngine, PackedMatrices

    random_state = penalties._check_random_state(random_state)
    if isinstance(matrices, PackedMatrices):
        packed = matrices
        shape_view = [_ShapeOnly(s) for s in packed.shapes]
    else:
        matrices = list(matrices)
        if not matrices and shard is not None and shard.lo == shard.hi:
            # a rank of a sharded run with no slice at all (more ranks than slices): it still takes part in every
            # all-reduce and computes the replicated C-mode state, on a 0 x K shard
            if not shard.n_cols:
                raise ValueError("an empty shard needs ShardSpec.n_cols (make_shard(..., n_cols=K))")
            packed = PackedMatrices.empty(shard.n_cols, torch.float32 if shard.dtype == "float32" else torch.float64,
                                          device)
        else:
            all_f32 = all(str(getattr(m, "dtype", "")).endswith("float32") for m in matrices)
            packed = PackedMatrices.from_list(matrices, torch.float32 if all_f32 else torch.float64, device)
        shape_view = matrices
    if shard is not None:
        if process_group is None:
            raise ValueError("`shard` needs a `process_group`")
        if packed.n_slices != shard.hi - shard.lo or any(
                int(s[0]) != int(j) for s, j in zip(packed.shapes, shard.row_counts[shard.lo:shard.hi])):
            raise ValueError("`matrices` must hold exactly the slices [shard.lo, shard.hi) of the global problem")
        shape_view = [_ShapeOnly((j, packed.K)) for j in shard.row_counts]  # the GLOBAL problem
    if mask is not None:
        counts = torch.tensor([mask.n_missing, mask.n_observed], dtype=torch.float64, device=device)
        if process_group is not None:
            torch.distributed.all_reduce(counts, group=process_group)
        n_missing, n_observed = (int(v) for v in counts.tolist())
        if n_observed == 0:
            raise ValueError("the mask has no observed entry")
        mask = mask.to(device) if n_missing else None  # no hole anywhere: exactly the unmasked run
    # default path: the big B-mode blocks (B_i, aux, dual) are drawn on the device from random_state's own MT19937
    # stream (bit-identical to host draws, see csrc/rng.cu); B2_HOST_RNG=1 forces the host draws
    dev_draw = None if os.environ.get("B2_HOST_RNG") else device
    # sharded run: draw only this rank's rows of every device-drawn variable and jump over the others in the stream
    # (B2_MT_JUMP=0 walks the whole global stream on every rank instead; same bits either way)
    draw_window = None
    if shard is not None and dev_draw is not None and os.environ.get("B2_MT_JUMP", _MT_JUMP_DEFAULT) != "0":
        draw_window = (shard.lo, shard.hi)
    if init == "random" and dev_draw is not None:
        penalties._DEVICE_DRAW["window"] = draw_window
        try:
            A0, B0, C0 = initialize_cmf(shape_view, rank, init, random_state=random_state, _device=dev_draw)
        finally:
            penalties._DEVICE_DRAW["window"] = None
    else:
        init_view = shape_view
        needs_data = isinstance(init, str) and (init in ("svd", "threshold_svd") or init in _ALS_INITS)
        if needs_data and not all(hasattr(m, "ndim") for m in shape_view):
            if shard is not None:
                raise NotImplementedError(
                    f'init="{init}" needs the stacked global data; not available for sharded inputs')
            host = packed.X[:packed.N, :packed.K].detach().to(torch.float64).cpu().numpy()  # device-resident input
            init_view = [host[a:b] for a, b in zip(packed.row_offsets[:-1], packed.row_offsets[1:])]
        w0, (A0, B0, C0) = initialize_cmf(init_view, rank, init, random_state=random_state,
                                         init_params=init_params)
        if w0 is not None:  # TensorLy starts carry weights; absorbed like a given factorization (:22-25)
            A0 = np.asarray(w0) * np.asarray(A0)

    l2_penalty = [l2 if l2 is not None else 0 for l2 in _listify(l2_penalty, "l2_penalty")]
    regs = _parse_all_penalties(
        non_negative=non_negative, lower_bound=lower_bound, upper_bound=upper_bound, l2_norm_bound=l2_norm_bound,
        unimodal=unimodal, parafac2=parafac2, l1_penalty=l1_penalty, tv_penalty=tv_penalty,
        generalized_l2_penalty=generalized_l2_penalty, svd=svd, regs=regs, dual_init=dual_init, aux_init=aux_init,
        verbose=verbose,
    )
    if not update_A:
        regs[0] = []
    if not update_B_is:
        regs[1] = []
    if not update_C:
        regs[2] = []

    # aux first, then dual, each in mode order from the same RandomState (decomposition.py:78-89)
    penalties._DEVICE_DRAW["device"] = dev_draw
    penalties._DEVICE_DRAW["window"] = draw_window
    try:
        auxes = [[reg.init_aux(shape_view, rank, m, random_state=random_state) for reg in regs[m]] for m in range(3)]
        duals = [[reg.init_dual(shape_view, rank, m, random_state=random_state) for reg in regs[m]] for m in range(3)]
    finally:
        penalties._DEVICE_DRAW["device"] = None
        penalties._DEVICE_DRAW["window"] = None

    if isinstance(constant_feasibility_penalty, str) and constant_feasibility_penalty not in {"A", "B"}:
        raise ValueError(
            f"If `constant_feasibility_penalty` is a string, it must be 'A' or 'B', not {constant_feasibility_penalty}"
        )
    both = constant_feasibility_penalty and not isinstance(constant_feasibility_penalty, str)
    constant_A = bool(both or constant_feasibility_penalty == "A")
    constant_B = bool(both or constant_feasibility_penalty == "B")

    engine = AOADMMEngine(packed, rank, regs, l2_penalty=l2_penalty,
                          feasibility_penalty_scale=feasibility_penalty_scale, constant_A=constant_A,
                          constant_B=constant_B, inner_n_iter_max=inner_n_iter_max,
                          update=(update_A, update_B_is, update_C), group=process_group,
                          shard_rows=None if shard is None else (shard.lo, shard.n_global), inner_tol=inner_tol,
                          mask=mask)
    if shard is not None:
        from .distributed import shard_state

        A0, B0, auxes, duals = shard_state(A0, B0, auxes, duals, regs, shard)
    engine.load_state(np.asarray(A0), B0, np.asarray(C0), auxes, duals)
    engine.prepare()
    norm_X_sq = engine.normX_sq

    # user-defined (Python) penalties: their value needs the factors on the host every evaluated iteration
    has_host_pen = any(reg._descriptor()[0] == _lib.PEN_HOST for mode_regs in regs for reg in mode_regs)
    host_factors = (lambda: engine.factors()) if has_host_pen else (lambda: None)

    diag = engine.diagnostics()
    rec_error, loss = _loss(diag, norm_X_sq, l2_penalty, regs, host_factors())
    rec_errors, losses, feasibility_gaps = [rec_error], [loss], [diag["gaps"]]
    if verbose and verbose > 0:
        print("Feasibility gaps for A: {}".format(diag["gaps"][0]))
        print("Feasibility gaps for the Bi-matrices: {}".format(diag["gaps"][1]))
        print("Feasibility gaps for C: {}".format(diag["gaps"][2]))

    satisfied_stopping_condition = False
    feasibility_criterion = None
    message = "MAXIMUM NUMBER OF ITERATIONS REACHED"
    it = -1
    want_diag = bool(tol or absolute_tol or return_errors)
    # use_cuda_graph: True = where the engine allows it, False = never, None = the engine's own policy (graph_auto:
    # single-GPU CMF-type problems, and only when the capture can pay for itself)
    if use_cuda_graph is None:
        use_graph = n_iter_max >= 16 and engine.graph_auto()
    else:
        use_graph = bool(use_cuda_graph) and engine.graph_eligible()
    if use_graph and hasattr(engine, "polar_cold_every"):
        engine.polar_cold_every = 1  # a replayed iteration starts its polar steps cold: the eager iterations do the same
    for it in range(n_iter_max):
        launched = None
        if use_graph and it >= 2:  # steady state: replay the captured launch sequence (see AOADMMEngine.graph_iteration)
            try:
                launched = engine.graph_iteration(want_diag)
            except Exception:
                if use_cuda_graph:  # asked for explicitly: report
                    raise
                engine._graph_failed, use_graph = True, False  # own policy: fall back to issuing the launches one by one
                engine.outer_iteration()
        else:
            engine.outer_iteration()

        if want_diag:
            diag = engine._read_diagnostics(launched) if launched is not None else engine.diagnostics()
            curr_gaps = diag["gaps"]
            feasibility_gaps.append(curr_gaps)
            if tol or absolute_tol:
                feasibility_criterion = feasibility_tol and _check_feasibility(curr_gaps, feasibility_tol)
                if not feasibility_criterion and not return_errors:
                    # the loss is NOT appended on infeasible iterations (decomposition.py:996-1011)
                    if verbose and it % verbose == 0 and verbose > 0:
                        print(
                            "Coupled matrix factorization iteration={}, ".format(it)
                            + "reconstruction error=NOT COMPUTED, "
                            + "regularized loss=NOT COMPUTED, "
                            + "regularized loss variation=NOT COMPUTED."
                        )
                        print("Feasibility gaps for A: {}".format(curr_gaps[0]))
                        print("Feasibility gaps for the Bi-matrices: {}".format(curr_gaps[1]))
                        print("Feasibility gaps for C: {}".format(curr_gaps[2]))
                    continue

            rec_error, loss = _loss(diag, norm_X_sq, l2_penalty, regs, host_factors())
            rec_errors.append(rec_error)
            losses.append(loss)
            if verbose and it % verbose == 0 and verbose > 0:
                print(
                    "Coupled matrix factorization iteration={}, ".format(it)
                    + "reconstruction error={}, ".format(rec_errors[-1])
                    + "regularized loss={} ".format(losses[-1])
                    + "regularized loss variation={}.".format(abs(losses[-2] - losses[-1]) / losses[-2])
                )
                print("Feasibility gaps for A: {}".format(curr_gaps[0]))
                print("Feasibility gaps for the Bi-matrices: {}".format(curr_gaps[1]))
                print("Feasibility gaps for C: {}".format(curr_gaps[2]))

            if tol:
                rel_loss_criterion = abs(losses[-2] - losses[-1]) < (tol * losses[-2])
                abs_loss_criterion = losses[-1] < absolute_tol
                if feasibility_criterion and rel_loss_criterion:
                    satisfied_stopping_condition = True
                    message = "FEASIBILITY GAP CRITERION AND RELATIVE LOSS CRITERION SATISFIED"
                    if verbose:
                        print("converged in {} iterations: {}".format(it, message))
                    break
                elif feasibility_criterion and abs_loss_criterion:
                    satisfied_stopping_condition = True
                    message = "FEASIBILITY GAP CRITERION AND ABSOLUTE LOSS CRITERION SATISFIED"
                    if verbose:
                        print("converged in {} iterations: {}".format(it, message))
                    break
        elif verbose and it % verbose == 0 and verbose > 0:
            print("Coupled matrix factorization iteration={}".format(it))
    else:
        if verbose:
            print("REACHED MAXIMUM NUMBER OF ITERATIONS")

    if feasibility_tol and return_errors:  # decomposition.py:1065-1070
        feasibility_criterion = _check_feasibility(engine.diagnostics()["gaps"], feasibility_tol)
    elif not feasibility_tol:
        feasibility_criterion = None

    A, B_is, C = engine.factors()
    if shard is not None and gather_factors:
        from .distributed import allgather_rows

        A = allgather_rows(A, shard, process_group)
        B_is = allgather_rows(B_is, shard, process_group)
    out = [CoupledMatrixFactorization((None, [A, B_is, C]))]
    if return_admm_vars:
        aux_out, dual_out = engine.admm_vars()  # rank-local share for modes 0 and 1 when sharded
        out.append(ADMMVars(auxes=tuple(aux_out), duals=tuple(dual_out)))
    if return_errors:
        if not satisfied_stopping_condition and not (tol or absolute_tol):
            satisfied_stopping_condition = None
        out.append(DiagnosticMetrics(
            rec_errors=rec_errors, feasibility_gaps=feasibility_gaps, regularized_loss=losses,
            satisfied_stopping_condition=satisfied_stopping_condition,
            satisfied_feasibility_condition=feasibility_criterion, message=message, n_iter=it + 1,
        ))
    return out[0] if len(out) == 1 else tuple(out)


def parafac2_aoadmm(
    matrices,
    rank,
    init="random",
    n_iter_max=1000,
    l2_penalty=0,
    tv_penalty=None,
    l1_penalty=None,
    non_negative=None,
    unimodal=None,
    generalized_l2_penalty=None,
    l2_norm_bound=None,
    lower_bound=None,
    upper_bound=None,
    regs=None,
    feasibility_penalty_scale=1,
    constant_feasibility_penalty=False,
    aux_init="random_uniform",
    dual_init="random_uniform",
    svd="truncated_svd",
    init_params=None,
    random_state=None,
    tol=1e-8,
    absolute_tol=1e-10,
    feasibility_tol=1e-4,
    inner_tol=None,
    inner_n_iter_max=5,
    update_A=True,
    update_B_is=True,
    update_C=True,
    return_errors=False,
    return_admm_vars=False,
    verbose=False,
    mask=None,
    **extra,
):
    """Alias of :func:`cmf_aoadmm` with the PARAFAC2 constraint on mode 1 (decomposition.py:1103-1179)."""
    return cmf_aoadmm(
        matrices=matrices, rank=rank, init=init, n_iter_max=n_iter_max, l2_penalty=l2_penalty, tv_penalty=tv_penalty,
        l1_penalty=l1_penalty, non_negative=non_negative, unimodal=unimodal,
        generalized_l2_penalty=generalized_l2_penalty, l2_norm_bound=l2_norm_bound, lower_bound=lower_bound,
        upper_bound=upper_bound, parafac2=True, regs=regs, feasibility_penalty_scale=feasibility_penalty_scale,
        constant_feasibility_penalty=constant_feasibility_penalty, aux_init=aux_init, dual_init=dual_init, svd=svd,
        init_params=init_params, random_state=random_state, tol=tol, absolute_tol=absolute_tol,
        feasibility_tol=feasibility_tol, inner_tol=inner_tol, inner_n_iter_max=inner_n_iter_max, update_A=update_A,
        update_B_is=update_B_is, update_C=update_C, return_errors=return_errors, return_admm_vars=return_admm_vars,
        verbose=verbose, mask=mask, **extra,
    )
