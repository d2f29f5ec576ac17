"""ADMM penalties with the call surface of ``matcouply.penalties`` (reference: src/matcouply/penalties.py).

Same class names, constructor arguments, attributes, ``__repr__`` and error behaviour as the reference
(``ADMMPenalty`` :21, ``MatricesPenalty`` :369, ``MatrixPenalty`` :389, ``RowVectorPenalty`` :426,
``HardConstraintMixin`` :466, ``NonNegativity`` :488, ``Box`` :511, ``L1Penalty`` :545, ``L2Ball`` :844,
``Unimodality`` :983, ``Parafac2`` :1018).  Inside :func:`matcouply_b200.decomposition.cmf_aoadmm` the objects act as
*descriptors*: the fused engine reads their parameters and runs the proximal operators as CUDA kernels.  The protocol
methods (``factor_matrix_update`` ...) are also callable on their own with NumPy arrays or torch tensors; they upload,
run the same CUDA kernels through the C ABI and return the input's array type.  There is no CPU implementation.

``GeneralizedL2Penalty`` (:595), ``TotalVariationPenalty`` (:750) and ``UnitSimplex`` (:928) run their proximal
operators as CUDA kernels too (csrc/prox_extra.cu), as does ``TemporalSmoothnessPenalty`` (no reference counterpart:
smoothness of the ``B_i`` over the slice order, csrc/prox_temporal.cu); user-defined subclasses that implement the protocol in Python are
bridged by the engine (``PEN_HOST``: the pre-image is handed to the Python method, the result goes back to HBM).
"""
from abc import ABC, abstractmethod

import numpy as np

from . import _lib

__all__ = [
    "ADMMPenalty", "MatricesPenalty", "MatrixPenalty", "RowVectorPenalty", "HardConstraintMixin", "NonNegativity",
    "Box", "L1Penalty", "L2Ball", "Unimodality", "Parafac2", "GeneralizedL2Penalty", "TotalVariationPenalty",
    "UnitSimplex", "TemporalSmoothnessPenalty",
]


def copy_ancestor_docstring(fn):
    """No-op decorator kept for source compatibility with custom penalties written for the reference
    (matcouply/_doc_utils.py:46-52)."""
    return fn


def _check_random_state(seed):
    if seed is None:
        return np.random.mtrand._rand
    if isinstance(seed, (int, np.integer)):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError("Seed should be None, int or np.random.RandomState")


# set by cmf_aoadmm around its own init_aux / init_dual calls (see _init_variable); None = draw on the host
_DEVICE_DRAW = {"device": None, "window": None}  # window: (lo, hi) slices of this rank in a sharded run, or None


def _device_rows_uniform(random_state, matrices, rank, device):
    """``[random_state.uniform(size=(J_i, rank)) for each matrix]`` as a DeviceRows (one packed CUDA tensor)."""
    from . import _ops
    from ._engine import DeviceRows

    off = np.concatenate([[0], np.cumsum([int(m.shape[0]) for m in matrices])]).astype(np.int64)
    window = _DEVICE_DRAW.get("window")
    if window is not None:
        # sharded run: skip the rows of the other ranks in the stream (MT19937 jump-ahead on the host, O(1) in the
        # number of skipped draws) and draw only this rank's rows; the generator ends where the global draw would
        from ._engine import ShardRows

        lo, hi = window
        n_local = int(off[hi] - off[lo])
        _ops.mt19937_skip(random_state, int(off[lo]) * rank)
        flat = _ops.mt19937_uniform(random_state, n_local * rank, device)
        _ops.mt19937_skip(random_state, int(off[-1] - off[hi]) * rank)
        return ShardRows(DeviceRows(flat.view(n_local, rank), off[lo:hi + 1] - off[lo]), lo, hi, len(matrices))
    flat = _ops.mt19937_uniform(random_state, int(off[-1]) * rank, device)
    return DeviceRows(flat.view(int(off[-1]), rank), off)


class _EyeBases:
    """The default PARAFAC2 basis matrices ``[np.eye(J_i, rank) for i]`` (penalties.py:1175) without materialising
    them: list-like, builds the NumPy matrices only when indexed / iterated."""

    def __init__(self, row_counts, rank):
        self.row_counts, self.rank = list(row_counts), int(rank)

    def __len__(self):
        return len(self.row_counts)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return _EyeBases(self.row_counts[i], self.rank)
        return np.eye(self.row_counts[i], self.rank)

    def __iter__(self):
        return (np.eye(j, self.rank) for j in self.row_counts)

    def cut(self, lo, hi):
        return _EyeBases(self.row_counts[lo:hi], self.rank)


def _is_tensor(x):
    if isinstance(x, np.ndarray):
        return True
    try:
        import torch

        return isinstance(x, torch.Tensor)
    except ImportError:  # pragma: no cover
        return False


# ----------------------------------------------------------------------------------------------------------
# device round trip used by the stand-alone protocol methods
# ----------------------------------------------------------------------------------------------------------
class _Dev:
    """Moves an array to the GPU (float32 stays float32, everything else becomes float64) and back."""

    def __init__(self, x):
        import torch

        self.torch = torch
        self.was_numpy = not isinstance(x, torch.Tensor)
        if self.was_numpy:
            arr = np.asarray(x)
            dt = torch.float32 if arr.dtype == np.float32 else torch.float64
            self.t = torch.as_tensor(np.ascontiguousarray(arr), dtype=dt).cuda()
        else:
            self.src_device = x.device
            dt = torch.float32 if x.dtype == torch.float32 else torch.float64
            self.t = x.detach().to(device="cuda", dtype=dt).contiguous()
            if self.t.data_ptr() == x.data_ptr():
                self.t = self.t.clone()

    def back(self, t):
        if self.was_numpy:
            return t.cpu().numpy()
        return t.to(self.src_device)


def _single_group_offsets(n, device):
    import torch

    return torch.tensor([0, n], dtype=torch.int64, device=device)


class ADMMPenalty(ABC):
    """Base class of all penalties (reference penalties.py:21-366)."""

    _kind = None  # B2_PEN_* code when the fused engine has a kernel for this penalty

    def __init__(self, aux_init="random_uniform", dual_init="random_uniform"):
        self.aux_init = aux_init
        self.dual_init = dual_init

    # -- initialisation of auxiliary / dual variables (penalties.py:36-147, 149-261) --------------------------
    def _init_variable(self, init, attr_name, matrices, rank, mode, random_state):
        random_state = _check_random_state(random_state)
        if not isinstance(rank, int):
            raise TypeError("Rank must be int, not {}".format(type(rank)))
        if not isinstance(mode, int):
            raise TypeError("Mode must be int, not {}".format(type(mode)))
        elif mode not in [0, 1, 2]:
            raise ValueError("Mode must be 0, 1, or 2.")
        if not isinstance(init, str) and not _is_tensor(init) and not isinstance(init, list):
            raise TypeError(
                "self.{} must be a tensor, a list of tensors or a string specifiying init method, not {}".format(
                    attr_name, type(init)
                )
            )
        n_slices = len(matrices)
        n_cols = matrices[0].shape[1]
        if mode in (0, 2) and _is_tensor(init):
            length_, rank_ = init.shape
            if rank != rank_ or (mode == 0 and length_ != n_slices):
                raise ValueError(
                    "Invalid shape for pre-specified auxiliary variable for mode 0"
                    "\nShould have shape {}, but has shape {}".format((n_slices, rank), (length_, rank_))
                )
            elif rank != rank_ or (mode == 2 and length_ != n_cols):
                raise ValueError(
                    "Invalid shape for pre-specified auxiliary variable for mode 2"
                    "\nShould have shape {}, but has shape {}".format((n_cols, rank), (length_, rank_))
                )
            return init
        if mode in (0, 2) and isinstance(init, list):
            raise TypeError("Cannot use list of matrices to initialize auxiliary matrices for mode 0 or 2.")
        if mode == 1 and isinstance(init, list):
            wanted = [(m.shape[0], rank) for m in matrices]
            if any(tuple(v.shape) != s for v, s in zip(init, wanted)):
                raise ValueError("Invalid shape for at least one of matrices in the auxiliary variable list for mode 1.")
            elif len(init) != n_slices:
                raise ValueError(
                    "Different number of pre-specified auxiliary factor matrices for mode 1 "
                    "than the number of coupled matrices."
                )
            return init
        if mode == 1 and _is_tensor(init):
            raise TypeError(
                "Cannot use a tensor (matrix) to initialize auxiliary matrices for mode 1. Must be a list instead."
            )

        if init == "random_uniform" and mode == 1 and _DEVICE_DRAW["device"] is not None:
            # fast path of cmf_aoadmm: the sum_i J_i x R block is drawn ON THE DEVICE from the same MT19937 stream
            # (identical bits, random_state advanced accordingly) and never touches host memory
            return _device_rows_uniform(random_state, matrices, rank, _DEVICE_DRAW["device"])
        if init == "random_uniform":
            draw = lambda shape: random_state.uniform(size=shape)  # noqa: E731
        elif init == "random_standard_normal":
            draw = lambda shape: random_state.standard_normal(size=shape)  # noqa: E731
        elif init == "zeros":
            draw = np.zeros
        else:
            raise ValueError("Unknown aux init: {}".format(init))
        if mode == 0:
            return draw((n_slices, rank))
        if mode == 2:
            return draw((n_cols, rank))
        return [draw((m.shape[0], rank)) for m in matrices]

    def init_aux(self, matrices, rank, mode, random_state=None):
        return self._init_variable(self.aux_init, "aux_init", matrices, rank, mode, random_state)

    def init_dual(self, matrices, rank, mode, random_state=None):
        return self._init_variable(self.dual_init, "dual_init", matrices, rank, mode, random_state)

    @abstractmethod
    def penalty(self, x):  # pragma: nocover
        raise NotImplementedError

    def subtract_from_auxes(self, auxes, duals):
        return [self.subtract_from_aux(aux, dual) for aux, dual in zip(auxes, duals)]

    def subtract_from_aux(self, aux, dual):
        return aux - dual

    def aux_as_matrix(self, aux):
        return aux

    def auxes_as_matrices(self, auxes):
        return [self.aux_as_matrix(aux) for aux in auxes]

    def _auto_add_param_to_repr(self, param):
        if param.startswith("_"):
            return False
        return param not in {"aux_init", "dual_init"}

    def __repr__(self):  # penalties.py:352-366 — exact text is asserted by the reference's tests
        parts = [f"{k}={repr(v)}" for k, v in self.__dict__.items() if self._auto_add_param_to_repr(k)]
        parts.append(f"aux_init='{self.aux_init}'" if isinstance(self.aux_init, str) else "aux_init=given_init")
        parts.append(f"dual_init='{self.dual_init}'" if isinstance(self.dual_init, str) else "dual_init=given_init")
        return f"<'{self.__module__}.{type(self).__name__}' with {', '.join(parts)})>"

    # descriptor handed to the fused engine: (kind, non_negativity, p0, p1).  The built-in penalties override it with
    # their CUDA kind; a user-defined subclass (which implements the protocol in Python, e.g. the reference's
    # examples/plot_custom_penalty.py:220-231) is bridged: the engine hands it the pre-image and takes the aux back.
    def _descriptor(self):
        return (_lib.PEN_HOST, False, 0.0, 0.0)


class MatricesPenalty(ADMMPenalty):
    @abstractmethod
    def factor_matrices_update(self, factor_matrices, feasibility_penalties, auxes):  # pragma: nocover
        raise NotImplementedError


class MatrixPenalty(MatricesPenalty):
    def factor_matrices_update(self, factor_matrices, feasibility_penalties, auxes):
        return [
            self.factor_matrix_update(fm, rho, aux)
            for fm, rho, aux in zip(factor_matrices, feasibility_penalties, auxes)
        ]

    @abstractmethod
    def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):  # pragma: nocover
        raise NotImplementedError


class RowVectorPenalty(MatrixPenalty):
    def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):
        return self.factor_matrix_row_update(factor_matrix, feasibility_penalty, aux)

    @abstractmethod
    def factor_matrix_row_update(self, factor_matrix_row, feasibility_penalty, aux_row):  # pragma: nocover
        raise NotImplementedError


class HardConstraintMixin:
    def penalty(self, x):
        return 0


class _ElementwiseMixin:
    """NonNegativity / Box / L1 share one CUDA kernel (csrc/admm.cu: prox_elem)."""

    def _elementwise(self, x, feasibility_penalty):
        from . import _ops

        dev = _Dev(x)
        kind, nn, p0, p1 = self._descriptor()
        out = dev.torch.empty_like(dev.t)
        _ops.prox_elementwise(dev.t, out, kind, nn, p0, p1, feasibility_penalty)
        return dev.back(out)

    def factor_matrix_row_update(self, factor_matrix_row, feasibility_penalty, aux_row):
        return self._elementwise(factor_matrix_row, feasibility_penalty)

    def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):
        return self._elementwise(factor_matrix, feasibility_penalty)


class NonNegativity(_ElementwiseMixin, HardConstraintMixin, RowVectorPenalty):
    """Projection onto the non-negative orthant (penalties.py:488-508)."""

    _kind = _lib.PEN_NONNEG

    def _descriptor(self):
        return (_lib.PEN_NONNEG, False, 0.0, 0.0)


class Box(_ElementwiseMixin, HardConstraintMixin, RowVectorPenalty):
    """Projection onto ``[min_val, max_val]`` (penalties.py:511-542)."""

    _kind = _lib.PEN_BOX

    def __init__(self, min_val, max_val, aux_init="random_uniform", dual_init="random_uniform"):
        super().__init__(aux_init=aux_init, dual_init=dual_init)
        self.min_val = min_val
        self.max_val = max_val

    def _descriptor(self):
        lo = -float("inf") if self.min_val is None else float(self.min_val)
        hi = float("inf") if self.max_val is None else float(self.max_val)
        return (_lib.PEN_BOX, False, lo, hi)


class L1Penalty(_ElementwiseMixin, RowVectorPenalty):
    """Soft thresholding (penalties.py:545-592)."""

    _kind = _lib.PEN_L1

    def __init__(self, reg_strength, non_negativity=False, aux_init="random_uniform", dual_init="random_uniform"):
        super().__init__(aux_init=aux_init, dual_init=dual_init)
        if reg_strength < 0:
            raise ValueError("Regularization strength must be nonnegative.")
        self.reg_strength = reg_strength
        self.non_negativity = non_negativity

    def _descriptor(self):
        return (_lib.PEN_L1, bool(self.non_negativity), float(self.reg_strength), 0.0)

    def penalty(self, x):  # penalties.py:589-592 — gamma * sum |x| of the primal factor
        from . import _ops

        xs = [x] if _is_tensor(x) else list(x)
        total = 0.0
        for xi in xs:
            dev = _Dev(xi)
            out = dev.torch.zeros(3, dtype=dev.torch.float64, device="cuda")
            ws = _ops.Workspace("cuda", 1, 1, dev.t.dtype)
            _ops.reduce_stats(dev.t, None, dev.t.numel(), out, ws)
            total += float(out[2].item())
        return total * self.reg_strength


class _ColumnCoupledMixin:
    """Penalties whose prox couples all rows of one matrix: run with one group = the whole matrix."""

    def _run(self, dual, out, row_off, n_rows, rank, ws):  # dual holds V on entry
        raise NotImplementedError

    def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):
        from . import _ops

        dev = _Dev(factor_matrix)
        V = dev.t if dev.t.dim() == 2 else dev.t.reshape(-1, 1)
        n_rows, rank = V.shape
        dual = V.clone()
        out = dev.torch.empty_like(V)
        ws = _ops.Workspace("cuda", 1, max(rank, 1), V.dtype)
        self._run(dual, out, _single_group_offsets(n_rows, "cuda"), n_rows, rank, ws)
        return dev.back(out.reshape(dev.t.shape))


class L2Ball(_ColumnCoupledMixin, HardConstraintMixin, MatrixPenalty):
    """Columns inside an L2 ball of radius ``norm_bound`` (penalties.py:844-925)."""

    _kind = _lib.PEN_L2BALL

    def __init__(self, norm_bound, non_negativity=False, aux_init="random_uniform", dual_init="random_uniform"):
        super().__init__(aux_init, dual_init)
        self.norm_bound = norm_bound
        self.non_negativity = non_negativity
        if norm_bound <= 0:
            raise ValueError("The norm bound must be positive.")

    def _descriptor(self):
        return (_lib.PEN_L2BALL, bool(self.non_negativity), float(self.norm_bound), 0.0)

    def _run(self, dual, out, row_off, n_rows, rank, ws):
        from . import _ops

        _ops.prox_l2ball(out, dual, row_off, 1, rank, self.norm_bound, self.non_negativity)


class Unimodality(_ColumnCoupledMixin, HardConstraintMixin, MatrixPenalty):
    """Unimodal columns, optionally non-negative (penalties.py:983-1015)."""

    _kind = _lib.PEN_UNIMODAL

    def __init__(self, non_negativity=False, aux_init="random_uniform", dual_init="random_uniform"):
        super().__init__(aux_init, dual_init)
        self.non_negativity = non_negativity

    def _descriptor(self):
        return (_lib.PEN_UNIMODAL, bool(self.non_negativity), 0.0, 0.0)

    def _run(self, dual, out, row_off, n_rows, rank, ws):
        from . import _ops

        _ops.prox_unimodal(out, dual, row_off, 1, rank, n_rows, self.non_negativity, ws)


class Parafac2(MatricesPenalty):
    """PARAFAC2 constraint ``B_i = P_i Delta`` with orthonormal ``P_i`` (penalties.py:1018-1324)."""

    _kind = _lib.PEN_PARAFAC2

    def __init__(self, svd="truncated_svd", n_iter=1, update_basis_matrices=True, update_coordinate_matrix=True,
                 aux_init="random_uniform", dual_init="random_uniform"):
        self.svd = svd
        self.aux_init = aux_init
        self.dual_init = dual_init
        self.update_basis_matrices = update_basis_matrices
        self.update_coordinate_matrix = update_coordinate_matrix
        self.n_iter = n_iter

    def _descriptor(self):
        return (_lib.PEN_PARAFAC2, False, 0.0, 0.0)

    def init_aux(self, matrices, rank, mode, random_state=None):  # penalties.py:1111-1222
        random_state = _check_random_state(random_state)
        if not isinstance(self.aux_init, (str, tuple)):
            raise TypeError(
                "Parafac2 auxiliary variables must be initialized using either a string"
                " or a tuple (containing the orthogonal basis matrices and the coordinate matrix)."
            )
        if not isinstance(rank, int):
            raise TypeError("Rank must be int, not {}".format(type(rank)))
        if not isinstance(mode, int):
            raise TypeError("Mode must be int, not {}".format(type(mode)))
        if mode != 1:
            raise ValueError("PARAFAC2 constraint can only be imposed with mode=1")

        if isinstance(self.aux_init, tuple):
            basis_matrices, coordinate_matrix = self.aux_init
            if not isinstance(basis_matrices, list) or not _is_tensor(coordinate_matrix):
                raise TypeError(
                    "If self.aux_init is a tuple, then its first element must be a list of basis matrices "
                    "and second element the coordinate matrix."
                )
            if not len(coordinate_matrix.shape) == 2:
                raise ValueError(
                    "The coordinate matrix must have two modes, not {}".format(len(coordinate_matrix.shape))
                )
            if coordinate_matrix.shape[0] != coordinate_matrix.shape[1] or coordinate_matrix.shape[0] != rank:
                raise ValueError(
                    "The coordinate matrix must be rank x rank, with rank={}, not {}".format(
                        rank, tuple(coordinate_matrix.shape)
                    )
                )
            for matrix, basis_matrix in zip(matrices, basis_matrices):
                if not _is_tensor(basis_matrix):
                    raise TypeError("Each basis matrix must be a tensorly tensor")
                if not len(basis_matrix.shape) == 2:
                    raise ValueError(
                        "Each basis matrix must be tensor with two modes, not {}".format(len(basis_matrix.shape))
                    )
                if matrix.shape[0] != basis_matrix.shape[0] or basis_matrix.shape[1] != rank:
                    raise ValueError(
                        "The i-th basis matrix must have shape J_i x rank, where J_i is the number of "
                        "rows in the i-th matrix."
                    )
                P = np.asarray(basis_matrix)
                if not np.sum((P.T @ P - np.eye(rank)) ** 2) < 1e-8:
                    raise ValueError("The basis matrices must be orthogonal")
            if len(basis_matrices) != len(matrices):
                raise ValueError("There must be as many basis matrices as there are matrices")
            return self.aux_init

        if self.aux_init == "random_uniform":
            coordinate_matrix = random_state.uniform(size=(rank, rank))
        elif self.aux_init == "random_standard_normal":
            coordinate_matrix = random_state.standard_normal(size=(rank, rank))
        elif self.aux_init == "zeros":
            coordinate_matrix = np.zeros((rank, rank))
        else:
            raise ValueError(f"Unknown aux init: {self.aux_init}")
        if _DEVICE_DRAW["device"] is not None:  # cmf_aoadmm fast path: P_i = eye(J_i, rank) is never built on the host
            return _EyeBases([int(M.shape[0]) for M in matrices], rank), coordinate_matrix
        return [np.eye(M.shape[0], rank) for M in matrices], coordinate_matrix

    def factor_matrices_update(self, factor_matrices, feasibility_penalties, auxes):  # penalties.py:1224-1250
        import torch

        from . import _ops

        _, coordinate_matrix = auxes
        devs = [_Dev(fm) for fm in factor_matrices]
        dtype = devs[0].t.dtype
        rank = int(coordinate_matrix.shape[0])
        sizes = [d.t.shape[0] for d in devs]
        n, n_groups = int(sum(sizes)), len(sizes)
        V = torch.cat([d.t.to(dtype) for d in devs], 0).contiguous()
        row_off = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64, device="cuda")
        gor = torch.repeat_interleave(torch.arange(n_groups, dtype=torch.int32, device="cuda"),
                                      torch.tensor(sizes, device="cuda"))
        delta = _Dev(coordinate_matrix).t.to(dtype).contiguous()
        rho = torch.as_tensor(np.asarray([float(r) for r in feasibility_penalties]), dtype=dtype).cuda()
        S = torch.empty(n_groups, rank, rank, dtype=dtype, device="cuda")
        Wm = torch.empty_like(S)
        num = torch.empty(n_groups, rank, rank, dtype=torch.float64, device="cuda")
        sums = torch.empty(rank * rank + 1, dtype=torch.float64, device="cuda")
        basis_in = auxes[0]
        new_delta = delta.clone()
        basis = None
        for it in range(int(self.n_iter)):  # penalties.py:1229-1248
            if self.update_basis_matrices:
                if it == 0:
                    _ops.slice_cross(V, None, row_off, n_groups, rank, None, S, None)
                if not bool(torch.any(new_delta != 0)):
                    # zero coordinate matrix (aux_init="zeros"): the reference's SVD of the zero matrix V_i Delta^T
                    # returns LAPACK's identity factors, i.e. P_i = eye(J_i, rank) (penalties.py:1233-1235)
                    basis = torch.cat([torch.eye(j, rank, dtype=dtype, device="cuda") for j in sizes], 0).contiguous()
                    _ops.pf2_fixed_basis(None, V, basis, None, row_off, n_groups, n, rank, rho, num, 1)
                else:
                    _ops.pf2_polar(S, new_delta, rho, n_groups, rank, Wm, num)
                    pd, basis = torch.empty_like(V), torch.empty_like(V)
                    _ops.pf2_apply(pd, V.clone(), basis, Wm, new_delta, gor, n, rank)
            if self.update_coordinate_matrix:
                if not self.update_basis_matrices:  # frozen P: numerator rho_g P_g^T V_g from the given bases
                    P = torch.cat([_Dev(b).t.to(dtype) for b in basis_in], 0).contiguous()
                    _ops.pf2_fixed_basis(None, V, P, None, row_off, n_groups, n, rank, rho, num, 1)
                _ops.pf2_delta(num, rho, n_groups, rank, new_delta, sums)
            if (not self.update_coordinate_matrix) or (not self.update_basis_matrices):
                break
        if basis is None:
            bases = list(basis_in)
        else:
            bases = [devs[i].back(b) for i, b in enumerate(torch.split(basis, sizes))]
        return bases, _Dev(coordinate_matrix).back(new_delta)

    def subtract_from_aux(self, aux, dual):
        raise TypeError("The PARAFAC2 constraint cannot shift a single factor matrix.")

    def subtract_from_auxes(self, auxes, duals):  # penalties.py:1256-1281
        P_is, coord_mat = auxes
        return [P_i @ coord_mat - dual for P_i, dual in zip(P_is, duals)]

    def aux_as_matrix(self, aux):
        raise TypeError("The PARAFAC2 constraint cannot convert a single aux to a matrix")

    def auxes_as_matrices(self, auxes):  # penalties.py:1287-1304
        P_is, coord_mat = auxes
        return [P_i @ coord_mat for P_i in P_is]

    def penalty(self, x):
        if not isinstance(x, list):
            raise TypeError("Cannot compute PARAFAC2 penalty of other types than a list of tensors")
        return 0


class _EnginePenaltyMixin:
    """Column-coupled penalties beyond L2Ball / Unimodality: the engine calls ``_engine_prox`` after every solve (the
    pre-image V = x + dual sits in ``dual``; the call must leave aux = prox(V) and dual = V - aux) and
    ``_engine_penalty`` for the value that enters the regularised loss (decomposition.py:1016-1023)."""

    def _engine_prox(self, eng, aux, dual, row_off, n_groups, max_rows, rho, n_rows):
        raise NotImplementedError

    def _engine_penalty(self, eng, x, row_off, n_groups, max_rows, n_rows, out):
        """Write the penalty value of the factor ``x`` (packed rows) into the 1-element device tensor ``out``."""
        out.zero_()

    def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):
        dev = _Dev(factor_matrix)
        V = dev.t if dev.t.dim() == 2 else dev.t.reshape(-1, 1)
        n_rows, rank = V.shape
        dual = V.clone()
        out = dev.torch.empty_like(V)
        rho = dev.torch.full((1,), float(feasibility_penalty), dtype=V.dtype, device="cuda")
        self._engine_prox(None, out, dual, _single_group_offsets(n_rows, "cuda"), 1, n_rows, rho, n_rows)
        return dev.back(out.reshape(dev.t.shape))

    def penalty(self, x):
        import torch

        xs = [x] if _is_tensor(x) else list(x)
        total = 0.0
        for xi in xs:
            dev = _Dev(xi)
            X = dev.t if dev.t.dim() == 2 else dev.t.reshape(-1, 1)
            out = torch.zeros(1, dtype=torch.float64, device="cuda")
            self._engine_penalty(None, X, _single_group_offsets(X.shape[0], "cuda"), 1, X.shape[0], X.shape[0], out)
            total += float(out.item())
        return total


class GeneralizedL2Penalty(_EnginePenaltyMixin, MatrixPenalty):
    """Penalty ``x^T M x`` on every column with a symmetric positive semidefinite ``M`` (penalties.py:595-747).
    The prox ``U diag(1 / (s + rho/2)) U^T (rho/2 x)`` (:724-730) runs as two batched GEMM-like kernels
    (csrc/prox_extra.cu).  The one-off spectral factorisation of ``M`` in the constructor is host LAPACK, like the
    reference's constructor (:720)."""

    _kind = _lib.PEN_GL2

    def __init__(self, norm_matrix, svd="truncated_svd", aux_init="random_uniform", dual_init="random_uniform",
                 validate=True):
        super().__init__(aux_init, dual_init)
        self.norm_matrix = norm_matrix
        self.svd = svd
        self.validate = validate
        M = np.asarray(norm_matrix.detach().cpu().numpy() if hasattr(norm_matrix, "detach") else norm_matrix,
                       dtype=np.float64)
        if validate and not np.all(M.T == M):
            raise ValueError("The norm matrix should be symmetric positive semidefinite")
        if validate and np.any(np.linalg.eigvals(M) < -1e-14):
            raise ValueError("The norm matrix should be symmetric positive semidefinite")
        self._M = M
        self._U, self._s, _ = np.linalg.svd(M, full_matrices=False)  # Vh ignored: the norm matrix is symmetric
        self._dev = {}

    def _descriptor(self):
        return (_lib.PEN_GL2, False, 0.0, 0.0)

    def _device_operands(self, dtype):
        import torch

        if dtype not in self._dev:
            up = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()  # noqa: E731
            self._dev[dtype] = (up(self._U), up(self._s), up(self._M))
        return self._dev[dtype]

    def _check_rows(self, n_rows, n_groups, max_rows):
        # b2_prox_gl2 / b2_quadform address slice g as rows [g J, (g + 1) J): EVERY slice must have exactly J rows
        # (heights that merely sum to n_groups * J would be processed in misaligned blocks; the reference fails with
        # a shape error in that case).  All heights <= max_rows and their sum == n_groups * J  <=>  all equal J.
        J = self._M.shape[0]
        if n_groups * J != n_rows or (n_groups > 0 and int(max_rows) != J):
            raise ValueError(
                f"GeneralizedL2Penalty with a {J} x {J} norm matrix needs factor matrices with {J} rows each "
                f"(got {n_rows} rows in {n_groups} matrices)")
        return J

    def _engine_prox(self, eng, aux, dual, row_off, n_groups, max_rows, rho, n_rows):
        from . import _ops

        J = self._check_rows(n_rows, n_groups, max_rows)
        U, s, _ = self._device_operands(aux.dtype)
        tmp = aux.new_empty((n_rows, aux.shape[1]))
        _ops.prox_gl2(aux, dual, n_groups, J, aux.shape[1], U, s, rho, tmp)

    def _engine_penalty(self, eng, x, row_off, n_groups, max_rows, n_rows, out):
        from . import _ops

        J = self._check_rows(n_rows, n_groups, max_rows)
        _, _, M = self._device_operands(x.dtype)
        _ops.quadform(M, x, n_groups, J, x.shape[1], out, x.new_empty((n_rows, x.shape[1])))


class TotalVariationPenalty(_EnginePenaltyMixin, MatrixPenalty):
    """Total variation (+ optional L1) on every column (penalties.py:750-841).  The reference delegates to the
    un-vendored GPL package ``condat_tv``; here Condat's direct algorithm runs as a CUDA kernel
    (csrc/prox_extra.cu::prox_tv_kernel), so no extra package is needed."""

    _kind = _lib.PEN_TV

    def __init__(self, reg_strength, l1_strength=0, aux_init="random_uniform", dual_init="random_uniform"):
        if reg_strength <= 0:
            raise ValueError("The TV regularization strength must be positive.")
        if l1_strength < 0:
            raise ValueError("The L1 regularization strength must be non-negative.")
        super().__init__(aux_init, dual_init)
        self.reg_strength = reg_strength
        self.l1_strength = l1_strength

    def _descriptor(self):
        return (_lib.PEN_TV, False, float(self.reg_strength), float(self.l1_strength))

    def _engine_prox(self, eng, aux, dual, row_off, n_groups, max_rows, rho, n_rows):
        from . import _ops

        _ops.prox_tv(aux, dual, row_off, n_groups, aux.shape[1], rho, self.reg_strength, self.l1_strength)

    def _engine_penalty(self, eng, x, row_off, n_groups, max_rows, n_rows, out):
        import torch

        from . import _ops

        _ops.tv_norm(x, row_off, n_groups, x.shape[1], out)
        out.mul_(float(self.reg_strength))
        if self.l1_strength:
            st = torch.zeros(3, dtype=torch.float64, device=x.device)
            _ops.reduce_stats(x, None, x.numel(), st, _ops.Workspace(x.device, 1, 1, x.dtype))
            out.add_(float(self.l1_strength) * st[2])


class UnitSimplex(_EnginePenaltyMixin, HardConstraintMixin, MatrixPenalty):
    """Non-negative columns that sum to one (penalties.py:928-980); the Lagrange multiplier of every column is found
    with the reference's bisection, all columns of a matrix at once (csrc/prox_extra.cu::prox_simplex_kernel)."""

    _kind = _lib.PEN_SIMPLEX

    def _descriptor(self):
        return (_lib.PEN_SIMPLEX, False, 0.0, 0.0)

    def _engine_prox(self, eng, aux, dual, row_off, n_groups, max_rows, rho, n_rows):
        from . import _ops

        _ops.prox_simplex(aux, dual, row_off, n_groups, max_rows, aux.shape[1])

    def penalty(self, x):
        return 0


class TemporalSmoothnessPenalty(_EnginePenaltyMixin, MatricesPenalty):
    """Smoothness of the mode-1 factor matrices over the slice order (temporal PARAFAC2 / CMF):

        g(B_0, ..., B_{I-1}) = smoothness_reg * sum_{i=1}^{I-1} ||B_i - B_{i-1}||_F^2

    i.e. ``x^T (smoothness_reg L) x`` with ``L`` the path-graph Laplacian over the slices, for every entry (j, r), in
    the convention of ``GeneralizedL2Penalty``.  The prox ``argmin g(Z) + sum_i rho_i / 2 ||Z_i - V_i||^2`` solves the
    tridiagonal system ``(diag(rho) + 2 smoothness_reg L) z = rho o v`` for every entry; all slices must have the same
    number of rows.  Mode 1 only (for smoothness over the rows of ``A`` or ``C`` use ``GeneralizedL2Penalty`` with a
    path-graph Laplacian).  The solve is a partition (spike) solve on the device (csrc/prox_temporal.cu); in a sharded
    run every rank is one block of it and the ranks exchange one small buffer per call."""

    _kind = _lib.PEN_TEMPORAL

    def __init__(self, smoothness_reg, aux_init="random_uniform", dual_init="random_uniform"):
        if not smoothness_reg > 0:
            raise ValueError("The smoothness regularization strength must be positive.")
        super().__init__(aux_init, dual_init)
        self.smoothness_reg = smoothness_reg
        self._ws = {}  # (n_slices, n_pos, world, device) -> device workspace of b2_prox_temporal

    def _descriptor(self):
        return (_lib.PEN_TEMPORAL, False, float(self.smoothness_reg), 0.0)

    @staticmethod
    def _check_heights(heights):
        found = sorted(set(int(h) for h in heights))
        if len(found) > 1:
            raise ValueError(
                "TemporalSmoothnessPenalty needs factor matrices with the same number of rows (B_i - B_(i-1) is "
                f"undefined otherwise); found heights {found}")
        return found[0] if found else 0

    def _workspace(self, n_slices, n_pos, world, device):
        from . import _ops

        key = (int(n_slices), int(n_pos), int(world), str(device))
        if key not in self._ws:
            self._ws[key] = _ops.prox_temporal_workspace(n_slices, n_pos, world, device)
        return self._ws[key]

    def _shape(self, eng, x, n_groups, max_rows, n_rows):
        """(slice height J, entries per slice J * R).  In an engine the height is the one checked at set-up, which
        a rank without slices also knows (the exchange buffers of a sharded run must have the same size on every
        rank)."""
        if eng is not None:
            J = eng.temporal_height
        else:
            J = int(max_rows) if n_groups else 0
            if n_groups * J != n_rows:
                raise ValueError(f"TemporalSmoothnessPenalty needs slices of equal height ({n_rows} rows in {n_groups} "
                                 f"slices of at most {max_rows} rows)")
        return J, J * x.shape[1]

    def _engine_prox(self, eng, aux, dual, row_off, n_groups, max_rows, rho, n_rows):
        import torch

        from . import _ops

        I = int(n_groups)
        _, P = self._shape(eng, aux, n_groups, max_rows, n_rows)
        lam = float(self.smoothness_reg)
        world = 1 if eng is None else eng.world
        ws = self._workspace(I, P, world, aux.device)
        if world == 1:
            _ops.prox_temporal(aux, dual, I, P, rho, lam, ws)
            return
        # sharded: this rank's slices are one block of the partition solve; the local solution's end values and the
        # ends of its two spike vectors go through one all-reduce, then every rank solves the 2 x world system
        lo, I_glob = eng.shard_rows
        rank = torch.distributed.get_rank(eng.group)
        xch = torch.zeros((world, 2 * P + 4), dtype=torch.float64, device=aux.device)
        kw = dict(has_left=lo > 0, has_right=lo + I < I_glob, xch=xch, world=world, rank=rank)
        _ops.prox_temporal(aux, dual, I, P, rho, lam, ws, stage=1, **kw)
        eng._allreduce(xch)
        _ops.prox_temporal(aux, dual, I, P, rho, lam, ws, stage=2, **kw)

    def _engine_penalty(self, eng, x, row_off, n_groups, max_rows, n_rows, out):
        import torch

        from . import _ops

        I = int(n_groups)
        J, P = self._shape(eng, x, n_groups, max_rows, n_rows)
        part = torch.empty(max(I, 1), dtype=torch.float64, device=x.device)
        lam = float(self.smoothness_reg)
        if eng is None or eng.world == 1:
            _ops.temporal_norm(x, I, P, lam, out, part)
            return
        # sharded: the pair (last slice of the previous rank with slices, first local slice) is counted here
        rank = torch.distributed.get_rank(eng.group)
        xch = torch.zeros((eng.world, P + 1), dtype=torch.float64, device=x.device)
        if I > 0:
            xch[rank, :P] = x[(I - 1) * J:].reshape(-1)
            xch[rank, P] = 1.0
        eng._allreduce(xch)
        _ops.temporal_norm(x, I, P, lam, out, part, xch=xch, rank=rank)

    def factor_matrices_update(self, factor_matrices, feasibility_penalties, auxes):
        import torch

        from . import _ops

        devs = [_Dev(fm) for fm in factor_matrices]
        if not devs:
            return []
        self._check_heights(d.t.shape[0] for d in devs)
        dtype = devs[0].t.dtype
        V = torch.cat([d.t.to(dtype).reshape(-1) for d in devs]).contiguous()
        I, P = len(devs), V.numel() // len(devs)
        rho = torch.as_tensor(np.asarray([float(r) for r in feasibility_penalties]), dtype=dtype).cuda()
        aux = torch.empty_like(V)
        _ops.prox_temporal(aux, V, I, P, rho, float(self.smoothness_reg), self._workspace(I, P, 1, V.device))
        return [d.back(a.view(d.t.shape)) for d, a in zip(devs, aux.view(I, P))]

    def penalty(self, x):
        import torch

        from . import _ops

        if not isinstance(x, list):
            raise TypeError("Cannot compute the temporal smoothness penalty of other types than a list of tensors")
        devs = [_Dev(xi) for xi in x]
        if len(devs) < 2:
            return 0.0
        self._check_heights(d.t.shape[0] for d in devs)
        dtype = devs[0].t.dtype
        X = torch.cat([d.t.to(dtype).reshape(-1) for d in devs]).contiguous()
        I = len(devs)
        out = torch.zeros(1, dtype=torch.float64, device="cuda")
        part = torch.empty(I, dtype=torch.float64, device="cuda")
        _ops.temporal_norm(X, I, X.numel() // I, float(self.smoothness_reg), out, part)
        return float(out.item())
