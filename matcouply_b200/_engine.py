"""Device-resident AO-ADMM engine: owns the packed data, the factor/aux/dual state in HBM and sequences the CUDA
kernels of one outer iteration (reference decomposition.py:945-988 -> admm_update_B :222, admm_update_C :295,
admm_update_A :120).  Host Python only launches kernels (through the C ABI) and reads back one small scalar pack per
outer iteration for the stopping rule.

Data layout in HBM (reference symbols: I slices X_i of J_i x K, N = sum J_i):
  X          N x ldx   packed row-major, ldx = K rounded up to 16 bytes (zero padded)  — read twice per outer iteration
  B, Y, W    N x R     packed per-slice factor, cached product Y = X C, scaled factor W = B o a (W has a 16-row zero tail)
  aux/dual   N x R     one pair per B-mode penalty (PARAFAC2: `pd` = P_i Delta in the aux slot, plus Delta R x R, W_i R x R)
  A, C       I x R, K x R with their aux/dual pairs
  per slice  rho (I), Minv (I x R x R), cross (I x R x R), rhsA (I x R)

X-stream schedule (exact Gauss-Seidel order of the reference, two passes instead of its three):
  Y = X C^(t)   (after the C-update; serves the A-update of iteration t and the B-update of iteration t+1)
  Z = X^T W     (after the B-update; serves the C-update)
Slice-local problems (every B-mode penalty row-local, fp64) run ONE pass per outer iteration (`fused_x1`, csrc/xfused.cu):
  per slice  Y_i = X_i C -> inner loop of the B-update -> G_i = X_i^T B_i -> Z += G_i diag(a_i)   while X_i is L2-resident;
  the A-update's diag(B_i^T X_i C_new) = colsum(G_i o C_new) then needs no further pass over X.

Sharding: with a process group, every rank holds a contiguous range of slices (X, B-state, A rows are rank-local);
C, Delta and all scalars are replicated through a few small all-reduces per outer iteration (SURVEY.md §8e).
"""
import os

import numpy as np
import torch

from . import _lib, _ops


# column-coupled kinds whose prox / penalty value is launched by the penalty object itself (penalties._EnginePenaltyMixin)
_ENGINE_PROX_KINDS = (_lib.PEN_GL2, _lib.PEN_SIMPLEX, _lib.PEN_TV, _lib.PEN_TEMPORAL)

# Kernel-fusion switches (tests flip them to cross-check the fused kernels against the one-kernel-per-step path).
# "x1": the single-read fused X-stream pass for slice-local B-updates (csrc/xfused.cu): one pass over X per outer
# iteration instead of two.  True = wherever the kernel applies, False = never, "auto" = where it is measured faster than
# the two-pass schedule: ranks <= 8 (one tensor-core column block), where the contraction is HBM-bound; from R = 9 on
# the two contractions of one launch are bound by the fp64 tensor pipe and the serial B-update between them is exposed
# (config 1, R = 16: 1.79 ms fused vs 1.57 ms for Y + Z + the fused ADMM loop; R = 8: 0.99 vs 1.44 ms; profiles/).
# Environment: B2_X1=1 / 0 / auto.
FUSION_DEFAULTS = {"local": True, "pf2": True, "overlap": True,
                   "x1": {"1": True, "0": False}.get(os.environ.get("B2_X1", "auto"), "auto")}
X1_AUTO_MAX_RANK = 8


class _Phase:
    """NVTX range around one phase of the outer iteration (SURVEY.md §5): makes nsys / ncu launch lists self-describing.
    A push/pop costs ~0.1 us without a profiler attached; B2_NVTX=0 turns the ranges off."""

    enabled = os.environ.get("B2_NVTX", "1") != "0"

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _Phase.enabled:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if _Phase.enabled:
            torch.cuda.nvtx.range_pop()
        return False


def _stack_rows(mats):
    """np.concatenate(mats, 0) without the copy when the matrices already are adjacent views of one array."""
    mats = [np.asarray(m) for m in mats]
    if len(mats) > 1 and all(m.flags.c_contiguous for m in mats):
        base = mats[0].base
        if isinstance(base, np.ndarray) and base.ndim == 2 and base.flags.c_contiguous and \
                all(m.base is base for m in mats) and mats[0].ctypes.data == base.ctypes.data and \
                all(b.ctypes.data == a.ctypes.data + a.nbytes for a, b in zip(mats[:-1], mats[1:])) and \
                sum(m.shape[0] for m in mats) == base.shape[0] and mats[0].shape[1] == base.shape[1]:
            return base
    return np.concatenate(mats, 0)


class PackedMatrices:
    """Ragged list of J_i x K matrices packed along rows (``np.concatenate(matrices, 0)``) on the device."""

    def __init__(self, X, row_offsets, K):
        self.X = X  # (N, ldx) CUDA tensor
        self.row_offsets = np.asarray(row_offsets, dtype=np.int64)
        self.K = int(K)
        self.N = int(self.row_offsets[-1])
        self.n_slices = len(self.row_offsets) - 1
        assert X.shape[0] >= self.N and X.shape[1] == _ops.padded_ld(self.K, X.dtype)

    @property
    def shapes(self):
        return [(int(j), self.K) for j in np.diff(self.row_offsets)]

    @classmethod
    def empty(cls, K, dtype, device):
        """No slice at all: the shard of a rank beyond the last slice of a sharded run."""
        return cls(torch.empty((0, _ops.padded_ld(int(K), dtype)), dtype=dtype, device=device), [0], int(K))

    @classmethod
    def from_list(cls, matrices, dtype, device):
        K = int(matrices[0].shape[1])
        sizes = [int(m.shape[0]) for m in matrices]
        for m in matrices:
            if len(m.shape) != 2 or int(m.shape[1]) != K:
                raise ValueError("All matrices must be two-dimensional with the same number of columns")
        N = int(sum(sizes))
        ld = _ops.padded_ld(K, dtype)
        X = torch.empty((N, ld), dtype=dtype, device=device)
        if ld != K:
            X[:, K:] = 0
        if all(isinstance(m, np.ndarray) for m in matrices):
            cls._upload_host_slices(X, matrices, sizes, K, dtype)
        else:
            r = 0
            for m in matrices:
                X[r:r + m.shape[0], :K] = torch.as_tensor(m).to(device=device, dtype=dtype)
                r += m.shape[0]
        return cls(X, np.concatenate([[0], np.cumsum(sizes)]), K)

    STAGE_BYTES = 128 << 20  # size of each of the two pinned staging buffers used for pageable inputs

    @classmethod
    def _upload_host_slices(cls, X, matrices, sizes, K, dtype):
        """Host -> HBM upload of the slice list, asynchronous on the current stream.

        Runs of slices that sit back to back in host memory are copied with one cudaMemcpyAsync each.  Page-locked
        inputs go straight from the caller's memory; pageable ones are staged through two alternating pinned buffers
        so the CPU-side gather of chunk n+1 overlaps the DMA of chunk n (no N x K pinned shadow copy)."""
        es = X.element_size()
        mats = [m if m.flags.c_contiguous else np.ascontiguousarray(m) for m in matrices]

        def root(a):
            while isinstance(getattr(a, "base", None), np.ndarray):
                a = a.base
            return a

        # merge slices that are views of ONE host allocation and adjacent in it (e.g. X[i] of a stacked array)
        runs, r = [], 0  # [first row, n rows, first slice index, n slices]
        for i, (m, J) in enumerate(zip(mats, sizes)):
            p = mats[i - 1] if i else None
            if runs and m.dtype == p.dtype and root(m) is root(p) and root(m) is not m and \
                    m.ctypes.data == p.ctypes.data + p.nbytes:
                runs[-1][1] += J
                runs[-1][3] += 1
            else:
                runs.append([r, J, i, 1])
            r += J

        def run_tensor(i0, cnt, nrows):
            m = mats[i0]
            if cnt > 1:
                m = np.lib.stride_tricks.as_strided(m, shape=(nrows, K), strides=(K * m.itemsize, m.itemsize),
                                                    writeable=False)
            return torch.from_numpy(m)

        stage, events, turn = [None, None], [None, None], 0
        for r0, nrows, i0, cnt in runs:
            if nrows == 0:
                continue
            import warnings

            with warnings.catch_warnings():
                warnings.simplefilter("ignore")  # read-only NumPy views: we only read
                src = run_tensor(i0, cnt, nrows)
            if src.is_pinned():
                X[r0:r0 + nrows, :K].copy_(src, non_blocking=True)
                continue
            # pageable: chunks of <= STAGE_BYTES through the pinned ring
            rows_per_chunk = max(1, cls.STAGE_BYTES // max(1, K * es))
            for c0 in range(0, nrows, rows_per_chunk):
                c1 = min(nrows, c0 + rows_per_chunk)
                if stage[turn] is None:
                    stage[turn] = torch.empty(rows_per_chunk * K, dtype=dtype, pin_memory=True)
                if events[turn] is not None:
                    events[turn].synchronize()  # the DMA that last read this buffer has finished
                buf = stage[turn][: (c1 - c0) * K].view(c1 - c0, K)
                buf.copy_(src[c0:c1])  # CPU gather (+ dtype conversion)
                X[r0 + c0:r0 + c1, :K].copy_(buf, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                events[turn] = ev
                turn ^= 1
        for ev in events:
            if ev is not None:
                ev.synchronize()  # staging buffers may be recycled by the allocator after return


class DeviceRows:
    """A list of per-slice ``J_i x R`` matrices held as ONE packed ``N x R`` CUDA tensor (what ``np.concatenate(list,
    0)`` would be).  Used for the B-mode variables that are drawn on the device (`_ops.mt19937_uniform`): they never
    exist on the host unless somebody indexes / iterates this object, which materialises NumPy arrays lazily."""

    def __init__(self, tensor, row_offsets):
        self.tensor = tensor
        self.row_offsets = np.asarray(row_offsets, dtype=np.int64)
        self._host = None

    def __len__(self):
        return len(self.row_offsets) - 1

    def _materialise(self):
        if self._host is None:
            flat = self.tensor.detach().to(torch.float64).cpu().numpy()
            self._host = [flat[a:b] for a, b in zip(self.row_offsets[:-1], self.row_offsets[1:])]
        return self._host

    def __getitem__(self, i):
        return self._materialise()[i]

    def __iter__(self):
        return iter(self._materialise())

    def cut(self, lo, hi):
        """Slices [lo, hi) as a DeviceRows (a view of the same device memory)."""
        off = self.row_offsets
        return DeviceRows(self.tensor[int(off[lo]):int(off[hi])], off[lo:hi + 1] - off[lo])


class ShardRows:
    """A mode-1 variable of a SHARDED run of which only this rank's slices ``[lo, hi)`` were drawn (the rest of the
    reference's RandomState stream was skipped with the MT19937 jump-ahead, `_ops.mt19937_skip`).  Stands in for the
    global list until `distributed.shard_state` cuts the rank's share out of it."""

    def __init__(self, local, lo, hi, n_global):
        self.local, self.lo, self.hi, self.n_global = local, int(lo), int(hi), int(n_global)

    def __len__(self):
        return self.n_global

    def cut(self, lo, hi):
        if (int(lo), int(hi)) != (self.lo, self.hi):
            raise ValueError(f"only slices [{self.lo}, {self.hi}) were drawn on this rank, not [{lo}, {hi})")
        return self.local

    def __getitem__(self, i):
        raise RuntimeError(f"only slices [{self.lo}, {self.hi}) of this variable exist on this rank")

    def __iter__(self):
        raise RuntimeError(f"only slices [{self.lo}, {self.hi}) of this variable exist on this rank")


class MaskCSR:
    """The missing entries of a mask as a CSR list over the packed rows: row n misses the columns
    ``col[row_ptr[n]:row_ptr[n+1]]`` (ascending).  ``row_ptr`` is int64 (N + 1), ``col`` int32; NumPy arrays when
    packed on the host, CUDA tensors once on the device."""

    def __init__(self, row_ptr, col, n_observed):
        self.row_ptr, self.col = row_ptr, col
        self.n_missing = int(row_ptr[-1]) if len(row_ptr) else 0
        self.n_observed = int(n_observed)

    def to(self, device):
        if isinstance(self.row_ptr, torch.Tensor):
            return MaskCSR(self.row_ptr.to(device), self.col.to(device), self.n_observed)
        return MaskCSR(torch.as_tensor(self.row_ptr).to(device), torch.as_tensor(self.col).to(device),
                       self.n_observed)

    def flat_index(self, ldx):
        """int64 offsets ``row * ldx + col`` of the missing entries in the flattened packed data (device tensors)."""
        n_rows = self.row_ptr.numel() - 1
        rows = torch.repeat_interleave(torch.arange(n_rows, device=self.col.device), torch.diff(self.row_ptr))
        return rows * int(ldx) + self.col.to(torch.int64)


def pack_mask(mask, shapes, require_observed=True):
    """Host packing of a per-slice mask (list of ``J_i x K`` arrays, NumPy or torch, bool or 0/1; 1 = observed) for
    data of the given slice shapes.  Raises ValueError for a shape mismatch, entries other than 0/1 or a mask without
    any observed entry."""
    shapes = [tuple(int(d) for d in s) for s in shapes]
    mask = list(mask)
    if len(mask) != len(shapes):
        raise ValueError(f"mask has {len(mask)} slices, the data has {len(shapes)}")
    counts, cols, n_obs = [np.zeros(1, dtype=np.int64)], [], 0
    for i, (m, s) in enumerate(zip(mask, shapes)):
        if isinstance(m, torch.Tensor):
            m = m.detach().cpu().numpy()
        m = np.asarray(m)
        if m.shape != s:
            raise ValueError(f"mask slice {i} has shape {m.shape}, the data slice has shape {s}")
        if m.dtype != np.bool_:
            if not np.all((m == 0) | (m == 1)):
                raise ValueError(f"mask slice {i} has entries other than 0 and 1")
            m = m != 0
        missing = ~m.reshape(s)
        counts.append(missing.sum(axis=1, dtype=np.int64))
        flat = np.flatnonzero(missing)  # row-major: ascending columns within each row
        cols.append((flat % max(s[1], 1)).astype(np.int32))
        n_obs += int(m.sum())
    if n_obs == 0 and require_observed:
        raise ValueError("the mask has no observed entry")
    row_ptr = np.cumsum(np.concatenate(counts)).astype(np.int64)
    col = np.concatenate(cols) if cols else np.zeros(0, dtype=np.int32)
    return MaskCSR(row_ptr, col, n_obs)


def pack_mask_device(mask, packed, require_observed=True):
    """Device packing of one ``(N, K)`` bool CUDA tensor over the packed rows of `packed` (PackedMatrices)."""
    if not isinstance(mask, torch.Tensor) or mask.dtype != torch.bool or mask.device != packed.X.device:
        raise ValueError(f"a single-tensor mask must be a bool tensor on {packed.X.device}")
    if tuple(mask.shape) != (packed.N, packed.K):
        raise ValueError(f"mask has shape {tuple(mask.shape)}, the packed data is {(packed.N, packed.K)}")
    missing = ~mask
    n_obs = int(mask.sum())
    if n_obs == 0 and require_observed:
        raise ValueError("the mask has no observed entry")
    row_ptr = torch.zeros(packed.N + 1, dtype=torch.int64, device=mask.device)
    torch.cumsum(missing.sum(dim=1), 0, out=row_ptr[1:])
    col = torch.nonzero(missing)[:, 1].to(torch.int32)  # row-major order: ascending within each row
    return MaskCSR(row_ptr, col, n_obs)


class _ModeState:
    """Factor matrix + per-penalty aux/dual of one mode, all flat (n x R) device tensors."""

    def __init__(self):
        self.x = None
        self.regs = []  # penalty objects (descriptors)
        self.desc = []  # (kind, nn, p0, p1)
        self.aux = []   # device tensors (PARAFAC2: P*Delta)
        self.dual = []
        self.descs_c = None


class AOADMMEngine:
    def __init__(self, packed, rank, regs, l2_penalty=(0, 0, 0), feasibility_penalty_scale=1.0, constant_A=False,
                 constant_B=False, inner_n_iter_max=5, update=(True, True, True), group=None, xstream_variant=None,
                 fuse_local=None, fuse_pf2=None, shard_rows=None, inner_tol=None, fuse_x1=None, mask=None):
        _lib.load()
        self.p = packed
        self.dev = packed.X.device
        self.dtype = packed.X.dtype
        self.R = int(rank)
        if not (1 <= self.R <= _lib.MAX_RANK):
            raise ValueError(f"matcouply_b200 supports rank 1..{_lib.MAX_RANK}, got {rank}")
        self.I, self.K, self.N = packed.n_slices, packed.K, packed.N
        self.l2 = [float(v) for v in l2_penalty]
        self.scale = float(feasibility_penalty_scale)
        self.const_A, self.const_B = bool(constant_A), bool(constant_B)
        self.n_inner = int(inner_n_iter_max)
        self.update_A, self.update_B, self.update_C = update
        self.group = group
        self.world = 1 if group is None else torch.distributed.get_world_size(group)
        # (first global slice index of this rank, global number of slices): needed by the matrix-wise mode-0 penalties
        self.shard_rows = (0, packed.n_slices) if shard_rows is None else (int(shard_rows[0]), int(shard_rows[1]))
        self.variant = _lib.VARIANT_AUTO if xstream_variant is None else xstream_variant
        self.fuse_local = FUSION_DEFAULTS["local"] if fuse_local is None else bool(fuse_local)
        self.fuse_pf2 = FUSION_DEFAULTS["pf2"] if fuse_pf2 is None else bool(fuse_pf2)
        # inner-loop convergence checks (decomposition.py:92-116) need a host decision after every inner iteration:
        # the one-kernel-per-step path is used and the fused whole-loop kernels are bypassed
        self.inner_tol = float(inner_tol) if inner_tol and inner_tol > 0 else None
        if self.inner_tol is not None:
            self.fuse_local = self.fuse_pf2 = False
        self.w_fresh = False
        R, I, K, N, dt, dev = self.R, self.I, self.K, self.N, self.dtype, self.dev

        self.row_off = torch.as_tensor(packed.row_offsets, dtype=torch.int64).to(dev)
        sizes = torch.as_tensor(np.diff(packed.row_offsets), dtype=torch.int64).to(dev)
        self.gor = torch.repeat_interleave(torch.arange(I, dtype=torch.int32, device=dev), sizes)
        self.max_rows = int(np.diff(packed.row_offsets).max()) if I else 0
        self.off_single_K = torch.tensor([0, K], dtype=torch.int64, device=dev)
        self.off_single_I = torch.tensor([0, I], dtype=torch.int64, device=dev)

        self.modes = [_ModeState(), _ModeState(), _ModeState()]
        for m in range(3):
            st = self.modes[m]
            st.mode = m
            st.regs = list(regs[m])
            if len(st.regs) > _lib.MAX_PENALTIES_PER_MODE:
                raise ValueError(f"at most {_lib.MAX_PENALTIES_PER_MODE} penalties per mode are supported")
            st.desc = [r._descriptor() for r in st.regs]
            if m != 1 and any(d[0] == _lib.PEN_TEMPORAL for d in st.desc):
                raise ValueError(
                    "TemporalSmoothnessPenalty can only be imposed with mode=1 (it couples B_i to B_(i-1)); for "
                    f"smoothness over the rows of {'A' if m == 0 else 'C'} use GeneralizedL2Penalty with a path-graph "
                    "Laplacian")
        if any(d[0] == _lib.PEN_TEMPORAL for d in self.modes[1].desc):
            self.temporal_height = self._common_slice_height(packed)
        for reg, (kind, *_) in zip(self.modes[0].regs, self.modes[0].desc):
            # a user-defined RowVectorPenalty has a row update; every other bridged / matrix-wise penalty needs ONE rho
            matrixwise = kind in _ENGINE_PROX_KINDS or (
                kind == _lib.PEN_HOST and not hasattr(reg, "factor_matrix_row_update"))
            if matrixwise:
                if not self.const_A:
                    raise AttributeError(
                        "Matrix-wise penalties on mode 0 have no row update: use constant_feasibility_penalty=True "
                        "(or 'A'), as with the reference"
                    )
            if matrixwise and self.world > 1:
                if kind == _lib.PEN_HOST:
                    raise NotImplementedError(
                        "user-defined matrix-wise penalties on a row-sharded mode 0 are not supported (their prox "
                        "couples all rows of A)")
                if shard_rows is None:
                    raise ValueError("matrix-wise penalties on a row-sharded mode 0 need `shard_rows`")
            if kind in (_lib.PEN_L2BALL, _lib.PEN_UNIMODAL):
                if not self.const_A:
                    raise AttributeError(
                        "Matrix-wise penalties (L2Ball, Unimodality) on mode 0 have no row update: "
                        "use constant_feasibility_penalty=True (or 'A'), as with the reference"
                    )
                if self.world > 1 and shard_rows is None:
                    raise ValueError("matrix-wise penalties on a row-sharded mode 0 need `shard_rows`")
            if kind == _lib.PEN_PARAFAC2:
                raise ValueError("PARAFAC2 constraint can only be imposed with mode=1")
        for kind, *_ in self.modes[2].desc:
            if kind == _lib.PEN_PARAFAC2:
                raise ValueError("PARAFAC2 constraint can only be imposed with mode=1")

        z = lambda *s: torch.zeros(s, dtype=dt, device=dev)  # noqa: E731
        self.Y = z(N, R)
        self.Wpad = _ops.alloc_w(N, R, dt, dev, self.variant)  # zero tail / pad columns required by b2_xstream_z
        self.ZL = z(K * R + R * R)             # Z (K x R) followed by lhs_C (R x R): one all-reduce buffer
        self.Z = self.ZL[: K * R].view(K, R)
        self.lhsC = self.ZL[K * R:].view(R, R)
        self.CtC = z(R, R)
        self.lhsB, self.MinvB, self.rhoB = z(I, R, R), z(I, R, R), z(I)
        self.cross, self.MinvA, self.rhoA, self.rhsA = z(I, R, R), z(I, R, R), z(I), z(I, R)
        self.BtB = z(I, R, R)  # per-slice Gram B_i^T B_i, refreshed whenever B changes
        self.MinvC, self.rhoC = z(1, R, R), z(1)
        self.rho_max = z(1)
        self.has_pf2 = any(d[0] == _lib.PEN_PARAFAC2 for d in self.modes[1].desc)
        if self.has_pf2:
            self.Delta = z(R, R)
            self.S, self.Wmat = z(I, R, R), z(I, R, R)
            self.num_part = torch.zeros(I, R, R, dtype=torch.float64, device=dev)
            self.pf2_sums = torch.zeros(R * R + 1, dtype=torch.float64, device=dev)
            self.pf2_basis0 = None   # initial basis matrices (host) until the first B-update replaces them
            self.pf2_fresh = False
            # deferred state: the PARAFAC2 dual slot holds the pre-image V of the last prox and (aux, dual) =
            # (V W_g Delta, V - V W_g Delta) exist only implicitly; _materialize_pf2() writes them out on demand
            self.pf2_deferred = False
            self.pf2_delta_zero = False  # Delta == 0 exactly (aux_init="zeros"): see _pf2_prox_unfused
            # One elementwise companion next to PARAFAC2 served by the steady-state row-pass kernel: the companion stays
            # ONE array T = x + dual across outer iterations too (`comp_T_state`: its dual slot holds T, aux is stale;
            # _materialize_companion() writes the pair out on demand) and its gap terms come out of the last row pass
            # (`comp_stats_fresh`: per-slice partials in comp_stats_part) instead of a pass over x and aux.
            d1 = self.modes[1].desc
            self.comp_keep_T = (len(d1) == 2 and d1[0][0] == _lib.PEN_PARAFAC2 and self.inner_tol is None and
                                _ops.pf2_rowpass_fused_stats_supported(R, dt, 2, d1[1][0], 1))
            self.comp_T_state = self.comp_stats_fresh = False
            self.comp_stats_part = torch.zeros(3 * max(I, 1), dtype=torch.float64, device=dev)
            self.pf2_gap_part = torch.zeros(3 * max(I, 1), dtype=torch.float64, device=dev)
            self.pf2_Q = torch.zeros(I, R, R, dtype=torch.float64, device=dev)  # Jacobi eigenvectors (warm start)
            self._polar_updates = 0
            self.polar_cold_every = max(1, int(os.environ.get("B2_POLAR_COLD_EVERY", "1")))
        # Single-read fused pass (SURVEY.md §8 row X1): applies when the whole B-update is slice-local and row-local.
        # The extra traffic is G (I x K x R, written by the pass and read once by the A-update), 2 R / mean(J_i) of X:
        # not worth it for very short slices.
        d1 = self.modes[1].desc
        want_x1 = FUSION_DEFAULTS.get("x1", "auto") if fuse_x1 is None else fuse_x1
        if want_x1 == "auto":
            want_x1 = R <= X1_AUTO_MAX_RANK
        self.fused_x1 = bool(
            want_x1 and self.fuse_local and self.update_B and I > 0 and N > 0 and dt == torch.float64
            and self.n_inner > 0 and len(d1) <= 2 and all(d[0] in (_lib.PEN_NONNEG, _lib.PEN_BOX, _lib.PEN_L1) for d in d1)
            and N >= 4 * R * I and _ops.xstream_fused_supported(K, R, dt, len(d1)))
        self.z_fresh = self.g_fresh = self.ctc_fresh = False
        if self.fused_x1:
            self.G = z(I, K, R)
            self.fws = _ops.FusedWorkspace(packed.row_offsets, K, R, dev)
        self.scal = torch.zeros(64, dtype=torch.float64, device=dev)
        self.normX_sq = None
        # Masked fitting (MaskCSR of the missing entries, or None): X holds the filled data F, whose missing entries are
        # refilled from the model after every outer iteration.  msum = [missing-entry part of ||F - X_hat||^2 of the
        # last refill, ||F||^2, ||F||^2 before the last refill]; kept out of `scal`, which is cleared per evaluation.
        self.mask = None
        if mask is not None:
            self.mask = mask.to(dev)
            if self.mask.row_ptr.numel() != N + 1:
                raise ValueError(f"the mask covers {self.mask.row_ptr.numel() - 1} rows, the data has {N}")
            self.msum = torch.zeros(3, dtype=torch.float64, device=dev)
            self.mask_ws = _ops.mask_refill_workspace(N, dev)
        uni = None
        if any(d[0] == _lib.PEN_UNIMODAL for d in self.modes[1].desc):
            uni = (I, R, self.max_rows)
        self.ws = _ops.Workspace(dev, K, R, dt, unimodal_shape=uni)
        # second stream for the fork/join of the PARAFAC2 inner iteration (see _step_B_pf2_fused)
        self.overlap_streams = FUSION_DEFAULTS.get("overlap", True) and self.world == 1
        if self.has_pf2:
            self._side = torch.cuda.Stream(device=dev)
            self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        self.n_xstream_launches = 0
        self.xstream_events = None  # set to {"y": [], "z": []} to record (start, end) CUDA events per launch

    def _common_slice_height(self, packed):
        """The height J shared by every slice of the (global) problem, for TemporalSmoothnessPenalty; sharded runs
        reduce the local minimum and maximum, so that every rank takes the same decision (a rank without slices
        learns J here)."""
        heights = sorted(set(int(h) for h in np.diff(packed.row_offsets)))
        if self.world > 1:
            mm = torch.tensor([heights[-1] if heights else -1, -heights[0] if heights else -(2 ** 52)],
                              dtype=torch.float64, device=self.dev)
            self._allreduce(mm, "max")
            lo_hi = (int(-mm[1].item()), int(mm[0].item()))
            heights = sorted(set(lo_hi)) if lo_hi[1] >= 0 else []
        if len(heights) > 1:
            raise ValueError(
                "TemporalSmoothnessPenalty needs factor matrices with the same number of rows (B_i - B_(i-1) is "
                f"undefined otherwise); found heights {heights if self.world == 1 else 'from %d to %d' % lo_hi}")
        return heights[0] if heights else 0

    # ------------------------------------------------------------------------------------------------------
    # state upload / download (host NumPy float64 <-> device)
    # ------------------------------------------------------------------------------------------------------
    def _up(self, a):
        return _ops.to_device(np.asarray(a), self.dtype, self.dev)

    def _up_rows(self, rows):
        """A mode-1 variable (list of J_i x R arrays, packed N x R array, or DeviceRows) as a packed device tensor."""
        if isinstance(rows, DeviceRows):
            src = rows.tensor
            t = src.to(device=self.dev, dtype=self.dtype)
            if t.data_ptr() != src.data_ptr():
                return t.contiguous()
            # same memory: adopt a freshly drawn block as the engine's state, but copy a shard cut out of the
            # (much larger) globally drawn block so that the latter can be freed
            whole = src.is_contiguous() and src.untyped_storage().nbytes() == src.numel() * src.element_size()
            return src if whole else src.clone()
        if isinstance(rows, np.ndarray):
            return self._up(rows)
        return self._up(_stack_rows(rows))

    def load_state(self, A, B_is, C, auxes, duals):
        """A: I x R, B_is: list of J_i x R (or packed N x R), C: K x R; auxes/duals: 3 lists as in ADMMVars."""
        st = self.modes
        self.z_fresh = self.g_fresh = self.ctc_fresh = False
        st[0].x = self._up(A)
        st[1].x = self._up_rows(B_is)
        st[2].x = self._up(C)
        for m in range(3):
            st[m].aux, st[m].dual = [], []
            for p, (kind, *_rest) in enumerate(st[m].desc):
                aux, dual = auxes[m][p], duals[m][p]
                if kind == _lib.PEN_PARAFAC2:
                    basis, delta = aux
                    self.pf2_fresh = False
                    self.pf2_deferred = False
                    self.pf2_delta_zero = not np.any(np.asarray(delta))
                    self.comp_T_state = self.comp_stats_fresh = False
                    self.Delta.copy_(self._up(delta))
                    if basis.__class__.__name__ == "_EyeBases":
                        # P_i = eye(J_i, R): row j < R of slice i of P_i Delta is Delta[j]; built on the device
                        self.pf2_basis0 = basis
                        pd = torch.zeros((self.N, self.R), dtype=self.dtype, device=self.dev)
                        starts, ends = self.row_off[:-1], self.row_off[1:]
                        for j in range(self.R):
                            ok = (ends - starts) > j
                            pd[(starts + j)[ok]] = self.Delta[j]
                        st[m].aux.append(pd)
                    else:
                        self.pf2_basis0 = [np.asarray(b, dtype=np.float64) for b in basis]
                        pd = np.concatenate([np.asarray(b) @ np.asarray(delta) for b in basis], 0)
                        st[m].aux.append(self._up(pd))
                elif m == 1:
                    st[m].aux.append(self._up_rows(aux))
                else:
                    st[m].aux.append(self._up(aux))
                if m == 1:
                    st[m].dual.append(self._up_rows(dual))
                else:
                    st[m].dual.append(self._up(dual))
            st[m].descs_c = _ops.make_descs(
                [(d[0], d[1], d[2], d[3], a, u) for d, a, u in zip(st[m].desc, st[m].aux, st[m].dual)])
        for m, n in ((0, self.I), (1, self.N), (2, self.K)):
            assert tuple(st[m].x.shape) == (n, self.R), (m, st[m].x.shape, (n, self.R))

    def load_state_device(self, seed=0):
        """Benchmark helper: uniform [0,1) factors / aux / dual drawn ON THE DEVICE (no host round trip of N x R
        arrays, no RNG parity with the reference — parity runs go through load_state)."""
        gen = torch.Generator(device=self.dev).manual_seed(int(seed))
        rnd = lambda *s: torch.rand(s, dtype=self.dtype, device=self.dev, generator=gen)  # noqa: E731
        st, R = self.modes, self.R
        self.z_fresh = self.g_fresh = self.ctc_fresh = False
        st[0].x, st[1].x, st[2].x = rnd(self.I, R), rnd(self.N, R), rnd(self.K, R)
        for m, n in ((0, self.I), (1, self.N), (2, self.K)):
            st[m].aux, st[m].dual = [], []
            for kind, *_r in st[m].desc:
                if kind == _lib.PEN_PARAFAC2:
                    self.Delta.copy_(rnd(R, R))
                    pd = torch.zeros((n, R), dtype=self.dtype, device=self.dev)
                    # P_i = eye(J_i, R): row j < R of slice i is Delta[j]
                    starts = self.row_off[:-1]
                    for j in range(R):
                        ok = (self.row_off[1:] - starts) > j
                        pd[(starts + j)[ok]] = self.Delta[j]
                    st[m].aux.append(pd)
                    self.pf2_basis0, self.pf2_fresh, self.pf2_deferred, self.pf2_delta_zero = None, False, False, False
                    self.comp_T_state = self.comp_stats_fresh = False
                else:
                    st[m].aux.append(rnd(n, R))
                st[m].dual.append(rnd(n, R))
            st[m].descs_c = _ops.make_descs(
                [(d[0], d[1], d[2], d[3], a, u) for d, a, u in zip(st[m].desc, st[m].aux, st[m].dual)])

    def _split(self, t):
        """Packed device rows -> list of per-slice NumPy arrays (views of ONE host array: no per-slice copies)."""
        t = t.detach().to(torch.float64)
        host_t = torch.empty(t.shape, dtype=torch.float64, pin_memory=True)  # DMA straight into page-locked memory
        host_t.copy_(t)
        host = host_t.numpy()
        return [host[a:b] for a, b in zip(self.p.row_offsets[:-1], self.p.row_offsets[1:])]

    def factors(self):
        st = self.modes
        f64 = lambda t: t.detach().to(torch.float64).cpu().numpy()  # noqa: E731
        return f64(st[0].x), self._split(st[1].x), f64(st[2].x)

    def admm_vars(self):
        """(auxes, duals) in the reference's ADMMVars layout (decomposition.py:1077-1081)."""
        f64 = lambda t: t.detach().to(torch.float64).cpu().numpy()  # noqa: E731
        self._materialize_companion()
        auxes, duals = ([], [], []), ([], [], [])
        for m in range(3):
            st = self.modes[m]
            for p, (kind, *_r) in enumerate(st.desc):
                if kind == _lib.PEN_PARAFAC2:
                    if self.pf2_fresh:
                        # P_i = V_i W_i with V = dual + P Delta (the pre-image of the last prox call)
                        self._materialize_pf2()
                        V = (st.dual[p] + st.aux[p]).contiguous()
                        basis, tmp = torch.empty_like(V), torch.empty_like(V)
                        _ops.pf2_apply(tmp, V, basis, self.Wmat, self.Delta, self.gor, self.N, self.R)
                        bases = self._split(basis)
                    else:
                        bases = list(self.pf2_basis0)
                    auxes[m].append((bases, f64(self.Delta)))
                elif m == 1:
                    auxes[m].append(self._split(st.aux[p]))
                else:
                    auxes[m].append(f64(st.aux[p]))
                duals[m].append(self._split(st.dual[p]) if m == 1 else f64(st.dual[p]))
        return auxes, duals

    # ------------------------------------------------------------------------------------------------------
    # collectives (no-ops on a single GPU)
    # ------------------------------------------------------------------------------------------------------
    def _allreduce(self, t, op="sum"):
        if self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == "sum" else dist.ReduceOp.MAX, group=self.group)

    # ------------------------------------------------------------------------------------------------------
    # pieces of one outer iteration
    # ------------------------------------------------------------------------------------------------------
    def _column_coupled(self, st, row_off, n_groups, max_rows, rho, gor, n_rows):
        """Finish the prox + dual update of the column-coupled penalties (V = x + dual is stored in `dual`)."""
        R = self.R
        for p, (kind, nn, p0, _p1) in enumerate(st.desc):
            if kind == _lib.PEN_L2BALL:
                _ops.prox_l2ball(st.aux[p], st.dual[p], row_off, n_groups, R, p0, nn)
            elif kind == _lib.PEN_UNIMODAL:
                _ops.prox_unimodal(st.aux[p], st.dual[p], row_off, n_groups, R, max_rows, nn, self.ws)
            elif kind in _ENGINE_PROX_KINDS:
                st.regs[p]._engine_prox(self, st.aux[p], st.dual[p], row_off, n_groups, max_rows, rho, n_rows)
            elif kind == _lib.PEN_HOST:
                self._host_prox(st, p, row_off, n_groups, rho)
            elif kind == _lib.PEN_PARAFAC2:
                self._pf2_prox_unfused(st, p, row_off, n_groups, rho, gor, n_rows)

    def _pf2_delta_update(self, rho, n_groups):
        """Delta = sum_g rho_g P_g^T V_g / sum_g rho_g from `num_part` (penalties.py:1240-1245); all-reduced when sharded."""
        R = self.R
        _ops.pf2_delta(self.num_part, rho, n_groups, R, self.Delta, self.pf2_sums)
        if self.world > 1:
            self._allreduce(self.pf2_sums)
            _ops.pf2_delta(self.num_part, rho, n_groups, R, self.Delta, None, self.pf2_sums)

    def _pf2_prox_unfused(self, st, p, row_off, n_groups, rho, gor, n_rows):
        """Parafac2.factor_matrices_update (penalties.py:1224-1250) with all its options: `n_iter` alternations of
        the basis update (polar factors) and the coordinate-matrix update on the same pre-image V; either update
        can be frozen (then a single pass, :1247-1248)."""
        reg, R = st.regs[p], self.R
        if reg.update_basis_matrices:
            _ops.slice_cross(st.dual[p], None, row_off, n_groups, R, None, self.S, None)
            n_it, polar_done = max(int(reg.n_iter), 0), False
            for it in range(n_it):
                if it == 0 and self.pf2_delta_zero:
                    # Delta == 0 (aux_init="zeros"): the reference takes the SVD of the ZERO matrix V_i Delta^T, for
                    # which LAPACK returns identity factors, i.e. P_i = eye(J_i, R) (penalties.py:1233-1235); the
                    # coordinate update then runs on that basis (:1240-1245)
                    if not reg.update_coordinate_matrix:
                        break
                    _ops.pf2_fixed_basis(None, st.dual[p], self._pf2_eye(), None, row_off, n_groups, n_rows, R, rho,
                                         self.num_part, 1)
                    self._pf2_delta_update(rho, n_groups)
                    self.pf2_delta_zero = False
                    continue
                _ops.pf2_polar(self.S, self.Delta, rho, n_groups, R, self.Wmat, self.num_part, self.pf2_Q,
                               warm=polar_done)
                polar_done = True
                if not reg.update_coordinate_matrix:
                    break
                self._pf2_delta_update(rho, n_groups)
            if polar_done:
                _ops.pf2_apply(st.aux[p], st.dual[p], None, self.Wmat, self.Delta, gor, n_rows, R)
                self.pf2_fresh = True
                return
            if n_it > 0:  # only the identity-basis step ran: P = eye(J_i, R), pd = P Delta
                from .penalties import _EyeBases

                self.pf2_basis0, self.pf2_fresh = _EyeBases(np.diff(self.p.row_offsets), R), False
                _ops.pf2_fixed_basis(st.aux[p], st.dual[p], self._pf2_eye(), self.Delta, row_off, n_groups, n_rows, R,
                                     None, None, 2)
                return
        # frozen basis matrices: P stays what it was given as (aux_init tuple or eye(J_i, R)); with n_iter == 0 the
        # reference returns the aux unchanged, which the same code covers (Delta untouched, pd = P Delta)
        P = self._pf2_fixed_basis()
        if reg.update_coordinate_matrix and int(reg.n_iter) > 0:
            _ops.pf2_fixed_basis(None, st.dual[p], P, None, row_off, n_groups, n_rows, R, rho, self.num_part, 1)
            self._pf2_delta_update(rho, n_groups)
        _ops.pf2_fixed_basis(st.aux[p], st.dual[p], P, self.Delta, row_off, n_groups, n_rows, R, None, None, 2)

    def _pf2_eye(self):
        """eye(J_i, R) of every slice as ONE packed N x R device tensor (built once)."""
        if getattr(self, "_pf2_eye_P", None) is None:
            P = torch.zeros((self.N, self.R), dtype=self.dtype, device=self.dev)
            starts, ends = self.row_off[:-1], self.row_off[1:]
            for j in range(self.R):
                ok = (ends - starts) > j
                P[(starts + j)[ok], j] = 1
            self._pf2_eye_P = P
        return self._pf2_eye_P

    def _pf2_fixed_basis(self):
        """The initial basis matrices as ONE packed N x R device tensor (built once)."""
        if getattr(self, "_pf2_P", None) is None:
            basis = self.pf2_basis0
            if basis is None or basis.__class__.__name__ == "_EyeBases":
                self._pf2_P = self._pf2_eye()
            else:
                self._pf2_P = self._up(np.concatenate([np.asarray(b) for b in basis], 0))
        return self._pf2_P

    def _host_prox(self, st, p, row_off, n_groups, rho):
        """Bridge to a user-defined ADMMPenalty subclass (examples/plot_custom_penalty.py:220-231 style): the
        pre-image V = x + dual (left in the dual slot by the solve kernel) and the current aux go to the Python
        method the reference would call (decomposition.py:202-211, 275-280, 333-337), the new aux comes back to HBM
        and dual = V - aux.  The prox itself is the user's code, wherever it runs; everything around it stays on
        the device."""
        reg, m = st.regs[p], st.mode
        V = st.dual[p].detach().to(torch.float64).cpu().numpy()
        aux = st.aux[p].detach().to(torch.float64).cpu().numpy()
        rhos = rho.detach().to(torch.float64).cpu().numpy()
        if m == 1:
            off = self.p.row_offsets
            cut = lambda a: [a[i:j] for i, j in zip(off[:-1], off[1:])]  # noqa: E731
            new = reg.factor_matrices_update(cut(V), [float(r) for r in rhos[:self.I]], cut(aux))
            new = np.concatenate([np.asarray(a) for a in new], 0)
        elif m == 2 or self.const_A:
            new = np.asarray(reg.factor_matrix_update(V, float(rhos[0]), aux))
        else:  # per-row feasibility penalties on mode 0 (decomposition.py:205-211)
            new = np.stack([np.asarray(reg.factor_matrix_row_update(V[i], float(rhos[i]), aux[i]))
                            for i in range(V.shape[0])], 0)
        st.aux[p].copy_(self._up(new))
        st.dual[p].sub_(st.aux[p])

    def _materialize_pf2(self):
        """Write out P Delta (aux slot) and dual = V - P Delta of the PARAFAC2 penalty if they are deferred."""
        if self.has_pf2 and self.pf2_deferred:
            st = self.modes[1]
            p = [d[0] for d in st.desc].index(_lib.PEN_PARAFAC2)
            _ops.pf2_apply(st.aux[p], st.dual[p], None, self.Wmat, self.Delta, self.gor, self.N, self.R)
            self.pf2_deferred = False

    def _materialize_companion(self):
        """Write out (aux, dual) = (prox(T), T - prox(T)) of the one-array companion if it is held as T."""
        if self.has_pf2 and self.comp_T_state:
            st = self.modes[1]
            kind, nn, p0, p1 = st.desc[1]
            # only rho-independent kinds are kept as T across outer iterations (non-negativity): rho = 1 is a dummy
            _ops.prox_elementwise(st.dual[1], st.aux[1], kind, nn, p0, p1, 1.0)
            st.dual[1].sub_(st.aux[1])
            self.comp_T_state = False

    def _timed(self, key, fn):
        """Run one kernel-family call; with `xstream_events` set (bench.py) bracket it with CUDA events on the
        launching stream.  Keys: "y" / "z" (X-stream passes), "rowpass", "polar", "unimodal", "local"."""
        if key in ("y", "z"):
            self.n_xstream_launches += 1
        if self.xstream_events is None:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        self.xstream_events.setdefault(key, []).append((e0, e1))

    def step_B(self):
        """admm_update_B (decomposition.py:222-292); rhs_i = Y_i o a_i with the cached Y = X C."""
        st, R, I = self.modes[1], self.R, self.I
        A, C = self.modes[0].x, self.modes[2].x
        if not self.ctc_fresh:  # refresh_products() of the previous iteration already left C^T C of this C behind
            _ops.gram(C, self.K, self.CtC, self.ws)
            self.ctc_fresh = True
        _ops.scale_gram(self.CtC, A, self.lhsB)
        _ops.rho_from_trace(self.lhsB, I, R, self.scale, self.rhoB, self.rho_max if self.const_B else None)
        if self.const_B:
            self._allreduce(self.rho_max, "max")
        _ops.factor_batch(self.lhsB, I, R, self.rhoB, self.rho_max if self.const_B else None, len(st.desc), self.l2[1],
                          self.MinvB)
        self.w_fresh = False
        if self.has_pf2:
            self.comp_stats_fresh = False
        if self.fused_x1:  # ONE pass over X: Y = X C, the inner loop, G_i = X_i^T B_i, Z and B_i^T B_i (csrc/xfused.cu)
            self._timed("fused", lambda: _ops.xstream_fused_local(
                self.p.X, self.N, self.K, self.row_off, I, self.fws, C, A, self.rhoB, self.MinvB, st.descs_c,
                len(st.desc), self.n_inner, st.x, self.Z, self.G, self.BtB))
            self.n_xstream_launches += 1
            self.z_fresh = self.g_fresh = True
            return
        self.z_fresh = self.g_fresh = False
        if self._row_local(st):  # whole inner loop in one fused pass, W = B o a emitted for the Z pass
            # W = B o a stays valid for the C-step: A only changes after the C-step (decomposition.py:948-988)
            self._timed("local", lambda: _ops.admm_local(
                self.N, R, self.Y, A, _lib.GROUP_INDEXED, self.gor, self.rhoB, self.MinvB, st.descs_c, len(st.desc),
                self.n_inner, st.x, self.Wpad, row_off=self.row_off, n_groups=I, BtB_out=self.BtB))
            self.w_fresh = True
            return
        if self.fuse_pf2 and self.n_inner > 0 and st.desc and st.desc[0][0] == _lib.PEN_PARAFAC2 and \
                not self.pf2_delta_zero and st.regs[0].update_basis_matrices and \
                st.regs[0].update_coordinate_matrix and int(st.regs[0].n_iter) >= 1:
            return self._step_B_pf2_fused()
        self._materialize_pf2()
        self._materialize_companion()
        for _ in range(self.n_inner):
            x_old = st.x.clone() if self.inner_tol is not None else None
            _ops.admm_solve(self.N, R, self.Y, A, _lib.GROUP_INDEXED, self.gor, self.rhoB, self.MinvB, st.descs_c,
                            len(st.desc), st.x)
            self._column_coupled(st, self.row_off, I, self.max_rows, self.rhoB, self.gor, self.N)
            if self._inner_converged(1, x_old):
                break
        _ops.slice_gram(st.x, self.row_off, I, R, self.BtB)

    def _step_B_pf2_fused(self):
        """PARAFAC2 B-mode inner loop with the fused row pass (csrc/pf2_fused.cu): per inner iteration one pass over
        the B-state (deferred prox of the previous iteration + solve + other penalties + Gram), the CTA-parallel polar
        step and the Delta reduction; P Delta / dual are materialised once at the end."""
        st, R, I = self.modes[1], self.R, self.I
        A = self.modes[0].x
        for it in range(self.n_inner):
            last = it == self.n_inner - 1
            # deferred from the start when the previous outer iteration left (V, W_g, Delta) behind
            # flag bits: 1 = PARAFAC2 prox deferred; 2 / 4 = the elementwise companions arrive / leave as ONE array
            # T = x + dual (aux = prox(T) and dual = T - aux are recomputed in registers): explicit (aux, dual) are only
            # read by the first and written by the last pass of a B-update, which saves two N x R arrays of traffic
            # per companion in every other pass
            deferred = it > 0 or self.pf2_deferred
            # the steady-state kernel (deferred prox) can leave the companion as T on the last pass too and emit its
            # gap terms; otherwise the last pass writes the explicit (aux, dual) pair
            keep_T = last and self.comp_keep_T and deferred
            tin = it > 0 or self.comp_T_state
            flags = (1 if deferred else 0) | (2 if tin else 0) | (4 if (not last or keep_T) else 0)
            stats = self.comp_stats_part if keep_T else None
            self._timed("rowpass", lambda: _ops.pf2_rowpass(
                self.row_off, I, R, self.Y, A, self.rhoB, self.MinvB, st.descs_c, len(st.desc), flags, self.Wmat,
                self.Delta, st.x if last else None, self.Wpad if last else None, self.S, self.BtB if last else None,
                stats))
            if last:
                self.comp_T_state = self.comp_stats_fresh = keep_T
            # The polar step + Delta reduction only need S (from the row pass); the column-coupled companions only
            # need their own pre-image.  With such companions (Unimodality above all: a latency-bound kernel that
            # leaves most of the SM idle) the two chains run on two streams and join before the next row pass.
            coupled = [p for p, d in enumerate(st.desc) if p > 0 and d[0] not in
                       (_lib.PEN_NONNEG, _lib.PEN_BOX, _lib.PEN_L1)]
            fork = bool(coupled) and self.overlap_streams
            def companion(p):  # V is in the companion's dual slot
                kind, nn, p0, _p1 = st.desc[p]
                if kind == _lib.PEN_L2BALL:
                    _ops.prox_l2ball(st.aux[p], st.dual[p], self.row_off, I, R, p0, nn)
                elif kind == _lib.PEN_UNIMODAL:
                    self._timed("unimodal", lambda: _ops.prox_unimodal(st.aux[p], st.dual[p], self.row_off, I, R,
                                                                       self.max_rows, nn, self.ws))
                elif kind in _ENGINE_PROX_KINDS:
                    st.regs[p]._engine_prox(self, st.aux[p], st.dual[p], self.row_off, I, self.max_rows, self.rhoB,
                                            self.N)
                elif kind == _lib.PEN_HOST:
                    self._host_prox(st, p, self.row_off, I, self.rhoB)

            if fork:
                # main stream: the most expensive companion (Unimodality if present); side stream: polar + Delta and
                # the remaining companions (independent arrays)
                order = sorted(coupled, key=lambda p: st.desc[p][0] != _lib.PEN_UNIMODAL)
                device_only = [p for p in order[1:] if st.desc[p][0] != _lib.PEN_HOST]
                main = torch.cuda.current_stream(self.dev)
                self._ev_fork.record(main)
                with torch.cuda.stream(self._side):
                    self._side.wait_event(self._ev_fork)
                    self._pf2_polar_delta(st, I, it)
                    for p in device_only:
                        companion(p)
                    self._ev_join.record(self._side)
                for p in order:
                    if p == order[0] or p not in device_only:
                        companion(p)
                main.wait_event(self._ev_join)
            else:
                for p in coupled:
                    companion(p)
                self._pf2_polar_delta(st, I, it)
        # P Delta and dual = V - P Delta stay implicit: the next row pass and the gap reduction apply W_g Delta on the fly
        self.pf2_deferred = True
        self.pf2_fresh = True
        self.w_fresh = True

    def _pf2_polar_delta(self, st, I, it):
        """Polar step + coordinate-matrix update of one inner iteration (penalties.py:1229-1245)."""
        # warm Jacobi start from the eigenvectors of the previous inner iteration (3-5 sweeps instead of 8-10); the first
        # inner iteration of every `polar_cold_every`-th B-update starts cold, which bounds the round-off drift of the
        # accumulated rotations.  Default 1 = every B-update: B2_POLAR_COLD_EVERY=8 saves 11 % of the polar time
        # (0.8 % of a config-2 step, profiles/r2_ab_polar_warm_s43.txt) but moves the trajectory by ~1e-13 per step,
        # which one of the 24 random differential configurations (UnitSimplex + PARAFAC2) amplifies to 1.3e-7 > 1e-7
        for sub in range(int(st.regs[0].n_iter)):  # Parafac2(n_iter=...): alternations on the same V
            # (a captured iteration is replayed as it is: keep its first polar step cold)
            cold = it == 0 and sub == 0 and (self._polar_updates % self.polar_cold_every == 0
                                             or torch.cuda.is_current_stream_capturing())
            self._timed("polar", lambda: _ops.pf2_polar(self.S, self.Delta, self.rhoB, I, self.R, self.Wmat,
                                                        self.num_part, self.pf2_Q, warm=not cold))
            self._pf2_delta_update(self.rhoB, I)
        if it == 0:
            self._polar_updates += 1

    def _row_local(self, st):
        """True when every penalty of the mode is elementwise (the fused b2_admm_local path applies)."""
        return self.fuse_local and self.n_inner > 0 and len(st.desc) <= 2 and all(
            d[0] in (_lib.PEN_NONNEG, _lib.PEN_BOX, _lib.PEN_L1) for d in st.desc)

    def step_C(self):
        """admm_update_C (decomposition.py:295-344); one X pass: Z = X^T (B o a)."""
        st, R, K = self.modes[2], self.R, self.K
        self.ctc_fresh = False  # C changes below
        if self.z_fresh:  # Z = sum_i G_i diag(a_i) came out of the fused pass (A has not changed since)
            self.z_fresh = False
        else:
            if not getattr(self, "w_fresh", False):
                _ops.rowscale(self.modes[1].x, self.modes[0].x, self.gor, self.N, R, self.Wpad)
            self._timed("z", lambda: _ops.xstream_z(self.p.X, self.N, K, self.Wpad, self.Z, self.ws, self.variant))
        self.w_fresh = False
        _ops.weighted_gram_sum(self.BtB, self.modes[0].x, self.I, R, self.lhsC)  # sum_i (B_i a_i)^T (B_i a_i)
        self._allreduce(self.ZL)
        _ops.rho_from_trace(self.lhsC, 1, R, self.scale, self.rhoC, None)
        _ops.factor_batch(self.lhsC, 1, R, self.rhoC, None, len(st.desc), self.l2[2], self.MinvC)
        if self._row_local(st):
            _ops.admm_local(K, R, self.Z, None, _lib.GROUP_SINGLE, None, self.rhoC, self.MinvC, st.descs_c,
                            len(st.desc), self.n_inner, st.x)
            return
        for _ in range(self.n_inner):
            x_old = st.x.clone() if self.inner_tol is not None else None
            _ops.admm_solve(K, R, self.Z, None, _lib.GROUP_SINGLE, None, self.rhoC, self.MinvC, st.descs_c,
                            len(st.desc), st.x)
            self._column_coupled(st, self.off_single_K, 1, K, self.rhoC, None, K)
            if self._inner_converged(2, x_old):
                break

    def refresh_products(self):
        """Y = X C (one X pass), CtC, cross_i = (B_i^T B_i) o CtC, rhsA_i = colsum(B_i o Y_i)
        (decomposition.py:138-158).  Also what the fit term needs (:446-449)."""
        C, B = self.modes[2].x, self.modes[1].x
        _ops.gram(C, self.K, self.CtC, self.ws)
        self.ctc_fresh = True
        _ops.hadamard_bcast(self.BtB, self.CtC, self.I, self.R, self.cross)
        if self.g_fresh:
            # G_i = X_i^T B_i of the current B is at hand (fused pass): diag(B_i^T X_i C) = colsum_k(G_i o C), no X pass.
            # The next B-update is a fused pass again and computes its own Y = X C.
            _ops.slice_gdot(self.G, C, self.I, self.K, self.R, self.rhsA)
            return
        self._timed("y", lambda: _ops.xstream_y(self.p.X, self.N, self.K, C, self.Y, self.ws, self.variant))
        _ops.slice_coldot(B, self.Y, self.row_off, self.I, self.R, self.rhsA)

    def step_A(self):
        """admm_update_A (decomposition.py:120-219) after refresh_products()."""
        st, R, I = self.modes[0], self.R, self.I
        _ops.rho_from_trace(self.cross, I, R, self.scale, self.rhoA, self.rho_max if self.const_A else None)
        if self.const_A:
            self._allreduce(self.rho_max, "max")
        _ops.factor_batch(self.cross, I, R, self.rhoA, self.rho_max if self.const_A else None, len(st.desc), self.l2[0],
                          self.MinvA)
        if self._row_local(st):
            _ops.admm_local(I, R, self.rhsA, None, _lib.GROUP_IDENTITY, None, self.rhoA, self.MinvA, st.descs_c,
                            len(st.desc), self.n_inner, st.x)
            return
        for _ in range(self.n_inner):
            x_old = st.x.clone() if self.inner_tol is not None else None
            _ops.admm_solve(I, R, self.rhsA, None, _lib.GROUP_IDENTITY, None, self.rhoA, self.MinvA, st.descs_c,
                            len(st.desc), st.x)
            if self.world > 1:
                self._column_coupled_A_sharded(st)
            else:
                self._column_coupled(st, self.off_single_I, 1, I, self.rhoA, None, I)
            if self._inner_converged(0, x_old):
                break

    def _inner_converged(self, mode, x_old):
        """_check_inner_convergence (decomposition.py:92-116): relative change of the factor <= inner_tol and, with
        penalties, every feasibility gap of this mode < inner_tol.  One fused reduction + one D2H per inner iteration;
        sharded modes (0, 1) all-reduce the sums so that every rank takes the same decision."""
        if self.inner_tol is None:
            return False
        st = self.modes[mode]
        n = (self.I, self.N, self.K)[mode] * self.R
        scal = self.scal
        scal.zero_()
        _ops.reduce_stats(st.x, x_old, n, scal[0:3], self.ws)
        for p in range(len(st.desc)):
            _ops.reduce_stats(st.x, st.aux[p], n, scal[3 + 3 * p:6 + 3 * p], self.ws)
        used = 3 + 3 * len(st.desc)
        if self.world > 1 and mode != 2:
            self._allreduce(scal[:used])
        host = scal[:used].cpu().numpy()
        change, norm = np.sqrt(host[0]), np.sqrt(host[1])
        if change > self.inner_tol * norm:
            return False
        if len(st.desc) == 0:
            return True
        gaps = [np.sqrt(host[3 + 3 * p]) / np.sqrt(host[4 + 3 * p]) for p in range(len(st.desc))]
        return max(gaps) < self.inner_tol

    def _column_coupled_A_sharded(self, st):
        """Matrix-wise penalties on mode 0 when the rows of A are sharded over ranks (SURVEY.md §8e, last row):
        L2Ball needs the column norms over ALL I rows -> all-reduce of R partial sums of squares (penalties.py:923);
        Unimodality needs whole columns -> the I x R pre-image is gathered (sum of disjoint row blocks), the prox runs
        replicated and every rank keeps its rows (penalties.py:1015)."""
        R, I = self.R, self.I
        lo, I_glob = self.shard_rows
        for p, (kind, nn, p0, _p1) in enumerate(st.desc):
            if kind == _lib.PEN_L2BALL:
                colsq = torch.zeros(R, dtype=torch.float64, device=self.dev)
                if I > 0:
                    _ops.prox_l2ball(st.aux[p], st.dual[p], self.off_single_I, 1, R, p0, nn, colsq, phase=1)
                self._allreduce(colsq)
                if I > 0:
                    _ops.prox_l2ball(st.aux[p], st.dual[p], self.off_single_I, 1, R, p0, nn, colsq, phase=2)
            elif kind == _lib.PEN_UNIMODAL:
                full = torch.zeros((I_glob, R), dtype=self.dtype, device=self.dev)
                full[lo:lo + I] = st.dual[p]
                self._allreduce(full)
                aux_full = torch.empty_like(full)
                off = torch.tensor([0, I_glob], dtype=torch.int64, device=self.dev)
                _ops.prox_unimodal(aux_full, full, off, 1, R, I_glob, nn, self.ws)
                st.aux[p].copy_(aux_full[lo:lo + I])
                st.dual[p].copy_(full[lo:lo + I])
            elif kind == _lib.PEN_HOST:
                # user-defined ROW-wise penalty (matrix-wise ones are refused for a sharded mode 0 in __init__): rows
                # are rank-local, the bridge runs on this rank's rows
                if I > 0:
                    self._host_prox(st, p, self.off_single_I, 1, self.rhoA)
            elif kind in _ENGINE_PROX_KINDS:
                # GeneralizedL2 / UnitSimplex / TV over all I rows: same gather, prox replicated, own rows kept
                full = self._gather_A_rows(st.dual[p])
                aux_full = torch.empty_like(full)
                off = torch.tensor([0, I_glob], dtype=torch.int64, device=self.dev)
                st.regs[p]._engine_prox(self, aux_full, full, off, 1, I_glob, self.rhoA[:1] if I > 0 else self.rho_max,
                                        I_glob)
                st.aux[p].copy_(aux_full[lo:lo + I])
                st.dual[p].copy_(full[lo:lo + I])

    def _gather_A_rows(self, local):
        """The complete I_glob x R matrix from the row shards (all-reduce of disjoint row blocks)."""
        lo, I_glob = self.shard_rows
        full = torch.zeros((I_glob, self.R), dtype=self.dtype, device=self.dev)
        full[lo:lo + self.I] = local
        self._allreduce(full)
        return full

    def prepare(self):
        """Before the first iteration: ||X||^2 and the products for the initial fit (decomposition.py:906-913).
        With a mask: the missing entries are zeroed, so that ||X||^2 = ||M o X||^2, and then filled from the initial
        factors (F^(0))."""
        out = self.scal[60:61]
        if self.mask is not None:
            self.p.X.view(-1)[self.mask.flat_index(self.p.X.shape[1])] = 0
        _ops.sumsq(self.p.X, self.N, self.K, out, self.ws)
        if self.mask is not None:
            self.msum[1].copy_(out[0])  # rank-local ||F||^2
        self._allreduce(out)
        self.normX_sq = float(out.item())
        _ops.slice_gram(self.modes[1].x, self.row_off, self.I, self.R, self.BtB)
        if self.mask is not None:
            self.refill(None)
            # F^(0) equals the initial model at the missing entries: the initial fit has no missing-entry term
            self.msum[2].copy_(self.msum[1])
            self.msum[0].zero_()
        self.refresh_products()

    def refill(self, Y):
        """F <- M o X + (1 - M) o X_hat(A, B, C) (b2_mask_refill); Y += the matching rank-R correction (if given)."""
        m = self.mask
        self.msum[2].copy_(self.msum[1])
        self.msum[0].zero_()
        self._timed("refill", lambda: _ops.mask_refill(
            self.p.X, self.N, self.K, m.row_ptr, m.col, self.gor, self.modes[0].x, self.modes[1].x, self.modes[2].x, Y,
            self.msum[0:2], self.mask_ws))

    def outer_iteration(self):
        """One pass of decomposition.py:945-988."""
        if self.update_B:
            with _Phase("b2:admm_update_B"):
                self.step_B()
        if self.update_C:
            with _Phase("b2:admm_update_C"):
                self.step_C()
        if self.update_B or self.update_C or self.mask is not None:  # F, and with it X C, changes with every refill
            with _Phase("b2:xstream_y+products"):
                self.refresh_products()
        if self.update_A:
            with _Phase("b2:admm_update_A"):
                self.step_A()
        if self.mask is not None:
            with _Phase("b2:mask_refill"):
                # the next B-update reads the cached Y = F C (two-pass schedule, PARAFAC2 row pass) unless it is the
                # single-read fused pass, which computes its own Y from X
                self.refill(None if self.fused_x1 else self.Y)

    # ------------------------------------------------------------------------------------------------------
    # diagnostics: one fused scalar pack, one device->host copy
    # ------------------------------------------------------------------------------------------------------
    def diagnostics(self):
        """Returns dict(gaps=(A_gaps, B_gaps, C_gaps), sse_terms=(inner, quad), sq=[|A|^2,|B|^2,|C|^2],
        l1=[[...],[...],[...]] sums of |x| per penalty) — everything the host loss/stopping logic needs
        (decomposition.py:351-417, 420-452, 617-627, 1016-1023)."""
        return self._read_diagnostics(self._launch_diagnostics())

    def _launch_diagnostics(self):
        """Launch the fused reductions into the scalar pack `self.scal`; returns (layout, n_slots). No host sync."""
        with _Phase("b2:gaps+fit"):
            return self._launch_diagnostics_impl()

    def _launch_diagnostics_impl(self):
        scal = self.scal
        scal.zero_()
        slot = 2  # [0:2] fit terms
        _ops.fit_terms(self.rhsA, self.cross, self.modes[0].x, self.I, self.R, scal[0:2], self.ws)
        if self.mask is not None:  # [2:4] ||F^(t-1)||^2 and the missing-entry term (rank-local: all-reduced part)
            scal[2].copy_(self.msum[2])
            scal[3].copy_(self.msum[0])
            slot = 4
        layout, deferred_A = [], []
        sizes = (self.I * self.R, self.N * self.R, self.K * self.R)
        # sharded modes first (A, B), replicated mode (C) last
        for m in (0, 1, 2):
            st = self.modes[m]
            if m == 2:
                shard_end = slot
            if len(st.desc) == 0:
                _ops.reduce_stats(st.x, None, sizes[m], scal[slot:slot + 3], self.ws)
                layout.append((m, -1, slot))
                slot += 3
            for p in range(len(st.desc)):
                if m == 1 and st.desc[p][0] == _lib.PEN_PARAFAC2 and self.pf2_deferred:
                    _ops.pf2_gap(st.dual[p], st.x, self.row_off, self.I, self.R, self.Wmat, self.Delta,
                                 scal[slot:slot + 3], self.pf2_gap_part)
                elif m == 1 and p == 1 and self.has_pf2 and self.comp_stats_fresh:
                    _ops.group_stats_sum(self.comp_stats_part, self.I, scal[slot:slot + 3])  # from the last row pass
                else:
                    if m == 1 and p == 1 and self.has_pf2:
                        self._materialize_companion()
                    _ops.reduce_stats(st.x, st.aux[p], sizes[m], scal[slot:slot + 3], self.ws)
                layout.append((m, p, slot))
                slot += 3
            for p in range(len(st.desc)):  # values of the penalties that are not hard constraints (loss terms)
                if st.desc[p][0] in _ENGINE_PROX_KINDS and st.desc[p][0] != _lib.PEN_SIMPLEX:
                    if m == 0 and self.world > 1:
                        deferred_A.append(p)  # couples all rows of A: evaluated on the gathered matrix below
                        continue
                    off_m, n_g, mx = ((self.off_single_I, 1, self.I), (self.row_off, self.I, self.max_rows),
                                      (self.off_single_K, 1, self.K))[m]
                    st.regs[p]._engine_penalty(self, st.x, off_m, n_g, mx, sizes[m] // self.R, scal[slot:slot + 1])
                    layout.append((m, -2 - p, slot))
                    slot += 1
        if deferred_A:  # replicated values (identical on every rank): after the all-reduced part of the pack
            I_glob = self.shard_rows[1]
            full = self._gather_A_rows(self.modes[0].x)
            off = torch.tensor([0, I_glob], dtype=torch.int64, device=self.dev)
            for p in deferred_A:
                self.modes[0].regs[p]._engine_penalty(self, full, off, 1, I_glob, I_glob, scal[slot:slot + 1])
                layout.append((0, -2 - p, slot))
                slot += 1
        if self.world > 1:
            self._allreduce(scal[:shard_end])
        return layout, slot

    def _read_diagnostics(self, launched):
        """The ONE device->host copy (and sync) of an outer iteration."""
        layout, slot = launched
        host = self.scal[:slot].cpu().numpy()
        gaps, sq, l1 = ([], [], []), [0.0, 0.0, 0.0], ([], [], [])
        extra = ({}, {}, {})
        for m, p, s in layout:
            if p <= -2:
                extra[m][-2 - p] = float(host[s])
                continue
            d2, x2, ab = host[s:s + 3]
            sq[m] = x2
            if p >= 0:
                gaps[m].append(np.sqrt(d2) / np.sqrt(x2))
                l1[m].append(ab)
        out = dict(gaps=gaps, fit=(host[0], host[1]), sq=sq, l1=l1, extra=extra)
        if self.mask is not None:
            out["masked"] = (host[2], host[3])
        return out

    # ------------------------------------------------------------------------------------------------------
    # CUDA-graph replay of the steady-state outer iteration (launch-bound problem sizes)
    # ------------------------------------------------------------------------------------------------------
    GRAPH_MAX_X_BYTES = 1 << 30  # below this an outer iteration is dominated by launch latency, not by HBM time

    def graph_eligible(self):
        """Small single-GPU problems: ~50-100 kernel launches per outer iteration cost more than the kernels.  The
        launch sequence of a steady-state iteration is fixed (same kernels, same buffers), so it is captured once
        into a CUDA graph and replayed; the host only reads the scalar pack.  Sharded runs stay eager (NCCL calls)."""
        return (self.world == 1 and self.xstream_events is None
                and (self.N * self.K * self.p.X.element_size() <= self.GRAPH_MAX_X_BYTES or self.graph_auto()))

    def graph_auto(self):
        """Problems for which the graph replay is switched on without being asked for: single GPU, no PARAFAC2 (its
        inner iteration forks onto a second stream and the replay measured SLOWER there: config 3 41.3 vs 28.6 ms), only
        penalties whose prox is one kernel on the main stream, no host decisions inside the iteration.  The ~45 short
        dependent launches of such an iteration leave 5-10 % of the step to launch gaps when issued one by one from
        Python (config 1: 2.01 -> 1.91 ms, the same shapes at R = 8 on the fused pass: 1.26 -> 1.14 ms)."""
        simple = (_lib.PEN_NONNEG, _lib.PEN_BOX, _lib.PEN_L1, _lib.PEN_L2BALL)
        return (self.world == 1 and self.xstream_events is None and not self.has_pf2 and self.inner_tol is None
                and not getattr(self, "_graph_failed", False)
                and all(d[0] in simple for m in self.modes for d in m.desc))

    def graph_iteration(self, with_diagnostics):
        """One outer iteration (+ the diagnostics reductions) as a graph replay; captured on first use.  Must only be
        called once the host-side state flags are steady (after >= 2 eager iterations).  Returns what
        _launch_diagnostics() returns, or None."""
        key = bool(with_diagnostics)
        if not hasattr(self, "_graphs"):
            self._graphs = {}
        entry = self._graphs.get(key)
        if entry is None:
            flags = (self.w_fresh, self.z_fresh, self.g_fresh, self.ctc_fresh, getattr(self, "pf2_deferred", None),
                     getattr(self, "pf2_fresh", None))
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            host_flags = ("w_fresh", "z_fresh", "g_fresh", "ctc_fresh")
            saved = {k: getattr(self, k) for k in host_flags}
            try:
                # capture_begin / capture_end directly on a side stream: `with torch.cuda.graph(g)` also runs
                # gc.collect() and torch.cuda.empty_cache() on entry, which costs ~0.1 s per capture once the
                # allocator holds gigabytes (measured through the e2e call of config 1: 0.21 -> 0.32 s)
                main = torch.cuda.current_stream(self.dev)
                cap = torch.cuda.Stream(device=self.dev)
                cap.wait_stream(main)
                with torch.cuda.stream(cap):
                    g.capture_begin()
                    try:
                        self.outer_iteration()
                        launched = self._launch_diagnostics() if with_diagnostics else None
                    finally:
                        g.capture_end()
                main.wait_stream(cap)
            except Exception:
                # nothing ran on the device during the failed capture: put the host-side bookkeeping back so that the
                # caller can issue the same iteration eagerly
                for k, v in saved.items():
                    setattr(self, k, v)
                self._graph_failed = True
                raise
            after = (self.w_fresh, self.z_fresh, self.g_fresh, self.ctc_fresh, getattr(self, "pf2_deferred", None),
                     getattr(self, "pf2_fresh", None))
            if flags != after:
                raise RuntimeError("graph capture outside the steady state of the engine")
            entry = self._graphs[key] = (g, launched)
        entry[0].replay()
        return entry[1]
