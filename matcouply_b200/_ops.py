"""Operator-level wrappers: torch CUDA tensors in, C-ABI kernel launches on torch's current stream.

torch is plumbing only (device memory + stream); every computation below is a hand-written sm_100a kernel from
``matcouply_b200/csrc``.  All functions require CUDA tensors and raise otherwise (no CPU fallback).
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._lib import PenaltyDesc, call, dtype_code


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("matcouply_b200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("matcouply_b200 kernels need contiguous tensors")
    return ctypes.c_void_p(t.data_ptr())


def padded_ld(K, dtype):
    """Row stride (elements) of the packed data matrix: rows must be multiples of 16 bytes for TMA."""
    q = 16 // torch.empty((), dtype=dtype).element_size()
    return (K + q - 1) // q * q


class Workspace:
    """Caller-owned scratch buffers handed to the C ABI (which never allocates)."""

    def __init__(self, device, K, R, dtype, unimodal_shape=None):
        lib = _lib.load()
        self.xs_bytes = int(lib.b2_xstream_workspace_bytes(K, R, dtype_code(dtype)))
        self.xs = torch.empty(self.xs_bytes, dtype=torch.uint8, device=device)
        sms = int(lib.b2_device_sm_count())
        self.red_bytes = 8 * max(3 * 4 * sms, 2 * R * R * sms, 4096)
        self.red = torch.empty(self.red_bytes, dtype=torch.uint8, device=device)
        self.uni = None
        self.uni_bytes = 0
        if unimodal_shape is not None:
            self.ensure_unimodal(*unimodal_shape)

    def ensure_unimodal(self, n_groups, R, max_rows):
        need = int(_lib.load().b2_unimodal_workspace_bytes(n_groups, R, max_rows))
        if need > self.uni_bytes:
            self.uni = torch.empty(need, dtype=torch.uint8, device=self.xs.device)
            self.uni_bytes = need


def xstream_y(X, n_rows, K, C, Y, ws, variant=_lib.VARIANT_AUTO, max_ctas=0):
    R = C.shape[1]
    call("b2_xstream_y", _ptr(X), n_rows, K, X.shape[1], _ptr(C), R, _ptr(Y), dtype_code(X.dtype), _ptr(ws.xs),
         ws.xs_bytes, resolve_variant(variant, X.dtype), max_ctas, _stream())


def xstream_z(X, n_rows, K, W, Z, ws, variant=_lib.VARIANT_AUTO, max_ctas=0):
    """W: (n_rows rounded up to 32, z_ldw(R, dtype, variant)) with zero padding (see alloc_w)."""
    R = Z.shape[1]
    call("b2_xstream_z", _ptr(X), n_rows, K, X.shape[1], _ptr(W), W.shape[1], R, _ptr(Z), dtype_code(X.dtype),
         _ptr(ws.xs), ws.xs_bytes, resolve_variant(variant, X.dtype), max_ctas, _stream())


def xstream_fused_supported(K, R, dtype, n_pen):
    """True when the single-read fused pass (csrc/xfused.cu) applies to such a problem."""
    return bool(_lib.load().b2_xstream_fused_local_supported(int(K), int(R), dtype_code(dtype), int(n_pen)))


def fused_schedule(row_offsets, n_ctas):
    """Balanced static schedule of the fused pass: slices sorted by height, each handed to the least loaded CTA
    (longest-processing-time rule).  Returns an int32 array [n_ctas x rounds], -1 padded."""
    import heapq

    sizes = np.diff(np.asarray(row_offsets, dtype=np.int64))
    n_ctas = max(1, min(int(n_ctas), len(sizes)))
    lists = [[] for _ in range(n_ctas)]
    heap = [(0, c) for c in range(n_ctas)]
    for g in np.argsort(-sizes, kind="stable"):
        load, c = heapq.heappop(heap)
        lists[c].append(int(g))
        heapq.heappush(heap, (load + int(sizes[g]), c))
    rounds = max(len(l) for l in lists) if len(sizes) else 0
    sched = np.full((n_ctas, max(rounds, 1)), -1, dtype=np.int32)
    for c, l in enumerate(lists):
        sched[c, :len(l)] = l
    return sched


class FusedWorkspace:
    """Schedule + scratch of the fused pass for one packed data set."""

    def __init__(self, row_offsets, K, R, device):
        lib = _lib.load()
        self.sched_host = fused_schedule(row_offsets, int(lib.b2_device_sm_count()))
        self.n_ctas, self.rounds = self.sched_host.shape
        self.sched = torch.as_tensor(self.sched_host).to(device)
        self.bytes = int(lib.b2_xstream_fused_workspace_bytes(int(K), int(R), self.n_ctas))
        self.buf = torch.empty(self.bytes, dtype=torch.uint8, device=device)


def xstream_fused_local(X, n_rows, K, row_off, n_slices, fws, C, A, rho, Minv, descs, n_pen, n_inner, B, Z, G, BtB):
    R = C.shape[1]
    call("b2_xstream_fused_local", _ptr(X), n_rows, K, X.shape[1], _ptr(row_off), n_slices, _ptr(fws.sched), fws.n_ctas,
         fws.rounds, _ptr(C), _ptr(A), _ptr(rho), _ptr(Minv), descs, n_pen, n_inner, R, _ptr(B), _ptr(Z), _ptr(G),
         _ptr(BtB), dtype_code(X.dtype), _ptr(fws.buf), fws.bytes, _stream())


def slice_gdot(G, C, n_groups, K, R, rhs):
    call("b2_slice_gdot", _ptr(G), _ptr(C), n_groups, K, R, _ptr(rhs), dtype_code(G.dtype), _stream())


def z_ldw(R, dtype, variant=_lib.VARIANT_AUTO):
    return int(_lib.load().b2_xstream_z_ldw(R, dtype_code(dtype), resolve_variant(variant, dtype)))


def alloc_w(n_rows, R, dtype, device, variant=_lib.VARIANT_AUTO):
    """Zero-initialised W buffer in the layout b2_xstream_z expects for this variant."""
    return torch.zeros(((n_rows + 31) // 32 * 32, z_ldw(R, dtype, variant)), dtype=dtype, device=device)


_DEFAULT_VARIANT = {"f64": _lib.VARIANT_DMMA}


def set_default_fp64_variant(variant):
    """Select the fp64 X-stream kernel flavour (FMA pipes or DMMA tensor cores) used for VARIANT_AUTO."""
    _DEFAULT_VARIANT["f64"] = variant


def resolve_variant(variant, dtype):
    if variant != _lib.VARIANT_AUTO:
        return variant
    return _DEFAULT_VARIANT["f64"] if dtype == torch.float64 else _lib.VARIANT_FMA


def sumsq(X, n_rows, K, out, ws):
    call("b2_sumsq", _ptr(X), n_rows, K, X.shape[1], dtype_code(X.dtype), _ptr(out), _ptr(ws.red), ws.red_bytes,
         _stream())


def mask_refill_workspace(n_rows, device):
    """Scratch of b2_mask_refill for n_rows packed rows."""
    return torch.empty(int(_lib.load().b2_mask_refill_workspace_bytes(int(n_rows))), dtype=torch.uint8, device=device)


def mask_refill(X, n_rows, K, row_ptr, miss_col, gor, A, B, C, Y, out, ws):
    """Missing entries of X <- (B o A[gor]) C^T, Y += d C (Y may be None), out[0:2] += (sum d^2, change of ||X||^2)."""
    call("b2_mask_refill", _ptr(X), n_rows, K, X.shape[1], _ptr(row_ptr), _ptr(miss_col), _ptr(gor), _ptr(A), _ptr(B),
         _ptr(C), C.shape[1], _ptr(Y), _ptr(out), dtype_code(X.dtype), _ptr(ws), ws.numel(), _stream())


def gram(M, n, G, ws):
    call("b2_gram", _ptr(M), n, G.shape[0], M.shape[1], _ptr(G), dtype_code(M.dtype), _ptr(ws.red), ws.red_bytes,
         _stream())


def scale_gram(G, A, lhs):
    call("b2_scale_gram", _ptr(G), _ptr(A), A.shape[0], A.shape[1], _ptr(lhs), dtype_code(G.dtype), _stream())


def rho_from_trace(lhs, n_groups, R, scale, rho, rho_max=None):
    call("b2_rho_from_trace", _ptr(lhs), n_groups, R, float(scale), _ptr(rho), _ptr(rho_max), dtype_code(lhs.dtype),
         _stream())


def factor_batch(lhs, n_groups, R, rho, rho_max, n_reg, l2, Minv):
    call("b2_factor_batch", _ptr(lhs), n_groups, R, _ptr(rho), _ptr(rho_max), int(n_reg), float(l2), _ptr(Minv),
         dtype_code(lhs.dtype), _stream())


def slice_cross(B, Y, row_off, n_groups, R, CtC, cross, rhs):
    call("b2_slice_cross", _ptr(B), _ptr(Y), _ptr(row_off), n_groups, R, _ptr(CtC), _ptr(cross), _ptr(rhs),
         dtype_code(B.dtype), _stream())


def rowscale(B, A, group_of_row, n, R, W):
    call("b2_rowscale", _ptr(B), _ptr(A), _ptr(group_of_row), n, R, _ptr(W), W.shape[1], dtype_code(B.dtype),
         _stream())


def make_descs(entries):
    """entries: list of (kind, non_negativity, p0, p1, aux_tensor, dual_tensor) -> ctypes array (host)."""
    arr = (PenaltyDesc * max(len(entries), 1))()
    for i, (kind, nn, p0, p1, aux, dual) in enumerate(entries):
        arr[i].kind = kind
        arr[i].non_negativity = int(bool(nn))
        arr[i].p0 = float(p0)
        arr[i].p1 = float(p1)
        arr[i].aux = aux.data_ptr()
        arr[i].dual = dual.data_ptr()
    return arr


def admm_solve(n, R, rhs, rhs_scale, group_mode, group_of_row, rho, Minv, descs, n_pen, x):
    call("b2_admm_solve", n, R, _ptr(rhs), _ptr(rhs_scale), group_mode, _ptr(group_of_row), _ptr(rho), _ptr(Minv),
         descs, n_pen, _ptr(x), dtype_code(x.dtype), _stream())


def prox_l2ball(aux, dual, row_off, n_groups, R, bound, nn, colsq=None, phase=0):
    """phase 0: whole prox; phase 1 / 2: local column sums of squares -> colsq / scale with the (all-reduced) colsq."""
    call("b2_prox_l2ball", _ptr(aux), _ptr(dual), _ptr(row_off), n_groups, R, float(bound), int(bool(nn)), _ptr(colsq),
         int(phase), dtype_code(aux.dtype), _stream())


def prox_unimodal(aux, dual, row_off, n_groups, R, max_rows, nn, ws, peaks=None):
    ws.ensure_unimodal(n_groups, R, max_rows)
    call("b2_prox_unimodal", _ptr(aux), _ptr(dual), _ptr(row_off), n_groups, R, max_rows, int(bool(nn)), _ptr(peaks),
         dtype_code(aux.dtype), _ptr(ws.uni), ws.uni_bytes, _stream())


def prox_simplex(aux, dual, row_off, n_groups, max_rows, R):
    call("b2_prox_simplex", _ptr(aux), _ptr(dual), _ptr(row_off), n_groups, int(max_rows), R, dtype_code(aux.dtype),
         _stream())


def prox_tv(aux, dual, row_off, n_groups, R, rho, reg_strength, l1_strength):
    """rho: device tensor with one value per group, or a single value shared by all groups."""
    call("b2_prox_tv", _ptr(aux), _ptr(dual), _ptr(row_off), n_groups, R, _ptr(rho), 1 if rho.numel() > 1 else 0,
         float(reg_strength), float(l1_strength), dtype_code(aux.dtype), _stream())


def tv_norm(x, row_off, n_groups, R, out):
    part = torch.empty(max(n_groups, 1), dtype=torch.float64, device=x.device)
    call("b2_tv_norm", _ptr(x), _ptr(row_off), n_groups, R, _ptr(out), _ptr(part), dtype_code(x.dtype), _stream())


def prox_temporal_workspace(n_slices, n_pos, world, device):
    """Scratch of b2_prox_temporal / b2_prox_temporal_serial for n_slices slices of n_pos = J * R entries."""
    need = int(_lib.load().b2_prox_temporal_workspace_bytes(int(n_slices), int(n_pos), int(world)))
    return torch.empty(max(need, 8), dtype=torch.uint8, device=device)


def prox_temporal(aux, dual, n_slices, n_pos, rho, lam, ws, stage=0, has_left=False, has_right=False, xch=None,
                  world=1, rank=0):
    """rho: device tensor with one value per slice, or a single value shared by all slices.  Stage 0 solves the whole
    system; stages 1 / 2 are the two halves of a sharded solve around the all-reduce of `xch` (see the C header)."""
    call("b2_prox_temporal", _ptr(aux), _ptr(dual), int(n_slices), int(n_pos), _ptr(rho), 1 if rho.numel() > 1 else 0,
         float(lam), int(stage), int(bool(has_left)), int(bool(has_right)), _ptr(xch), int(world), int(rank),
         dtype_code(aux.dtype), _ptr(ws), ws.numel(), _stream())


def prox_temporal_serial(aux, dual, n_slices, n_pos, rho, lam, ws):
    call("b2_prox_temporal_serial", _ptr(aux), _ptr(dual), int(n_slices), int(n_pos), _ptr(rho),
         1 if rho.numel() > 1 else 0, float(lam), dtype_code(aux.dtype), _ptr(ws), ws.numel(), _stream())


def temporal_norm(x, n_slices, n_pos, lam, out, part, xch=None, rank=0):
    """out[0] = lam * sum_i ||x_i - x_{i-1}||^2; part: >= n_slices doubles of scratch."""
    call("b2_temporal_norm", _ptr(x), int(n_slices), int(n_pos), float(lam), _ptr(xch), int(rank), _ptr(out),
         _ptr(part), dtype_code(x.dtype), _stream())


def prox_gl2(aux, dual, n_groups, J, R, U, s, rho, tmp):
    call("b2_prox_gl2", _ptr(aux), _ptr(dual), n_groups, J, R, _ptr(U), _ptr(s), _ptr(rho),
         1 if rho.numel() > 1 else 0, _ptr(tmp), dtype_code(aux.dtype), _stream())


def quadform(M, x, n_groups, J, R, out, tmp):
    part = torch.empty(256, dtype=torch.float64, device=x.device)
    call("b2_quadform", _ptr(M), _ptr(x), n_groups, J, R, _ptr(out), _ptr(tmp), _ptr(part), dtype_code(x.dtype),
         _stream())


def pf2_fixed_basis(pd, dual, P, Delta, row_off, n_groups, n, R, rho, num_part, phase):
    call("b2_pf2_fixed_basis", _ptr(pd), _ptr(dual), _ptr(P), _ptr(Delta), _ptr(row_off), n_groups, n, R, _ptr(rho),
         _ptr(num_part), int(phase), dtype_code(dual.dtype), _stream())


def pf2_polar(S, Delta, rho, n_groups, R, Wmat, num_part, Qstore=None, warm=False):
    call("b2_pf2_polar", _ptr(S), _ptr(Delta), _ptr(rho), n_groups, R, _ptr(Wmat), _ptr(num_part), _ptr(Qstore),
         int(bool(warm)), dtype_code(S.dtype), _stream())


def pf2_delta(num_part, rho, n_groups, R, Delta_new, sums, sums_in=None):
    call("b2_pf2_delta", _ptr(num_part), _ptr(rho), n_groups, R, _ptr(Delta_new), _ptr(sums), _ptr(sums_in),
         dtype_code(Delta_new.dtype), _stream())


def pf2_apply(pd, dual, basis, Wmat, Delta_new, group_of_row, n, R):
    call("b2_pf2_apply", _ptr(pd), _ptr(dual), _ptr(basis), _ptr(Wmat), _ptr(Delta_new), _ptr(group_of_row), n, R,
         dtype_code(pd.dtype), _stream())


def reduce_stats(x, y, n, out, ws):
    call("b2_reduce_stats", _ptr(x), _ptr(y), n, _ptr(out), dtype_code(x.dtype), _ptr(ws.red), ws.red_bytes, _stream())


def fit_terms(rhs, cross, A, n_groups, R, out, ws):
    call("b2_fit_terms", _ptr(rhs), _ptr(cross), _ptr(A), n_groups, R, _ptr(out), dtype_code(A.dtype), _ptr(ws.red),
         ws.red_bytes, _stream())


def prox_elementwise(v, out, kind, nn, p0, p1, rho):
    call("b2_prox_elementwise", _ptr(v), _ptr(out), v.numel(), kind, int(bool(nn)), float(p0), float(p1), float(rho),
         dtype_code(v.dtype), _stream())


def microbench_flops(kind, iters):
    """Returns (flops_issued, milliseconds) for one launch of the peak micro-benchmark (CUDA-event timed)."""
    sink = torch.zeros(8, dtype=torch.float64, device="cuda")
    flops = ctypes.c_double(0.0)
    call("b2_microbench_flops", kind, 16, ctypes.byref(flops), _ptr(sink), _stream())  # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    call("b2_microbench_flops", kind, iters, ctypes.byref(flops), _ptr(sink), _stream())
    e1.record()
    torch.cuda.synchronize()
    return flops.value, e0.elapsed_time(e1)


def to_device(a, dtype, device):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device)


def admm_local(n, R, rhs, rhs_scale, group_mode, group_of_row, rho, Minv, descs, n_pen, n_inner, x, w_out=None,
               row_off=None, n_groups=0, BtB_out=None):
    call("b2_admm_local", n, R, _ptr(rhs), _ptr(rhs_scale), group_mode, _ptr(group_of_row), _ptr(row_off), n_groups,
         _ptr(rho), _ptr(Minv), descs, n_pen, n_inner, _ptr(x), _ptr(w_out),
         0 if w_out is None else w_out.shape[1], _ptr(BtB_out), dtype_code(x.dtype), _stream())


def pf2_rowpass(row_off, n_groups, R, Y, A, rho, Minv, descs, n_pen, deferred, Wmat, Delta, x, w_out, S_out,
                BtB_out=None, comp_stats_part=None):
    call("b2_pf2_rowpass", _ptr(row_off), n_groups, R, _ptr(Y), _ptr(A), _ptr(rho), _ptr(Minv), descs, n_pen,
         int(deferred), _ptr(Wmat), _ptr(Delta), _ptr(x), _ptr(w_out), 0 if w_out is None else w_out.shape[1],
         _ptr(S_out), _ptr(BtB_out), _ptr(comp_stats_part), dtype_code(Y.dtype), _stream())


def pf2_rowpass_fused_stats_supported(R, dtype, n_pen, companion_kind, deferred):
    """True when b2_pf2_rowpass serves `comp_stats_part` (and the one-array companion on the last pass) for such a call."""
    return bool(_lib.load().b2_pf2_rowpass_fused_stats_supported(int(R), dtype_code(dtype), int(n_pen),
                                                                   int(companion_kind), int(deferred)))


def group_stats_sum(part, n_groups, out):
    """out[0:3] = sum over groups of the per-slice partials part[3 g + 0:3] (fixed order)."""
    call("b2_group_stats_sum", _ptr(part), int(n_groups), _ptr(out), _stream())


def pf2_gap(V, x, row_off, n_groups, R, Wmat, Delta, out, part):
    """out[0:3] = (sum ||V W Delta - x||^2, sum x^2, sum |x|); part: scratch of >= 3 * n_groups doubles."""
    call("b2_pf2_gap", _ptr(V), _ptr(x), _ptr(row_off), n_groups, R, _ptr(Wmat), _ptr(Delta), _ptr(out),
         dtype_code(V.dtype), _ptr(part), part.numel() * part.element_size(), _stream())


def slice_gram(B, row_off, n_groups, R, BtB):
    call("b2_slice_gram", _ptr(B), _ptr(row_off), n_groups, R, _ptr(BtB), dtype_code(B.dtype), _stream())


def slice_coldot(B, Y, row_off, n_groups, R, rhs):
    call("b2_slice_coldot", _ptr(B), _ptr(Y), _ptr(row_off), n_groups, R, _ptr(rhs), dtype_code(B.dtype), _stream())


def weighted_gram_sum(BtB, A, n_groups, R, out):
    call("b2_weighted_gram_sum", _ptr(BtB), _ptr(A), n_groups, R, _ptr(out), dtype_code(BtB.dtype), _stream())


def hadamard_bcast(BtB, CtC, n_groups, R, cross):
    call("b2_hadamard_bcast", _ptr(BtB), _ptr(CtC), n_groups, R, _ptr(cross), dtype_code(BtB.dtype), _stream())


def mt19937_uniform(random_state, n, device):
    """The next ``n`` doubles of ``random_state.uniform(size=n)`` (== ``random_sample``), generated ON THE DEVICE with
    identical bits; ``random_state`` (a legacy ``np.random.RandomState``) is advanced exactly as if it had drawn them."""
    name, key, pos, has_gauss, cached = random_state.get_state(legacy=True)
    if name != "MT19937":
        raise TypeError("device draws need a MT19937 RandomState")
    st = np.empty(625, dtype=np.uint32)
    st[:624] = key
    st[624] = pos
    n_chunks = int(os.environ.get("B2_MT_CHUNKS", "1"))  # opt-in until measured on the GPU (DESIGN.md §7)
    if n_chunks > 1 and int(n) >= _MT_CHUNK_MIN_DRAWS:
        bounds, starts, final = mt_chunk_plan(st, int(n), n_chunks)
        out = _mt19937_uniform_chunked(bounds, starts, device)
        random_state.set_state(("MT19937", final[:624].copy(), int(final[624]), has_gauss, cached))
        return out
    # a side stream: the generator kernel (one CTA) overlaps whatever the caller's stream is doing (cmf_aoadmm: the
    # H2D copy of the data), and reading back the advanced state only waits for the generator
    main = torch.cuda.current_stream(device)
    side = _side_stream(device)
    with torch.cuda.stream(side):
        dstate = torch.from_numpy(st.view(np.int32)).to(device)
        out = torch.empty(int(n), dtype=torch.float64, device=device)
        call("b2_mt19937_uniform", _ptr(dstate), _ptr(out), int(n), _stream())
        new = dstate.cpu().numpy().view(np.uint32)
    main.wait_stream(side)
    out.record_stream(main)
    random_state.set_state(("MT19937", new[:624].copy(), int(new[624]), has_gauss, cached))
    return out


_MT_CHUNK_MIN_DRAWS = 1 << 20


def mt_chunk_plan(state, n, n_chunks):
    """Cut the next ``n`` doubles of the MT19937 stream whose 625-word state is ``state`` into ``n_chunks`` consecutive
    chunks: returns (bounds [n_chunks + 1], start state of every chunk [n_chunks x 625], state after all n draws),
    each start obtained from the previous one with the host jump-ahead (``b2_mt19937_jump_host``, 2 ms per jump)."""
    bounds = np.linspace(0, int(n), int(n_chunks) + 1).astype(np.int64)
    cur = np.array(state, dtype=np.uint32)
    starts = np.empty((int(n_chunks), 625), dtype=np.uint32)
    for c in range(int(n_chunks)):
        starts[c] = cur
        call("b2_mt19937_jump_host", cur.ctypes.data, 2 * int(bounds[c + 1] - bounds[c]))
    return bounds, starts, cur


def _mt19937_uniform_chunked(bounds, starts, device):
    """The chunks of `mt_chunk_plan` generated concurrently: the sequential one-CTA generator kernel of csrc/rng.cu once
    per chunk, every launch on its own stream and from its own jumped start state (same bits as one long walk)."""
    n_chunks, n = len(starts), int(bounds[-1])
    main = torch.cuda.current_stream(device)
    streams = [_side_stream(device, c) for c in range(n_chunks)]
    with torch.cuda.stream(streams[0]):
        dstates = torch.from_numpy(np.ascontiguousarray(starts).view(np.int32)).to(device)
        out = torch.empty(n, dtype=torch.float64, device=device)
    for c, side in enumerate(streams):
        if c:
            side.wait_stream(streams[0])  # the allocation and the state upload belong to the first side stream
        lo, cnt = int(bounds[c]), int(bounds[c + 1] - bounds[c])
        if cnt:
            with torch.cuda.stream(side):
                call("b2_mt19937_uniform", _ptr(dstates[c]), ctypes.c_void_p(out.data_ptr() + 8 * lo), cnt, _stream())
        main.wait_stream(side)
        out.record_stream(side)
        dstates.record_stream(side)
    out.record_stream(main)
    return out


def mt19937_skip(random_state, n):
    """Advance ``random_state`` (legacy MT19937 ``np.random.RandomState``) exactly as ``random_state.uniform(size=n)``
    would, without drawing: host-side jump-ahead (``b2_mt19937_jump_host``), cost independent of ``n``."""
    name, key, pos, has_gauss, cached = random_state.get_state(legacy=True)
    if name != "MT19937":
        raise TypeError("skipping needs a MT19937 RandomState")
    st = np.empty(625, dtype=np.uint32)
    st[:624] = key
    st[624] = pos
    call("b2_mt19937_jump_host", st.ctypes.data, 2 * int(n))
    random_state.set_state(("MT19937", st[:624].copy(), int(st[624]), has_gauss, cached))


_SIDE_STREAMS = {}


def _side_stream(device, which=0):
    dev = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    key = dev if which == 0 else (dev, which)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]
