"""Masked fitting at the sizes it runs at (DESIGN.md §10).

1. ``b2_mask_refill`` against NumPy float64 (``masked_oracle.refill_reference``) at row counts derived from the SM
   count: under one wave, past 256 blocks (the strided loop of the finish kernel) and several waves (the grid-stride
   loop); K = 512, 1030, 2048; rows whose missing count sits on the edges of the 32-entry chunks and fully missing rows
   (up to 64 chunks); R = 1 .. 32; fp64 and fp32, with and without ``Y``; and the host-side argument checks.
2. The engine's bookkeeping at full config-1 size and at the config-2 slice shape, against dense float64 products on
   the device (cuBLAS): observed entries untouched, missing entries equal to the model, ``Y = F C``, the tracked
   ``‖F‖²`` and the loss identity behind ``rec_errors``.
3. Masked trajectories at the baseline widths of configs 1-4 (fewer slices) against ``ao_admm_masked``.
4. The public API's remaining masked edges: frozen modes, ``inner_tol``, constant feasibility penalty, planted
   matrix completion run to the stopping rule, and a 4-rank run in which one rank holds no slice.
"""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from masked_oracle import ao_admm_masked, observed_error, refill_reference  # noqa: E402


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


# ---------------------------------------------------------------------------------------------------------------
# 1. the refill kernel against NumPy float64
# ---------------------------------------------------------------------------------------------------------------
ROWS_PER_BLOCK = 8  # one row per warp, 8 warps per block (csrc/mask.cu)
SENTINEL = -1234.5  # written into the padding columns [K, ldx) before a launch


def _blocks_per_wave():
    from matcouply_b200 import _lib

    return 4 * int(_lib.load().b2_device_sm_count())


def _n_rows(case):
    """Row count of a case, from the grid of b2_mask_refill: min(ceil(N / 8), 4 x SMs) blocks."""
    cap = _blocks_per_wave()
    if case == "one_wave":  # <= 256 blocks, every warp takes one row
        return ROWS_PER_BLOCK * min(200, cap) - 5
    if case == "past_256_blocks":  # more than 256 partials for the finish kernel, still one wave
        if cap <= 257:
            pytest.skip(f"{cap} blocks per wave: no row count lies between 256 blocks and one wave")
        return ROWS_PER_BLOCK * (256 + (cap - 256) // 2) + 3
    if case == "several_waves":  # every warp takes at least 4 rows
        return max(40000, 4 * ROWS_PER_BLOCK * cap + 77)
    raise KeyError(case)


def _refill_problem(N, K, R, dtype, seed):
    """Host CSR of the missing entries and the factors; the data X lives on the device.

    Every row set of `special` is placed at the start, in the middle and at the end of the rows, and past the first
    wave: missing counts 1, 31, 32, 33, 63, 64 (the edges of the 32-entry chunks), K (a fully missing row), 0, and
    holes in column 0 only, in column K-1 only and in both.  The other rows miss 5 % of their entries at random.
    Slices of 0 and 1 rows sit among the ragged slices."""
    rs = np.random.RandomState(seed)
    miss = np.zeros((N, K), dtype=bool)
    for r0 in range(0, N, 1 << 14):
        r1 = min(N, r0 + (1 << 14))
        miss[r0:r1] = rs.random_sample((r1 - r0, K)) < 0.05
    special = []
    for c in (1, 31, 32, 33, 63, 64, K):
        row = np.zeros(K, dtype=bool)
        row[rs.choice(K, size=min(c, K), replace=False)] = True
        special.append(row)
    special.append(np.zeros(K, dtype=bool))
    for cols in ([0], [K - 1], [0, K - 1]):
        row = np.zeros(K, dtype=bool)
        row[cols] = True
        special.append(row)
    special = np.array(special)
    for at in sorted({0, N // 2, max(0, N - len(special)), min(N - len(special), _blocks_per_wave() * ROWS_PER_BLOCK + 9)}):
        if at >= 0:
            n = min(len(special), N - at)
            miss[at:at + n] = special[:n]
    sizes = rs.randint(2, 300, size=N + 8)
    sizes[[1, 4]] = 0
    sizes[[2, 6]] = 1
    gor = np.repeat(np.arange(len(sizes)), sizes)[:N].astype(np.int32)
    n_slices = int(gor[-1]) + 1 if N else 0
    row_ptr = np.concatenate([[0], np.cumsum(miss.sum(axis=1))]).astype(np.int64)
    col = np.nonzero(miss)[1].astype(np.int32)
    A = rs.uniform(size=(max(n_slices, 1), R))
    B, C, Y = rs.standard_normal((N, R)), rs.standard_normal((K, R)), rs.standard_normal((N, R))
    if dtype == torch.float32:
        A, B, C, Y = (a.astype(np.float32).astype(np.float64) for a in (A, B, C, Y))
    return row_ptr, col, gor, A, B, C, Y


def _ulp32(v):
    return np.spacing(np.abs(v.astype(np.float32))).astype(np.float64)


def _check_refill(N, K, R, dtype, seed=0):
    from matcouply_b200 import _ops

    dev = torch.device("cuda")
    row_ptr, col, gor, A, B, C, Y = _refill_problem(N, K, R, dtype, seed)
    ld = _ops.padded_ld(K, dtype)
    gen = torch.Generator(device=dev).manual_seed(seed)
    X0 = torch.randn((N, ld), dtype=dtype, device=dev, generator=gen)
    X0[:, K:] = SENTINEL
    rp_d, col_d = torch.as_tensor(row_ptr, device=dev), torch.as_tensor(col, device=dev)
    flat = torch.repeat_interleave(torch.arange(N, device=dev), torch.diff(rp_d)) * ld + col_d.to(torch.int64)
    x_old = X0.view(-1)[flat].double().cpu().numpy()
    ref = refill_reference(x_old, row_ptr, col, gor, A, B, C, Y=Y, dtype=np.float32 if dtype == torch.float32
                           else np.float64)
    t = lambda a: torch.as_tensor(a, dtype=dtype, device=dev).contiguous()  # noqa: E731
    Ad, Bd, Cd, Y0 = t(A), t(B), t(C), t(Y)
    gor_d = torch.as_tensor(gor, device=dev)
    ws = _ops.mask_refill_workspace(N, dev)
    start = (3.25, -1.5)

    def launch(use_y):
        X, Yd = X0.clone(), Y0.clone()
        out = torch.tensor(start, dtype=torch.float64, device=dev)
        _ops.mask_refill(X, N, K, rp_d, col_d, gor_d, Ad, Bd, Cd, Yd if use_y else None, out, ws)
        return X, Yd, out

    X, Yd, out = launch(True)
    # missing entries: the model value
    got = X.view(-1)[flat].double().cpu().numpy()
    if dtype == torch.float64:
        bound = 1e-13 * ref["scale"]
        assert np.all(np.abs(got - ref["xhat"]) <= bound), np.max(np.abs(got - ref["xhat"]) - bound)
    else:  # one fp32 ulp of the fp64 value rounded to fp32
        bound = _ulp32(ref["xhat"]) + 1e-13 * ref["scale"]
        assert np.all(np.abs(got - ref["new"]) <= bound), np.max(np.abs(got - ref["new"]) - bound)
    # observed entries and padding: bit-unchanged
    Xc = X.clone()
    Xc.view(-1)[flat] = X0.view(-1)[flat]
    ibits = torch.int64 if dtype == torch.float64 else torch.int32
    assert torch.equal(Xc.view(ibits), X0.view(ibits))
    del Xc
    # Y += sum_k d C[k]
    Yg = Yd.double().cpu().numpy()
    ybound = 1e-13 * ref["yscale"] + (0 if dtype == torch.float64 else _ulp32(ref["Y"]))
    assert np.all(np.abs(Yg - ref["Y"]) <= ybound), np.max(np.abs(Yg - ref["Y"]) - ybound)
    # out accumulates onto its start values
    og = out.cpu().numpy()
    s0, s1 = ref["sums"]
    assert abs((og[0] - start[0]) - s0) <= 1e-12 * s0 + 1e-12, (og[0] - start[0], s0)
    assert abs((og[1] - start[1]) - s1) <= 1e-12 * ref["sums_scale"] + 1e-12, (og[1] - start[1], s1)
    # the same input gives the same bits; without Y the same X and out, and Y is not written
    X2, Y2, out2 = launch(True)
    assert torch.equal(X2.view(ibits), X.view(ibits)) and torch.equal(Y2.view(ibits), Yd.view(ibits))
    assert torch.equal(out2, out)
    X3, Y3, out3 = launch(False)
    assert torch.equal(X3.view(ibits), X.view(ibits)) and torch.equal(out3, out)
    assert torch.equal(Y3.view(ibits), Y0.view(ibits))
    return int(row_ptr[-1])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("K", [512, 1030, 2048])
@pytest.mark.parametrize("rows", ["one_wave", "past_256_blocks", "several_waves"])
def test_refill_kernel_at_wave_and_block_edges(rows, K, dtype):
    """The grid-stride loop over rows, the finish kernel's loop over more than 256 block partials and rows of up to
    64 chunks of missing entries, against NumPy float64."""
    R = {"one_wave": 16, "past_256_blocks": 20, "several_waves": 32}[rows]
    N = _n_rows(rows)
    n_missing = _check_refill(N, K, R, dtype, seed=K + N)
    print(f"[refill] {rows}: N={N} K={K} R={R} {dtype}: {n_missing} missing entries")


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("R", [1, 2, 8, 15, 16, 17, 20, 31, 32])
def test_refill_kernel_ranks(R, dtype):
    """Every lane count around the half-warp boundary, past 256 blocks, K = 1030 (padded in fp32, not in fp64)."""
    _check_refill(_n_rows("past_256_blocks"), 1030, R, dtype, seed=R)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("N", [0, 1, 2])
def test_refill_kernel_tiny_calls(N, dtype):
    """No row (nothing launched, out unchanged) and one or two rows (one partially filled block)."""
    from matcouply_b200 import _ops

    if N:
        _check_refill(N, 512, 16, dtype, seed=N)
        return
    dev = torch.device("cuda")
    X = torch.zeros((0, 512), dtype=dtype, device=dev)
    out = torch.tensor([1.0, 2.0], dtype=torch.float64, device=dev)
    e = lambda *s, dt=dtype: torch.zeros(s, dtype=dt, device=dev)  # noqa: E731
    _ops.mask_refill(X, 0, 512, e(1, dt=torch.int64), e(0, dt=torch.int32), e(0, dt=torch.int32), e(1, 4), e(0, 4),
                     e(512, 4), e(0, 4), out, _ops.mask_refill_workspace(0, dev))
    assert out.tolist() == [1.0, 2.0]


def test_refill_rejects_bad_arguments():
    """Host-side checks before any launch: rank outside 1..32, ldx < K, a workspace one block too small."""
    from matcouply_b200 import _ops

    dev = torch.device("cuda")
    N, K, R = 3000, 40, 4
    row_ptr, col, gor, A, B, C, Y = _refill_problem(N, K, R, torch.float64, 1)
    t = lambda a: torch.as_tensor(a, device=dev).contiguous()  # noqa: E731
    X = torch.randn((N, K), dtype=torch.float64, device=dev)
    X0 = X.clone()
    out = torch.tensor([5.0, 6.0], dtype=torch.float64, device=dev)
    ws = _ops.mask_refill_workspace(N, dev)
    args = lambda Cm, Kc=K, w=ws: (X, N, Kc, t(row_ptr), t(col), t(gor), t(A), t(B), Cm, None, out, w)  # noqa: E731
    with pytest.raises(RuntimeError, match=r"b2_mask_refill: rank 0 outside 1\.\.32"):
        _ops.mask_refill(*args(torch.zeros((K, 0), dtype=torch.float64, device=dev)))
    with pytest.raises(RuntimeError, match=r"b2_mask_refill: rank 33 outside 1\.\.32"):
        _ops.mask_refill(*args(torch.zeros((K, 33), dtype=torch.float64, device=dev)))
    with pytest.raises(RuntimeError, match=r"b2_mask_refill: bad shape \(n_rows 3000, K 41, ldx 40\)"):
        _ops.mask_refill(*args(t(C), Kc=K + 1))
    with pytest.raises(RuntimeError, match="b2_mask_refill workspace too small"):
        _ops.mask_refill(*args(t(C), w=ws[:ws.numel() - 16]))  # 2 doubles per block
    torch.cuda.synchronize()
    assert torch.equal(X, X0) and out.tolist() == [5.0, 6.0]  # nothing was launched
    _ops.mask_refill(*args(t(C)))  # the exact size is enough
    assert not torch.equal(X, X0) and out.tolist() != [5.0, 6.0]


# ---------------------------------------------------------------------------------------------------------------
# 2. engine bookkeeping at full config-1 size and at the config-2 slice shape
# ---------------------------------------------------------------------------------------------------------------
ENGINE_CHECKS = (0, 1, 2, 5, 50)  # after prepare() and after these outer iterations
CHUNK_ROWS = 1 << 16


def _engine_case(shape, dtype, pattern):
    import bench

    from matcouply_b200._engine import AOADMMEngine, pack_mask_device

    dev = torch.device("cuda")
    cfg = dict(bench.CONFIGS["c1"]) if shape == "c1" else dict(bench.CONFIGS["c2"], I=1024)
    packed = bench.gen_device_data(cfg, bench.slice_sizes(cfg), 0, cfg["I"], dtype, dev)
    gen = torch.Generator(device=dev).manual_seed(17)
    if pattern == "rows":
        observed = (torch.rand(packed.N, device=dev, generator=gen) >= 0.1)[:, None].expand(packed.N, packed.K)
        observed = observed.contiguous()
    else:
        observed = torch.rand((packed.N, packed.K), device=dev, generator=gen) >= 0.1
    regs = bench.make_regs(cfg["kw"])
    X0 = packed.X.clone()
    eng = AOADMMEngine(packed, cfg["R"], regs, mask=pack_mask_device(observed, packed))
    eng.load_state_device(seed=1)
    return eng, regs, X0, observed


def _dense_checks(eng, X0, observed):
    """(a) observed entries and padding bit-equal to X0; (b) worst excess of the missing entries over their bound;
    (c) ||Y - F C||^2 and ||F C||^2; (d) sum F^2; (e) the dense observed SSE and ||M o X||^2.  Chunks of rows,
    float64 cuBLAS products."""
    X, K, R = eng.p.X, eng.K, eng.R
    A, B, C = (eng.modes[m].x.double() for m in range(3))
    ibits = torch.int64 if X.dtype == torch.float64 else torch.int32
    same, worst = True, 0.0
    y_err = y_ref = f_sq = sse = obs_sq = 0.0
    for r0 in range(0, eng.N, CHUNK_ROWS):
        r1 = min(eng.N, r0 + CHUNK_ROWS)
        F, F0, obs = X[r0:r1], X0[r0:r1], observed[r0:r1]
        same &= torch.equal(F[:, K:].view(ibits), F0[:, K:].view(ibits))
        same &= torch.equal(torch.where(obs, F[:, :K], 0).view(ibits), torch.where(obs, F0[:, :K], 0).view(ibits))
        W = B[r0:r1] * A[eng.gor[r0:r1].long()]
        Xh = W @ C.T
        Fd = F[:, :K].double()
        if X.dtype == torch.float64:
            bound = 1e-12 * (W.abs() @ C.abs().T)
        else:
            x32 = Xh.float()
            bound = (torch.nextafter(x32.abs(), torch.tensor(float("inf"), device=X.device)) - x32.abs()).double() \
                + 1e-12 * (W.abs() @ C.abs().T)
        worst = max(worst, float(torch.where(obs, -1.0, (Fd - Xh).abs() - bound).max()))
        if not eng.fused_x1:
            Yr = Fd @ C
            y_err += float(((eng.Y[r0:r1].double() - Yr) ** 2).sum())
            y_ref += float((Yr ** 2).sum())
        f_sq += float((Fd ** 2).sum())
        sse += float(torch.where(obs, Fd - Xh, 0.0).pow(2).sum())
        obs_sq += float(torch.where(obs, Fd, 0.0).pow(2).sum())
    return same, worst, (y_err, y_ref), f_sq, sse, obs_sq


@pytest.mark.parametrize("shape,dtype,pattern", [
    ("c1", torch.float64, "random"), ("c1", torch.float64, "rows"),
    ("c1", torch.float32, "random"), ("c1", torch.float32, "rows"),
    ("c2_slices", torch.float64, "random"), ("c2_slices", torch.float64, "rows"),
], ids=["c1-f64-random", "c1-f64-rows", "c1-f32-random", "c1-f32-rows", "c2slices-f64-random", "c2slices-f64-rows"])
def test_engine_bookkeeping_at_full_size(shape, dtype, pattern):
    """Config 1 at full size (4096 x 256 x 512, R = 16) and the config-2 slice shape (1024 ragged slices x 1024,
    R = 20, PARAFAC2 + L1), 10 % of the entries or 10 % of whole rows missing, over 50 outer iterations."""
    from matcouply_b200.decomposition import _loss

    eng, regs, X0, observed = _engine_case(shape, dtype, pattern)
    f64 = dtype == torch.float64
    assert not eng.fused_x1  # the two-pass schedule: the refill corrects the cached Y
    eng.prepare()
    diag = eng.diagnostics()
    report = []
    for it in range(max(ENGINE_CHECKS) + 1):
        if it:
            eng.outer_iteration()
            diag = eng.diagnostics()
        if it not in ENGINE_CHECKS:
            continue
        same, worst, (y_err, y_ref), f_sq, sse, obs_sq = _dense_checks(eng, X0, observed)
        assert same, f"observed entries or padding changed after {it} iterations"
        assert worst <= 0, (it, worst)
        assert np.sqrt(y_err / y_ref) < (1e-12 if f64 else 1e-5), (it, np.sqrt(y_err / y_ref))
        msum = float(eng.msum[1])
        assert abs(msum - f_sq) <= 1e-12 * f_sq, (it, msum, f_sq)
        assert abs(eng.normX_sq - obs_sq) <= 1e-12 * obs_sq
        rec, _ = _loss(diag, eng.normX_sq, [0, 0, 0], regs)
        d = abs(rec ** 2 - sse / obs_sq)
        assert d <= (1e-12 if f64 else 1e-5), (it, rec ** 2, sse / obs_sq)
        report.append((it, f"{d:.1e}", f"{np.sqrt(y_err / y_ref):.1e}", f"{abs(msum - f_sq) / f_sq:.1e}"))
    print(f"[masked engine] {shape} {dtype} {pattern}: N={eng.N} missing={eng.mask.n_missing} "
          f"(it, |rel^2 - dense|, |Y - FC|/|FC|, |msum - sum F^2|/sum F^2) = {report}")


# ---------------------------------------------------------------------------------------------------------------
# 3. masked trajectories at the baseline widths
# ---------------------------------------------------------------------------------------------------------------
TWIN_SLICES = {"c1": 32, "c2": 16, "c3": 8, "c4": 12}
TWIN_ITERS = {"c1": 50, "c2": 50, "c3": 50, "c4": 50}
CHECKPOINTS = (1, 2, 5, 10, 20, 35, 50)


def masked_twin(name, dtype=np.float64):
    """The exact K, J range, R and penalties of a config with fewer slices (bench.py's host sample), 10 % of the
    entries missing at random, a whole row missing in every fourth slice and one whole column missing everywhere."""
    import bench

    cfg = dict(bench.CONFIGS[name])
    cfg["I"] = TWIN_SLICES[name]
    X = bench.gen_host_sample(cfg, bench.slice_sizes(cfg), cfg["I"])
    rs = np.random.RandomState(11)
    M = [rs.uniform(size=x.shape) >= 0.1 for x in X]
    col = rs.randint(cfg["K"])
    for i, m in enumerate(M):
        m[:, col] = False
        if i % 4 == 0:
            m[rs.randint(m.shape[0])] = False
    X = [np.where(m, x, np.nan).astype(dtype) for x, m in zip(X, M)]  # missing values are never read
    return cfg, X, M


class _Checkpoints(list):
    """`trajectory` sink of the oracle that keeps the factors of the checkpoint iterations only."""

    def __init__(self, keep):
        super().__init__()
        self.keep, self.n = set(keep), 0

    def append(self, snap):
        self.n += 1
        if self.n in self.keep:
            super().append((self.n, snap["A"], np.concatenate(snap["B_is"], 0), snap["C"]))


_ORACLE = {}


def masked_oracle_run(key, X, M, R, kw, n_iter, keep):
    """(checkpoint factors, losses, rec_errors) of the masked oracle; one run per case."""
    if key not in _ORACLE:
        traj = _Checkpoints(keep)
        o = ao_admm_masked([np.asarray(x, dtype=np.float64) for x in X], R, M, n_iter_max=n_iter, tol=None,
                           absolute_tol=None, random_state=0, trajectory=traj, **kw)
        _ORACLE[key] = (list(traj), np.asarray(o["regularized_loss"]), np.asarray(o["rec_errors"]))
    return _ORACLE[key]


def _trajectory_parity(key, X, M, R, kw, n_iter, **run_kw):
    from matcouply_b200 import cmf_aoadmm

    keep = [k for k in CHECKPOINTS if k <= n_iter]
    traj, losses, recs = masked_oracle_run(key, X, M, R, kw, n_iter, keep)
    worst = 0.0
    for k, A_o, B_o, C_o in traj:
        (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, mask=M, n_iter_max=k, tol=None, absolute_tol=None, random_state=0,
                                             return_errors=True, **kw, **run_kw)
        errs = (rel(A, A_o), rel(np.concatenate(B_is, 0), B_o), rel(C, C_o))
        worst = max(worst, *errs)
        assert max(errs) < 1e-8, (key, k, errs)
        np.testing.assert_allclose(diag.rec_errors, recs[:k + 1], rtol=1e-8)
        np.testing.assert_allclose(diag.regularized_loss, losses[:k + 1], rtol=1e-8)
    print(f"[masked width parity] {key}: worst relative factor difference over {keep} = {worst:.3e}")
    return worst


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_masked_trajectory_at_baseline_width(name):
    cfg, X, M = masked_twin(name)
    _trajectory_parity(name, X, M, cfg["R"], cfg["kw"], TWIN_ITERS[name])


def test_masked_config1_graph_replay_equals_eager_at_width(monkeypatch):
    """c1 twin, R = 16: the engine's own launch policy replays a captured graph from the third iteration on; 50
    iterations of it are bit-identical to 50 eager iterations."""
    from matcouply_b200 import _engine, cmf_aoadmm

    cfg, X, M = masked_twin("c1")
    replays = []
    real = _engine.AOADMMEngine.graph_iteration
    monkeypatch.setattr(_engine.AOADMMEngine, "graph_iteration",
                        lambda self, d: (replays.append(1), real(self, d))[1])
    runs = [cmf_aoadmm(X, cfg["R"], mask=M, n_iter_max=50, tol=None, absolute_tol=None, random_state=0,
                       return_errors=True, use_cuda_graph=g, **cfg["kw"]) for g in (None, False)]
    assert len(replays) == 48
    (_, fa), da = runs[0]
    (_, fb), db = runs[1]
    np.testing.assert_array_equal(fa[0], fb[0])
    np.testing.assert_array_equal(fa[2], fb[2])
    np.testing.assert_array_equal(np.concatenate(fa[1], 0), np.concatenate(fb[1], 0))
    assert da.rec_errors == db.rec_errors and da.regularized_loss == db.regularized_loss


def test_masked_config1_single_read_pass_at_width(monkeypatch):
    """c1 twin at R = 8 on the single-read fused pass (forced on), where the refill gets no Y."""
    from matcouply_b200 import _engine, _ops
    from matcouply_b200 import penalties as P

    cfg, X, M = masked_twin("c1")
    ys = set()
    real = _ops.mask_refill
    monkeypatch.setattr(_ops, "mask_refill", lambda *a: (ys.add(a[9] is None), real(*a))[1])
    monkeypatch.setitem(_engine.FUSION_DEFAULTS, "x1", True)
    packed = _engine.PackedMatrices.from_list([np.nan_to_num(x) for x in X], torch.float64, torch.device("cuda"))
    assert _engine.AOADMMEngine(packed, 8, [[P.NonNegativity()] for _ in range(3)]).fused_x1
    _trajectory_parity("c1_r8_fused", X, M, 8, cfg["kw"], 50, use_cuda_graph=False)
    assert ys == {True}


def test_masked_fp32_config3_at_baseline_width():
    """c3 in fp32 against the fp64 masked oracle on the fp32-rounded inputs, at the tolerances of the unmasked
    width test (factors within 2e-2 over the first 20 iterations, the loss within 1e-3)."""
    from matcouply_b200 import cmf_aoadmm

    cfg, X32, M = masked_twin("c3", np.float32)
    n = TWIN_ITERS["c3"]
    traj, losses, _ = masked_oracle_run("c3_f32_inputs", X32, M, cfg["R"], cfg["kw"], n, (5, n))
    for k, A_o, B_o, C_o in traj:
        (_, (A, B_is, C)), diag = cmf_aoadmm(X32, cfg["R"], mask=M, n_iter_max=k, tol=None, absolute_tol=None,
                                             random_state=0, return_errors=True, **cfg["kw"])
        errs = (rel(A, A_o), rel(np.concatenate(B_is, 0), B_o), rel(C, C_o))
        assert max(errs) < 2e-2, (k, errs)
    loss_err = abs(diag.regularized_loss[-1] - losses[-1]) / losses[-1]
    assert loss_err < 1e-3, loss_err
    assert np.all(np.isfinite(diag.regularized_loss))


@pytest.mark.parametrize("name", ["c1", "c2"])
def test_masked_stopping_rule_at_baseline_width(name):
    """Run to the stopping rule, loosened so that it fires (c1 after 43 iterations, c2 after 4): the same stopping
    iteration, message and losses as the oracle."""
    from matcouply_b200 import cmf_aoadmm

    cfg, X, M = masked_twin(name)
    loose = dict(n_iter_max=60, tol=1e-2, feasibility_tol=1.0) if name == "c1" else \
        dict(n_iter_max=30, tol=2e-3, feasibility_tol=0.3)
    kw = dict(cfg["kw"], random_state=0, **loose)
    o = ao_admm_masked(X, cfg["R"], M, **kw)
    assert o["n_iter"] < kw["n_iter_max"]
    _, diag = cmf_aoadmm(X, cfg["R"], mask=M, return_errors=True, **kw)
    assert diag.n_iter == o["n_iter"] and diag.message == o["message"], (diag.n_iter, o["n_iter"], diag.message)
    assert str(diag.satisfied_stopping_condition) == str(o["satisfied_stopping_condition"])
    np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"], rtol=1e-8)


# ---------------------------------------------------------------------------------------------------------------
# 4. the public API's remaining masked edges
# ---------------------------------------------------------------------------------------------------------------
def _small_problem(seed, Js, K, R, noise=0.1, frac=0.2):
    """Non-negative rank-R ragged data with a random mask (True = observed), NaN at the missing positions."""
    rs = np.random.RandomState(seed)
    A, C = rs.uniform(0.1, 1.1, size=(len(Js), R)), rs.uniform(size=(K, R))
    X = [(rs.uniform(size=(J, R)) * A[i]) @ C.T + noise * rs.standard_normal((J, K)) for i, J in enumerate(Js)]
    M = [rs.uniform(size=x.shape) >= frac for x in X]
    return [np.where(m, x, np.nan) for x, m in zip(X, M)], M


@pytest.mark.parametrize("option", ["update_A", "update_B_is", "inner_tol", "constant_feasibility_penalty"])
def test_masked_api_options_match_oracle(option):
    X, M = _small_problem(21, np.random.RandomState(3).randint(15, 35, size=8), 24, 4)
    kw = dict(non_negative=True, l1_penalty={2: 0.05})
    kw.update({"update_A": dict(update_A=False), "update_B_is": dict(update_B_is=False),
               "inner_tol": dict(inner_tol=1e-3), "constant_feasibility_penalty":
               dict(constant_feasibility_penalty=True)}[option])
    _trajectory_parity(f"api_{option}", X, M, 4, kw, 35)


def test_masked_planted_completion_loss_identity_to_the_stopping_rule():
    """Noise-free rank-3 data with 20 % missing and no penalty, fitted to the stopping rule (the loss below 1e-12, an
    observed error near 1e-6): the observed error reported through the engine's identity stays within 1e-12
    (squared, relative) of the dense one at every checked iteration, all the way down."""
    from matcouply_b200 import cmf_aoadmm

    rs = np.random.RandomState(3)
    Js, K, R = rs.randint(20, 40, size=10), 25, 3
    A, C = rs.uniform(0.5, 1.5, (10, R)), rs.uniform(size=(K, R))
    X = [(rs.uniform(size=(J, R)) * A[i]) @ C.T for i, J in enumerate(Js)]
    M = [rs.uniform(size=x.shape) >= 0.2 for x in X]
    X_obs = [np.where(m, x, 0.0) for x, m in zip(X, M)]
    norm_sq = sum(float(np.sum(x ** 2)) for x in X_obs)
    kw = dict(random_state=0, return_errors=True)
    _, diag = cmf_aoadmm(X, R, mask=M, n_iter_max=3000, tol=1e-10, absolute_tol=1e-12, **kw)
    n = diag.n_iter
    assert n < 3000 and diag.message == "FEASIBILITY GAP CRITERION AND ABSOLUTE LOSS CRITERION SATISFIED", (n, diag.message)
    assert diag.rec_errors[-1] < 2e-6, diag.rec_errors[-1]
    for k in sorted({1, 2, 5, 10, 30, 100, 300, 1000, n} & set(range(1, n + 1))):
        (_, (Ak, Bk, Ck)), dk = cmf_aoadmm(X, R, mask=M, n_iter_max=k, tol=None, absolute_tol=None, **kw)
        dense_sq = observed_error(X_obs, M, Ak, Bk, Ck) ** 2 / norm_sq
        assert abs(dk.rec_errors[-1] ** 2 - dense_sq) <= 1e-12, (k, dk.rec_errors[-1] ** 2, dense_sq)
        np.testing.assert_allclose(dk.rec_errors[-1], diag.rec_errors[k], rtol=1e-12)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_case():
    """3 slices; holes in slices 0 and 2 only, so that the rank holding slice 1 has data but no missing entry."""
    X, M = _small_problem(31, [30, 26, 22], 16, 3)
    M[1][:] = True
    X = [np.where(m, np.nan_to_num(x, nan=0.7), np.nan) for x, m in zip(X, M)]
    return X, M, 3, dict(non_negative=True)


def _sharded_worker(rank, world, port, k_iter, out_dir):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.distributed import make_shard

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    if torch.cuda.device_count() >= world:
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, M, R, kw = _sharded_case()
        sh = make_shard([x.shape[0] for x in X], rank, world, n_cols=X[0].shape[1])
        cmf, diag = cmf_aoadmm(X[sh.lo:sh.hi], R, mask=M[sh.lo:sh.hi], n_iter_max=k_iter, tol=None, absolute_tol=None,
                               return_errors=True, random_state=0, process_group=dist.group.WORLD, shard=sh, **kw)
        _, (A, B_is, C) = cmf
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), A=np.asarray(A), C=C, lo=sh.lo, hi=sh.hi,
                 B=np.concatenate(B_is, 0),
                 loss=np.asarray(diag.regularized_loss), rec=np.asarray(diag.rec_errors))
    finally:
        dist.destroy_process_group()


def test_four_rank_masked_run_with_an_empty_rank_equals_single_gpu_run(tmp_path):
    import torch.multiprocessing as mp

    from matcouply_b200 import cmf_aoadmm

    k, world = 20, 4
    mp.spawn(_sharded_worker, args=(world, _free_port(), k, str(tmp_path)), nprocs=world, join=True)
    ranks = [np.load(os.path.join(str(tmp_path), f"rank{r}.npz")) for r in range(world)]
    X, M, R, kw = _sharded_case()
    spans = [(int(r["lo"]), int(r["hi"])) for r in ranks]
    assert any(lo == hi for lo, hi in spans)  # a rank without a slice
    assert any(lo <= 1 < hi and hi - lo == 1 for lo, hi in spans)  # a rank whose data has no hole
    (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, mask=M, n_iter_max=k, tol=None, absolute_tol=None, return_errors=True,
                                         random_state=0, **kw)
    for r in ranks:  # every rank returns the gathered factors
        for key in ("A", "B", "C", "loss", "rec"):
            np.testing.assert_array_equal(r[key], ranks[0][key])
    r0 = ranks[0]
    assert rel(r0["A"], A) < 1e-8 and rel(r0["C"], C) < 1e-8 and rel(r0["B"], np.concatenate(B_is, 0)) < 1e-8
    np.testing.assert_allclose(r0["rec"], diag.rec_errors, rtol=1e-8)
    np.testing.assert_allclose(r0["loss"], diag.regularized_loss, rtol=1e-8)
