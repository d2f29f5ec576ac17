"""TemporalSmoothnessPenalty on the GPU: the partition-solve kernel (b2_prox_temporal) and the value reduction
(b2_temporal_norm) against NumPy fp64 at the sizes they run at, trajectories against the oracle driving
tests/temporal_oracle.py, masked fitting, graph replay, sharded runs, refusals and a planted recovery."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import temporal_oracle as T  # noqa: E402
from masked_oracle import ao_admm_masked  # noqa: E402

from oracle import aoadmm_oracle as O  # noqa: E402

CHUNK = 32  # kChunk of csrc/prox_temporal.cu
CHECKPOINTS = (1, 2, 10, 50)
EPS = {torch.float64: np.finfo(np.float64).eps, torch.float32: np.finfo(np.float32).eps}


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


# ---------------------------------------------------------------------------------------------------------------
# kernel against NumPy fp64
# ---------------------------------------------------------------------------------------------------------------
def _run_kernel(V, rho, lam, dtype, serial=False):
    from matcouply_b200 import _ops

    I, P = V.shape
    dev = torch.device("cuda")
    Vd = torch.as_tensor(V, dtype=dtype, device=dev).contiguous()
    dual, aux = Vd.clone(), torch.empty_like(Vd)
    rho_d = torch.as_tensor(np.asarray(rho), dtype=dtype, device=dev).reshape(-1)
    ws = _ops.prox_temporal_workspace(I, P, 1, dev)
    if serial:
        _ops.prox_temporal_serial(aux, dual, I, P, rho_d, lam, ws)
    else:
        _ops.prox_temporal(aux, dual, I, P, rho_d, lam, ws)
    return Vd, aux, dual


KERNEL_SHAPES = [(1, 33), (2, 31), (3, 32), (CHUNK - 1, 33), (CHUNK, 1), (CHUNK + 1, 64), (5 * CHUNK + 7, 97),
                 (8192, 32), (300, 8192)]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("I,P", KERNEL_SHAPES)
@pytest.mark.parametrize("rho_kind", ["constant", "spread"])
def test_prox_kernel_matches_numpy(I, P, rho_kind, dtype):
    rs = np.random.RandomState(I * 7 + P)
    V = rs.standard_normal((I, P))
    if dtype == torch.float32:
        V = V.astype(np.float32).astype(np.float64)
    rho = np.full(1, 3.0) if rho_kind == "constant" else 10 ** rs.uniform(-2, 2, size=I)
    if dtype == torch.float32:
        rho = rho.astype(np.float32).astype(np.float64)
    rho_full = np.broadcast_to(rho, (I,))
    for ratio in (1e-6, 1e-2, 1.0, 1e2, 1e6):
        lam = ratio * float(np.median(rho_full))
        want = T.prox_stacked(V, rho_full, lam)
        Vd, aux, dual = _run_kernel(V, rho, lam, dtype)
        z = aux.double().cpu().numpy()
        bound = T.cond_bound(rho_full, lam)
        fwd = np.abs(z - want).max() / np.abs(want).max()
        assert fwd <= 64 * EPS[dtype] * bound, (I, P, ratio, fwd, bound)
        # relative residual of the computed solution in fp64
        if I > 1:
            Tz = 2 * lam * (np.vstack([z[:1] - z[1:2], 2 * z[1:-1] - z[:-2] - z[2:], z[-1:] - z[-2:-1]])
                            if I > 2 else np.vstack([z[0] - z[1], z[1] - z[0]])) + rho_full[:, None] * z
            res = np.abs(Tz - rho_full[:, None] * V).max() / (np.abs(rho_full[:, None] * V).max() + 1e-300)
            assert res <= 64 * EPS[dtype] * (1 + 8 * lam / rho_full.min()), (I, P, ratio, res)
        else:
            assert torch.equal(aux, Vd)  # one slice: the identity prox
        assert torch.equal(dual, Vd - aux)  # dual = V - aux exactly as stored
        _, aux2, dual2 = _run_kernel(V, rho, lam, dtype)
        assert torch.equal(aux, aux2) and torch.equal(dual, dual2)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_prox_kernel_at_the_config3_state(dtype):
    """I = 8192 slices of J = 1024 rows at R = 8: the whole mode-1 state of config 3 (and its one-thread-per-position
    baseline, which the partition solve must agree with)."""
    I, P = 8192, 1024 * 8
    g = torch.Generator(device="cuda").manual_seed(5)
    Vd = torch.rand((I, P), dtype=dtype, device="cuda", generator=g)
    rho = torch.rand(I, dtype=dtype, device="cuda", generator=g) * 10 + 0.1
    lam = 2.0
    from matcouply_b200 import _ops

    ws = _ops.prox_temporal_workspace(I, P, 1, "cuda")
    outs = []
    for serial in (False, True):
        dual, aux = Vd.clone(), torch.empty_like(Vd)
        (_ops.prox_temporal_serial if serial else _ops.prox_temporal)(aux, dual, I, P, rho, lam, ws)
        outs.append((aux, dual))
    (aux, dual), (aux_s, _) = outs
    assert torch.equal(dual, Vd - aux)
    cols = torch.arange(0, P, 97, device="cuda")
    Vc, zc = Vd[:, cols].double().cpu().numpy(), aux[:, cols].double().cpu().numpy()
    rho_h = rho.double().cpu().numpy()
    want = T.prox_stacked(Vc, rho_h, lam)
    bound = T.cond_bound(rho_h, lam)
    assert np.abs(zc - want).max() / np.abs(want).max() <= 64 * EPS[dtype] * bound
    diff = (aux.double() - aux_s.double()).abs().max().item() / aux.double().abs().max().item()
    assert diff <= 64 * EPS[dtype] * bound, diff


def test_prox_kernel_argument_errors():
    from matcouply_b200 import _ops

    V = torch.rand(40, 8, dtype=torch.float64, device="cuda")
    rho = torch.ones(40, dtype=torch.float64, device="cuda")
    ws = _ops.prox_temporal_workspace(40, 8, 1, "cuda")
    aux = torch.empty_like(V)
    with pytest.raises(RuntimeError, match="smoothness_reg must be positive"):
        _ops.prox_temporal(aux, V.clone(), 40, 8, rho, 0.0, ws)
    with pytest.raises(RuntimeError, match="workspace too small"):
        _ops.prox_temporal(aux, V.clone(), 40, 8, rho, 1.0, ws[:64])
    with pytest.raises(RuntimeError, match="stage 3 outside"):
        _ops.prox_temporal(aux, V.clone(), 40, 8, rho, 1.0, ws, stage=3)
    with pytest.raises(RuntimeError, match="stage 1 with world"):
        _ops.prox_temporal(aux, V.clone(), 40, 8, rho, 1.0, ws, stage=1)  # no exchange buffer
    with pytest.raises(RuntimeError, match="smoothness_reg must be positive"):
        _ops.temporal_norm(V, 40, 8, -1.0, torch.zeros(1, dtype=torch.float64, device="cuda"),
                           torch.empty(40, dtype=torch.float64, device="cuda"))


@pytest.mark.parametrize("I,J,R", [(1, 5, 3), (2, 4, 2), (40, 0, 3), (CHUNK * 3 + 5, 33, 4), (8192, 64, 8)])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_penalty_value_matches_numpy(I, J, R, dtype):
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    rs = np.random.RandomState(I + J)
    Bs = [rs.standard_normal((J, R)).astype(np.float32 if dtype == torch.float32 else np.float64) for _ in range(I)]
    lam = 0.37
    want = T.TemporalSmoothnessP(lam).value([b.astype(np.float64) for b in Bs])
    pen = TemporalSmoothnessPenalty(lam)
    got = pen.penalty(Bs)
    assert abs(got - want) <= 1e-12 * max(abs(want), 1e-300) + (0 if want else 1e-300)
    assert pen.penalty(Bs) == got  # fixed reduction order


def test_standalone_prox_matches_numpy():
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    rs = np.random.RandomState(4)
    Bs = [rs.standard_normal((6, 3)) for _ in range(45)]
    rhos = list(10 ** rs.uniform(-1, 1, size=45))
    got = TemporalSmoothnessPenalty(0.8).factor_matrices_update(Bs, rhos, None)
    want = T.TemporalSmoothnessP(0.8).prox_list(Bs, rhos, None)
    assert rel(np.concatenate(got), np.concatenate(want)) < 1e-13
    tgot = TemporalSmoothnessPenalty(0.8).factor_matrices_update([torch.as_tensor(b) for b in Bs], rhos, None)
    assert all(isinstance(t, torch.Tensor) for t in tgot)
    assert rel(np.concatenate([t.numpy() for t in tgot]), np.concatenate(want)) < 1e-13


# ---------------------------------------------------------------------------------------------------------------
# trajectories against the oracle
# ---------------------------------------------------------------------------------------------------------------
def _problem(seed, I, J, K, R, noise=0.1):
    """Non-negative data whose B_i drift smoothly over i."""
    rs = np.random.RandomState(seed)
    A, C = rs.uniform(0.1, 1.1, size=(I, R)), rs.uniform(size=(K, R))
    B0, B1 = rs.uniform(size=(J, R)), rs.uniform(size=(J, R))
    Bs = [(1 - s) * B0 + s * B1 + 0.2 * rs.uniform(size=(J, R)) for s in np.linspace(0, 1, I)]
    X = [(B * A[i]) @ C.T for i, B in enumerate(Bs)]
    return [x + noise * rs.standard_normal(x.shape) for x in X]


def _case(name):
    """(X, R, lam, keywords).  lam keeps the penalty between 1 % and 50 % of the regularised loss at iteration 50."""
    if name == "c1_twin":        # config 1 structure: non-negative CMF
        return _problem(1, 40, 16, 24, 4), 4, 3e-6, dict(non_negative=True)
    if name == "c3_twin":        # config 3 structure: PARAFAC2 + non-negativity + the penalty (fused row pass, fork)
        return _problem(2, 40, 20, 16, 3), 3, 1e-4, dict(non_negative=True, parafac2=True)
    if name == "c3_unfused":     # the unfused PARAFAC2 path (FUSION_DEFAULTS["pf2"] = False)
        return _problem(2, 40, 20, 16, 3), 3, 1e-4, dict(non_negative=True, parafac2=True)
    if name == "c3_unimodal":    # unimodality as a second column-coupled companion
        return _problem(3, 40, 20, 16, 3), 3, 3e-5, dict(non_negative=True, parafac2=True, unimodal={1: True})
    if name == "inner_tol":
        return _problem(2, 40, 20, 16, 3), 3, 1e-4, dict(non_negative=True, parafac2=True, inner_tol=1e-3)
    if name == "const_B":
        return _problem(1, 40, 16, 24, 4), 4, 3e-6, dict(non_negative=True, constant_feasibility_penalty="B")
    raise KeyError(name)


@pytest.mark.parametrize("name", ["c1_twin", "c3_twin", "c3_unfused", "c3_unimodal", "inner_tol", "const_B"])
def test_trajectory_matches_oracle(name):
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case(name)
    traj = []
    pen_o = T.TemporalSmoothnessP(lam)
    o = O.ao_admm(X, R, regs=[[], [pen_o], []], random_state=0, n_iter_max=50, tol=None, absolute_tol=None,
                  trajectory=traj, **kw)
    frac = pen_o.value(o["B_is"]) / o["regularized_loss"][-1]
    assert 0.01 <= frac <= 0.5, frac
    from matcouply_b200 import _engine

    for k in CHECKPOINTS:
        _engine.FUSION_DEFAULTS.update(pf2=name != "c3_unfused")
        try:
            (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []],
                                                 random_state=0, n_iter_max=k, tol=None, absolute_tol=None,
                                                 return_errors=True, **kw)
        finally:
            _engine.FUSION_DEFAULTS.update(pf2=True)
        errs = (rel(A, traj[k - 1]["A"]), rel(np.concatenate(B_is, 0), np.concatenate(traj[k - 1]["B_is"], 0)),
                rel(C, traj[k - 1]["C"]))
        assert max(errs) < 1e-8, (name, k, errs)
        np.testing.assert_allclose(diag.rec_errors, o["rec_errors"][:k + 1], rtol=1e-8)
        np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"][:k + 1], rtol=1e-8)


def test_stopping_iteration_matches_oracle():
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case("c3_twin")
    o = O.ao_admm(X, R, regs=[[], [T.TemporalSmoothnessP(lam)], []], random_state=0, n_iter_max=300, tol=1e-6,
                  **kw)
    _, diag = cmf_aoadmm(X, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], random_state=0, n_iter_max=300,
                         tol=1e-6, return_errors=True, **kw)
    assert diag.n_iter == o["n_iter"] and diag.message == o["message"], (diag.n_iter, o["n_iter"])
    np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"], rtol=1e-8)


def test_fp32_config3_twin_tracks_the_fp64_oracle():
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case("c3_twin")
    X32 = [x.astype(np.float32) for x in X]
    kw = dict(kw, random_state=0, n_iter_max=30, tol=None, absolute_tol=None)
    o = O.ao_admm([x.astype(np.float64) for x in X32], R, regs=[[], [T.TemporalSmoothnessP(lam)], []], **kw)
    _, (A, B_is, C) = cmf_aoadmm(X32, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], **kw)
    assert rel(A, o["A"]) < 5e-3 and rel(C, o["C"]) < 5e-3
    assert rel(np.concatenate(B_is, 0), np.concatenate(o["B_is"], 0)) < 5e-3


def test_masked_trajectory_matches_the_masked_oracle():
    """Temporal PARAFAC2 on incomplete data: 10 % of the entries and some whole rows missing."""
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case("c3_twin")
    rs = np.random.RandomState(11)
    M = [rs.uniform(size=x.shape) >= 0.1 for x in X]
    for i in range(0, len(M), 5):
        M[i][i % M[i].shape[0]] = False
    Xn = [np.where(m, x, np.nan) for x, m in zip(X, M)]
    traj = []
    o = ao_admm_masked(Xn, R, M, regs=[[], [T.TemporalSmoothnessP(lam)], []], random_state=0, n_iter_max=50,
                       tol=None, absolute_tol=None, trajectory=traj, **kw)
    for k in (1, 10, 50):
        (_, (A, B_is, C)), diag = cmf_aoadmm(Xn, R, mask=M, regs=[[], [TemporalSmoothnessPenalty(lam)], []],
                                             random_state=0, n_iter_max=k, tol=None, absolute_tol=None,
                                             return_errors=True, **kw)
        errs = (rel(A, traj[k - 1]["A"]), rel(np.concatenate(B_is, 0), np.concatenate(traj[k - 1]["B_is"], 0)),
                rel(C, traj[k - 1]["C"]))
        assert max(errs) < 1e-8, (k, errs)
        np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"][:k + 1], rtol=1e-8)


@pytest.mark.parametrize("name", ["c1_twin", "c3_twin"])
def test_graph_replay_equals_eager_launches(name):
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case(name)
    runs = [cmf_aoadmm(X, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], random_state=0, n_iter_max=30,
                       tol=None, absolute_tol=None, return_errors=True, use_cuda_graph=g, **kw) for g in (True, False)]
    (_, fa), da = runs[0]
    (_, fb), db = runs[1]
    assert np.array_equal(fa[0], fb[0]) and np.array_equal(fa[2], fb[2])
    assert np.array_equal(np.concatenate(fa[1], 0), np.concatenate(fb[1], 0))
    assert da.rec_errors == db.rec_errors and da.regularized_loss == db.regularized_loss


# ---------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------
def test_refusals():
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    X, R, lam, kw = _case("c1_twin")
    for mode in (0, 2):
        regs = [[], [], []]
        regs[mode] = [TemporalSmoothnessPenalty(lam)]
        with pytest.raises(ValueError, match="GeneralizedL2Penalty with a path-graph Laplacian"):
            cmf_aoadmm(X, R, regs=regs, n_iter_max=2, constant_feasibility_penalty=True)
    ragged = [X[0], X[1][:-3]] + X[2:]
    with pytest.raises(ValueError, match=r"found heights \[13, 16\]"):
        cmf_aoadmm(ragged, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], n_iter_max=2)
    with pytest.raises(ValueError, match=r"found heights"):
        TemporalSmoothnessPenalty(lam).factor_matrices_update([np.ones((3, 2)), np.ones((4, 2))], [1.0, 1.0], None)
    with pytest.raises(TypeError):
        TemporalSmoothnessPenalty(lam).penalty(np.ones((3, 2)))


# ---------------------------------------------------------------------------------------------------------------
# planted behaviour
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_smoothness_improves_recovery_of_drifting_factors(seed):
    """B_i drift smoothly over i, noisy data with 30 % of the entries missing: with the penalty the recovered B_i
    are closer to the truth than without it (the masked NumPy oracle gives 0.16-0.18 against 0.49-0.72)."""
    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    rs = np.random.RandomState(100 + seed)
    I, J, K, R = 60, 15, 30, 2
    A, C = rs.uniform(0.5, 1.5, size=(I, R)), rs.uniform(size=(K, R))
    t = np.linspace(0, 2 * np.pi, I)
    Bs = [np.abs(np.stack([np.sin(t[i] + np.linspace(0, 3, J)) + 1.2,
                           np.cos(0.5 * t[i] + np.linspace(0, 2, J)) + 1.2], 1)) for i in range(I)]
    X = [(B * A[i]) @ C.T for i, B in enumerate(Bs)]
    X = [x + 0.3 * rs.standard_normal(x.shape) for x in X]
    M = [rs.uniform(size=x.shape) >= 0.3 for x in X]
    Xn = [np.where(m, x, np.nan) for x, m in zip(X, M)]

    def err(regs):
        _, (Ah, Bh, Ch) = cmf_aoadmm(Xn, R, mask=M, regs=regs, non_negative=True, random_state=seed,
                                     n_iter_max=300, tol=1e-9, absolute_tol=1e-12)
        # the stacked B_i up to the scale of each component (which A absorbs), best of both component orders
        true = np.concatenate(Bs) / np.linalg.norm(np.concatenate(Bs), axis=0)
        est = np.concatenate(Bh) / np.linalg.norm(np.concatenate(Bh), axis=0)
        return min(np.linalg.norm(est[:, perm] - true) / np.linalg.norm(true) for perm in ([0, 1], [1, 0]))

    plain = err([[], [], []])
    smooth = err([[], [TemporalSmoothnessPenalty(0.1)], []])
    assert smooth < 0.5 * plain, (smooth, plain)


# ---------------------------------------------------------------------------------------------------------------
# sharded runs
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_case(name):
    if name == "c3_twin":
        X, R, lam, kw = _case("c3_twin")
        return X, R, lam, kw
    if name == "c1_few_slices":  # fewer slices than ranks at 4 ranks; a rank with one slice at 2
        X = _problem(5, 3, 16, 24, 4)
        return X, 4, 1e-3, dict(non_negative=True)
    if name == "c1_single_slice_rank":
        X = _problem(6, 9, 16, 24, 4)
        return X, 4, 3e-5, dict(non_negative=True)
    raise KeyError(name)


def _sharded_worker(rank, world, port, name, k_iter, cuts, out_dir):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.distributed import ShardSpec
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    if torch.cuda.device_count() >= world:
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, R, lam, kw = _sharded_case(name)
        lo, hi = cuts[rank], cuts[rank + 1]
        sh = ShardSpec(tuple(x.shape[0] for x in X), lo, hi, X[0].shape[1])
        cmf, diag = cmf_aoadmm(X[lo:hi], R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], n_iter_max=k_iter,
                               tol=None, absolute_tol=None, return_errors=True, random_state=0,
                               process_group=dist.group.WORLD, shard=sh, **kw)
        _, (A, B_is, C) = cmf
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), A=A, B=np.concatenate(B_is, 0), C=C,
                 loss=np.asarray(diag.regularized_loss), rec=np.asarray(diag.rec_errors))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name,cuts", [
    ("c3_twin", (0, 17, 40)),                 # 2 ranks
    ("c3_twin", (0, 1, 20, 21, 40)),          # 4 ranks, two of them with a single slice
    ("c1_single_slice_rank", (0, 1, 9)),      # 2 ranks, the first with one slice
    ("c1_few_slices", (0, 1, 2, 3, 3)),       # 4 ranks, 3 slices: one rank holds none
    ("c1_few_slices", (0, 0, 2, 2, 3)),       # empty ranks first and in the middle
])
def test_sharded_run_equals_single_gpu_run(name, cuts, tmp_path):
    import torch.multiprocessing as mp

    from matcouply_b200 import cmf_aoadmm
    from matcouply_b200.penalties import TemporalSmoothnessPenalty

    world, k = len(cuts) - 1, 20
    mp.spawn(_sharded_worker, args=(world, _free_port(), name, k, cuts, str(tmp_path)), nprocs=world, join=True)
    res = [np.load(os.path.join(str(tmp_path), f"rank{r}.npz")) for r in range(world)]
    for r in res[1:]:
        for key in ("A", "B", "C", "loss", "rec"):
            np.testing.assert_array_equal(res[0][key], r[key])
    X, R, lam, kw = _sharded_case(name)
    (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, regs=[[], [TemporalSmoothnessPenalty(lam)], []], n_iter_max=k,
                                         tol=None, absolute_tol=None, return_errors=True, random_state=0, **kw)
    errs = (rel(res[0]["A"], A), rel(res[0]["B"], np.concatenate(B_is, 0)), rel(res[0]["C"], C))
    assert max(errs) < 1e-10, errs
    np.testing.assert_allclose(res[0]["rec"], diag.rec_errors, rtol=1e-10)
    np.testing.assert_allclose(res[0]["loss"], diag.regularized_loss, rtol=1e-10)
