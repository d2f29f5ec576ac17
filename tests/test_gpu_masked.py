"""Masked fitting on the GPU: the b2_mask_refill kernel against NumPy, masked trajectories against the oracle's
restatement of the EM semantics (tests/masked_oracle.py), graph replay, the no-hole case, the
caller's buffer and the sharded run."""
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
from masked_oracle import ao_admm_masked  # noqa: E402

CHECKPOINTS = (1, 2, 5, 10, 20, 35, 50)


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


def _problem(seed, Js, K, R, noise=0.1, frac=0.2):
    """Non-negative rank-R ragged data with a random mask (1 = observed); NaN at the missing positions."""
    rs = np.random.RandomState(seed)
    A, C = rs.uniform(0.1, 1.1, size=(len(Js), R)), rs.uniform(size=(K, R))
    X = [(rs.uniform(size=(J, R)) * A[i]) @ C.T for i, J in enumerate(Js)]
    X = [x + noise * rs.standard_normal(x.shape) for x in X]
    M = [rs.uniform(size=x.shape) >= frac for x in X]
    return [np.where(m, x, np.nan) for x, m in zip(X, M)], M


# ---------------------------------------------------------------------------------------------------------------
# kernel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("R", [1, 3, 8, 16, 20, 32])
def test_mask_refill_kernel_matches_numpy(R, dtype):
    from matcouply_b200 import _ops
    from matcouply_b200._engine import pack_mask

    rs = np.random.RandomState(R)
    K = 37
    Js = [5, 0, 40, 1, 33]  # an empty slice and a one-row slice
    N = sum(Js)
    masks = [rs.uniform(size=(J, K)) >= 0.3 for J in Js]
    masks[2][3] = True      # a row with no missing entry
    masks[2][4] = False     # a fully missing row
    masks[4][::2] = True    # every other row complete
    pm = pack_mask(masks, [(J, K) for J in Js])
    ld = _ops.padded_ld(K, dtype)
    X = np.zeros((N, ld))
    X[:, :K] = rs.standard_normal((N, K))
    A, B, C, Y = rs.uniform(size=(len(Js), R)), rs.standard_normal((N, R)), rs.standard_normal((K, R)), \
        rs.standard_normal((N, R))
    gor = np.repeat(np.arange(len(Js)), Js).astype(np.int32)
    if dtype == torch.float32:
        X, A, B, C, Y = (a.astype(np.float32).astype(np.float64) for a in (X, A, B, C, Y))

    # NumPy reference
    Xr, Yr = X.copy(), Y.copy()
    out_ref = np.zeros(2)
    miss = np.zeros((N, K), dtype=bool)
    miss[:, :] = ~np.concatenate(masks, 0)
    rows, cols = np.nonzero(miss)
    xhat = np.einsum("nr,nr,nr->n", B[rows], A[gor[rows]], C[cols])
    d = xhat - X[rows, cols]
    out_ref[0] = np.sum(d ** 2)
    out_ref[1] = np.sum(xhat ** 2 - X[rows, cols] ** 2)
    np.add.at(Yr, rows, d[:, None] * C[cols])
    Xr[rows, cols] = xhat

    dev = torch.device("cuda")
    t = lambda a: torch.as_tensor(a, dtype=dtype, device=dev).contiguous()  # noqa: E731
    mdev = pm.to(dev)
    ws = _ops.mask_refill_workspace(N, dev)
    tol = 1e-13 if dtype == torch.float64 else 1e-5
    results = []
    for use_y in (True, False):
        for _rep in range(2):
            Xd, Yd = t(X), t(Y)
            out = torch.zeros(2, dtype=torch.float64, device=dev)
            _ops.mask_refill(Xd, N, K, mdev.row_ptr, mdev.col, torch.as_tensor(gor, device=dev), t(A), t(B), t(C),
                             Yd if use_y else None, out, ws)
            Xg, Yg, og = Xd.cpu().double().numpy(), Yd.cpu().double().numpy(), out.cpu().numpy()
            assert rel(Xg, Xr) < tol, rel(Xg, Xr)
            assert rel(Yg, Yr if use_y else Y) < tol
            assert abs(og[0] - out_ref[0]) <= tol * abs(out_ref[0])
            assert abs(og[1] - out_ref[1]) <= tol * np.sum(np.abs(xhat ** 2) + X[rows, cols] ** 2)
            results.append((Xg, Yg, og))
    for a, b in ((0, 1), (2, 3)):  # the same input gives the same bits
        for u, v in zip(results[a], results[b]):
            assert np.array_equal(u, v)


# ---------------------------------------------------------------------------------------------------------------
# trajectories against the oracle (fp64)
# ---------------------------------------------------------------------------------------------------------------
def _case(name):
    rs = np.random.RandomState(7)
    if name == "nn_cmf_r16":             # (a) two-pass schedule, graph replay from iteration 2 on
        X, M = _problem(1, rs.randint(20, 40, size=8), 30, 16)
        return X, M, 16, dict(non_negative=True)
    if name == "nn_cmf_r8_fused":        # (b) single-read fused pass
        X, M = _problem(2, rs.randint(40, 60, size=6), 40, 8)
        return X, M, 8, dict(non_negative=True)
    if name == "pf2_nn_ragged":          # (c)
        X, M = _problem(3, rs.randint(8, 40, size=10), 24, 3)
        return X, M, 3, dict(non_negative=True, parafac2=True)
    if name == "pf2_unimodal_l2ball":    # (d) forked eager PARAFAC2 path
        X, M = _problem(4, [40] * 8, 16, 3)
        return X, M, 3, dict(non_negative=True, parafac2=True, unimodal={1: True}, l2_norm_bound=[0, 1, 1])
    if name == "rows_and_column":        # (e) whole rows and a whole column missing
        X, M = _problem(5, rs.randint(10, 30, size=8), 20, 4, frac=0.05)
        for i, m in enumerate(M):
            m[:, 7] = False
            m[i % m.shape[0]] = False
        X = [np.where(m, x, np.nan) for x, m in zip(X, M)]
        return X, M, 4, dict(non_negative=True)
    if name == "frozen_C":               # (f) update_C=False
        X, M = _problem(6, rs.randint(10, 30, size=8), 20, 4)
        return X, M, 4, dict(non_negative=True, update_C=False)
    raise KeyError(name)


CASES = ["nn_cmf_r16", "nn_cmf_r8_fused", "pf2_nn_ragged", "pf2_unimodal_l2ball", "rows_and_column", "frozen_C"]


@pytest.mark.parametrize("name", CASES)
def test_masked_trajectory_matches_oracle(name):
    from matcouply_b200 import cmf_aoadmm

    X, M, R, kw = _case(name)
    if name == "nn_cmf_r8_fused":
        from matcouply_b200 import penalties as P
        from matcouply_b200._engine import AOADMMEngine, PackedMatrices

        packed = PackedMatrices.from_list([np.nan_to_num(x) for x in X], torch.float64, torch.device("cuda"))
        assert AOADMMEngine(packed, R, [[P.NonNegativity()] for _ in range(3)]).fused_x1
    traj = []
    o = ao_admm_masked(X, R, M, random_state=0, n_iter_max=50, tol=None, absolute_tol=None, trajectory=traj, **kw)
    for k in CHECKPOINTS:
        (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, mask=M, random_state=0, n_iter_max=k, tol=None, absolute_tol=None,
                                             return_errors=True, **kw)
        errs = (rel(A, traj[k - 1]["A"]), rel(np.concatenate(B_is, 0), np.concatenate(traj[k - 1]["B_is"], 0)),
                rel(C, traj[k - 1]["C"]))
        assert max(errs) < 1e-8, (name, k, errs)
        np.testing.assert_allclose(diag.rec_errors, o["rec_errors"][:k + 1], rtol=1e-8)
        np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"][:k + 1], rtol=1e-8)


@pytest.mark.parametrize("name", ["rows_and_column", "pf2_nn_ragged"])
def test_masked_stopping_rule_matches_oracle(name):
    from matcouply_b200 import cmf_aoadmm

    X, M, R, kw = _case(name)
    o = ao_admm_masked(X, R, M, random_state=0, n_iter_max=400, tol=1e-6, **kw)
    _, diag = cmf_aoadmm(X, R, mask=M, random_state=0, n_iter_max=400, tol=1e-6, return_errors=True, **kw)
    assert diag.n_iter == o["n_iter"] and diag.message == o["message"], (diag.n_iter, o["n_iter"], diag.message)
    assert diag.n_iter < 400
    np.testing.assert_allclose(diag.rec_errors, o["rec_errors"], rtol=1e-8)
    np.testing.assert_allclose(diag.regularized_loss, o["regularized_loss"], rtol=1e-8)


def test_masked_fp32_tracks_the_fp64_oracle():
    from matcouply_b200 import cmf_aoadmm

    X, M, R, kw = _case("pf2_nn_ragged")
    X32 = [x.astype(np.float32) for x in X]
    kw = dict(kw, l1_penalty={2: 0.1}, random_state=0, n_iter_max=30, tol=None, absolute_tol=None)
    o = ao_admm_masked([x.astype(np.float64) for x in X32], R, M, **kw)
    _, (A, B_is, C) = cmf_aoadmm(X32, R, mask=M, **kw)
    assert rel(A, o["A"]) < 5e-3 and rel(C, o["C"]) < 5e-3
    assert rel(np.concatenate(B_is, 0), np.concatenate(o["B_is"], 0)) < 5e-3


def test_masked_graph_replay_equals_eager_launches():
    from matcouply_b200 import cmf_aoadmm

    X, M, R, kw = _case("nn_cmf_r16")
    runs = [cmf_aoadmm(X, R, mask=M, random_state=0, n_iter_max=30, tol=None, absolute_tol=None, return_errors=True,
                       use_cuda_graph=g, **kw) for g in (True, False)]
    (_, fa), da = runs[0]
    (_, fb), db = runs[1]
    for a, b in zip(fa, fb):
        assert np.array_equal(np.concatenate(a, 0) if isinstance(a, list) else a,
                              np.concatenate(b, 0) if isinstance(b, list) else b)
    assert da.rec_errors == db.rec_errors and da.regularized_loss == db.regularized_loss


@pytest.mark.parametrize("name", ["nn_cmf_r16", "nn_cmf_r8_fused", "pf2_nn_ragged"])
def test_mask_without_holes_is_the_unmasked_run(name):
    from matcouply_b200 import _lib, cmf_aoadmm

    X, M, R, kw = _case(name)
    X = [np.nan_to_num(x, nan=0.5) for x in X]
    lib = _lib.load()
    out, launches = [], []
    for mask in (None, [np.ones(x.shape, dtype=bool) for x in X]):
        per_k = []
        for k in (20, 21):
            c0 = lib.b2_launch_count()
            res = cmf_aoadmm(X, R, mask=mask, random_state=0, n_iter_max=k, tol=None, absolute_tol=None,
                             return_errors=True, **kw)
            per_k.append(lib.b2_launch_count() - c0)
        out.append(res)
        launches.append(per_k[1] - per_k[0])  # launches of one outer iteration
    (_, fa), da = out[0]
    (_, fb), db = out[1]
    assert np.array_equal(fa[0], fb[0]) and np.array_equal(fa[2], fb[2])
    assert np.array_equal(np.concatenate(fa[1], 0), np.concatenate(fb[1], 0))
    assert da.rec_errors == db.rec_errors and da.regularized_loss == db.regularized_loss
    assert da.feasibility_gaps == db.feasibility_gaps
    assert launches[0] == launches[1]


def test_packed_input_with_nan_holes_is_restored():
    from matcouply_b200 import PackedMatrices, cmf_aoadmm

    X, M, R, kw = _case("nn_cmf_r16")
    dev = torch.device("cuda")
    packed = PackedMatrices.from_list(X, torch.float64, dev)
    before = packed.X.clone()
    mask_t = torch.as_tensor(np.concatenate(M, 0), device=dev)
    for mask in (M, mask_t):
        (_, (A, B_is, C)), diag = cmf_aoadmm(packed, R, mask=mask, random_state=0, n_iter_max=20, tol=None,
                                             absolute_tol=None, return_errors=True, **kw)
        assert all(np.all(np.isfinite(v)) for v in (A, C, np.concatenate(B_is, 0), diag.rec_errors,
                                                     diag.regularized_loss))
        assert torch.equal(packed.X.isnan(), before.isnan())
        assert torch.equal(torch.nan_to_num(packed.X), torch.nan_to_num(before))  # bit-identical, NaN included
        o = ao_admm_masked(X, R, M, random_state=0, n_iter_max=20, tol=None, absolute_tol=None, **kw)
        assert rel(A, o["A"]) < 1e-8 and rel(C, o["C"]) < 1e-8
    # an exception inside the fit, after the first refills: the caller's values come back too
    from matcouply_b200.penalties import MatrixPenalty

    class Failing(MatrixPenalty):
        calls = 0

        def factor_matrix_update(self, factor_matrix, feasibility_penalty, aux):
            Failing.calls += 1
            if Failing.calls > 3:
                raise RuntimeError("penalty failed")
            return np.maximum(factor_matrix, 0)

        def penalty(self, x):
            return 0.0

    with pytest.raises(RuntimeError, match="penalty failed"):
        cmf_aoadmm(packed, R, mask=M, random_state=0, n_iter_max=5, tol=None, absolute_tol=None,
                   regs=[[], [], [Failing()]], **kw)
    assert Failing.calls == 4
    assert torch.equal(torch.nan_to_num(packed.X), torch.nan_to_num(before))
    assert torch.equal(packed.X.isnan(), before.isnan())


# ---------------------------------------------------------------------------------------------------------------
# sharded
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _masked_worker(rank, world, port, name, k_iter, out_dir):
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
        X, M, R, kw = _case(name)
        sh = make_shard([x.shape[0] for x in X], rank, world, n_cols=X[0].shape[1])
        cmf, diag = cmf_aoadmm(X[sh.lo:sh.hi], R, mask=M[sh.lo:sh.hi], n_iter_max=k_iter, tol=None, absolute_tol=None,
                               return_errors=True, random_state=0, process_group=dist.group.WORLD, shard=sh, **kw)
        _, (A, B_is, C) = cmf
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), A=A, B=np.concatenate(B_is, 0), C=C,
                 loss=np.asarray(diag.regularized_loss), rec=np.asarray(diag.rec_errors))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name", ["nn_cmf_r16", "pf2_nn_ragged"])
def test_two_rank_masked_run_equals_single_gpu_run(name, tmp_path):
    import torch.multiprocessing as mp

    from matcouply_b200 import cmf_aoadmm

    k = 20
    mp.spawn(_masked_worker, args=(2, _free_port(), name, k, str(tmp_path)), nprocs=2, join=True)
    r0 = np.load(os.path.join(str(tmp_path), "rank0.npz"))
    r1 = np.load(os.path.join(str(tmp_path), "rank1.npz"))
    for key in ("A", "B", "C", "loss", "rec"):
        np.testing.assert_array_equal(r0[key], r1[key])
    X, M, R, kw = _case(name)
    (_, (A, B_is, C)), diag = cmf_aoadmm(X, R, mask=M, n_iter_max=k, tol=None, absolute_tol=None, return_errors=True,
                                         random_state=0, **kw)
    assert rel(r0["A"], A) < 1e-8 and rel(r0["C"], C) < 1e-8 and rel(r0["B"], np.concatenate(B_is, 0)) < 1e-8
    np.testing.assert_allclose(r0["rec"], diag.rec_errors, rtol=1e-8)
    np.testing.assert_allclose(r0["loss"], diag.regularized_loss, rtol=1e-8)
