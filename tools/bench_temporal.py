"""Cost of TemporalSmoothnessPenalty on device-resident seeded data.

    python tools/bench_temporal.py [--steps 5] [--reps 3] [--out profiles/temporal_bench.json]

Shapes: BASELINE config 3 (8192 slices 1024 x 256, R = 8, non-negative PARAFAC2 + unimodality + L2Ball, fp64) and config 1 (4096
slices 256 x 512, R = 16, non-negative CMF, fp64), each with TemporalSmoothnessPenalty added on mode 1.  Reported:

- the b2_prox_temporal time by CUDA events on the whole mode-1 state (I slices x J * R positions), its rate against
  the traffic model 4 N R sizeof(T) (V read twice, aux and dual written once), and the same numbers for the
  one-thread-per-position baseline b2_prox_temporal_serial;
- the steady-state outer-iteration time with and without the penalty, alternated in one process (diagnostics read
  every iteration, as with a tolerance set);
- one or two outer iterations with the same penalty written as a Python MatricesPenalty (host bridge, SciPy banded
  solve), for scale.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.linalg import solve_banded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from matcouply_b200 import _ops  # noqa: E402
from matcouply_b200._engine import AOADMMEngine, PackedMatrices  # noqa: E402
from matcouply_b200.decomposition import _parse_all_penalties  # noqa: E402
from matcouply_b200.penalties import MatricesPenalty, TemporalSmoothnessPenalty  # noqa: E402

SHAPES = {
    "c3": dict(I=8192, J=1024, K=256, R=8, kw=dict(non_negative=True, parafac2=True, unimodal={1: True},
                                                   l2_norm_bound=[0, 1, 1]),
               host_iters=1),
    "c1": dict(I=4096, J=256, K=512, R=16, kw=dict(non_negative=True), host_iters=2),
}
LAM = 1e-3


class HostTemporal(MatricesPenalty):
    """The same penalty in Python: the engine hands the pre-image to the host and takes the aux back."""

    def __init__(self, lam):
        super().__init__()
        self.lam = lam

    def factor_matrices_update(self, factor_matrices, feasibility_penalties, auxes):
        V = np.stack([np.asarray(m).reshape(-1) for m in factor_matrices])
        rho = np.asarray(feasibility_penalties, dtype=np.float64)
        I = V.shape[0]
        deg = np.zeros(I)
        deg[1:] += 1
        deg[:-1] += 1
        ab = np.zeros((3, I))
        ab[0, 1:] = ab[2, :-1] = -2 * self.lam
        ab[1] = rho + 2 * self.lam * deg
        z = solve_banded((1, 1), ab, rho[:, None] * V)
        return [zi.reshape(np.shape(m)) for zi, m in zip(z, factor_matrices)]

    def penalty(self, x):
        X = np.stack([np.asarray(b).reshape(-1) for b in x])
        return self.lam * float(np.sum((X[1:] - X[:-1]) ** 2))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in q.strip().split(",")[:2]]
    except Exception:  # noqa: BLE001 - the name from torch is enough when nvidia-smi is unavailable
        name, power = torch.cuda.get_device_name(), "not measured"
    return name, power


def make_data(shape, seed, dev):
    I, J, K = shape["I"], shape["J"], shape["K"]
    off = (np.arange(I + 1) * J).astype(np.int64)
    gen = torch.Generator(device=dev).manual_seed(seed)
    X = torch.zeros((I * J, _ops.padded_ld(K, torch.float64)), dtype=torch.float64, device=dev)
    X[:, :K] = torch.rand((I * J, K), dtype=torch.float64, device=dev, generator=gen)
    return PackedMatrices(X, off, K)


def make_engine(packed, shape, extra):
    kw = shape["kw"]
    regs = _parse_all_penalties(svd="truncated_svd", regs=[[], list(extra), []], dual_init="random_uniform",
                                aux_init="random_uniform", verbose=False, lower_bound=None, upper_bound=None,
                                tv_penalty=None, generalized_l2_penalty=None, l1_penalty=None,
                                **{k: kw.get(k) for k in ("non_negative", "parafac2", "unimodal", "l2_norm_bound")})
    eng = AOADMMEngine(packed, shape["R"], regs)
    eng.load_state_device(seed=1)
    eng.prepare()
    eng.use_graph = eng.graph_auto()  # cmf_aoadmm's policy
    for _ in range(2):
        step(eng, graph=False)
    return eng


def step(eng, graph=True):
    launched = eng.graph_iteration(True) if (graph and eng.use_graph) else None
    if launched is None:
        eng.outer_iteration()
        eng.diagnostics()
    else:
        eng._read_diagnostics(launched)


def time_steps(eng, n):
    step(eng)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        step(eng)  # ends in the device->host read of the scalar pack
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n


def event_time(fn, n):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n * 1e-3


def kernel_times(shape, dev, n):
    I, P = shape["I"], shape["J"] * shape["R"]
    gen = torch.Generator(device=dev).manual_seed(3)
    V = torch.rand((I, P), dtype=torch.float64, device=dev, generator=gen)
    rho = torch.rand(I, dtype=torch.float64, device=dev, generator=gen) + 0.5
    aux, dual = torch.empty_like(V), V.clone()
    ws = _ops.prox_temporal_workspace(I, P, 1, dev)
    model = 4 * I * P * 8
    out = {}
    for name, fn in (("partition", lambda: _ops.prox_temporal(aux, dual, I, P, rho, LAM, ws)),
                     ("serial_baseline", lambda: _ops.prox_temporal_serial(aux, dual, I, P, rho, LAM, ws))):
        t = event_time(fn, n)
        out[name] = dict(seconds=t, model_bytes=model, model_TBps=model / t / 1e12)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-launches", type=int, default=20)
    ap.add_argument("--shapes", default="c3,c1")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_temporal.py needs a GPU")
    dev = torch.device("cuda")
    name, power = card()
    results = []
    for key in args.shapes.split(","):
        shape = SHAPES[key]
        res = dict(shape=key, I=shape["I"], J=shape["J"], K=shape["K"], R=shape["R"], lam=LAM,
                   kernel=kernel_times(shape, dev, args.kernel_launches))
        torch.cuda.empty_cache()
        packed = make_data(shape, 1, dev)
        engines = {"without": make_engine(packed, shape, []),
                   "with": make_engine(packed, shape, [TemporalSmoothnessPenalty(LAM)])}
        steps = {k: [] for k in engines}
        for _ in range(args.reps):
            for k, eng in engines.items():  # alternated in one process
                steps[k].append(time_steps(eng, args.steps))
        res["step_seconds"] = {k: dict(median=float(np.median(v)), all=v) for k, v in steps.items()}
        res["graph_replay"] = {k: bool(e.use_graph) for k, e in engines.items()}
        del engines
        torch.cuda.empty_cache()
        eng = make_engine(packed, shape, [HostTemporal(LAM)])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(shape["host_iters"]):
            step(eng, graph=False)
        torch.cuda.synchronize()
        res["host_bridge_step_seconds"] = (time.perf_counter() - t0) / shape["host_iters"]
        res["host_bridge_iterations"] = shape["host_iters"]
        del eng, packed
        torch.cuda.empty_cache()
        print(json.dumps(res), flush=True)
        results.append(res)
    out = dict(card=name, power_limit=power, steps=args.steps, reps=args.reps, results=results)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
