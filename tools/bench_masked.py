"""Cost of masked fitting (missing entries, EM refill after every outer iteration) on device-resident seeded data.

    python tools/bench_masked.py [--steps 10] [--reps 3] [--out profiles/masked_bench.json]

Shapes: BASELINE config 1 (4096 slices 256 x 512, R = 16, non-negative CMF, fp64) and the config-2 slice shape with
fewer slices (1024 ragged slices J_i in 256..2048 x 1024, R = 20, non-negative PARAFAC2 + L1 on C, fp64).  Patterns:
1 %, 10 %, 30 % of the entries missing uniformly at random, and 10 % of whole rows missing.  For every pattern, in one
process and alternating the two arms: the steady-state outer-iteration time with and without the mask (graph policy
as in cmf_aoadmm, diagnostics read every iteration as with a tolerance set), the b2_mask_refill time by CUDA events,
its bytes from the model below, and its time relative to one b2_xstream_y launch (Y = X C) on the same data.

Byte model of one refill: the distinct 32-byte sectors of X that hold a missing entry, read and written; miss_col
(4 B per missing entry); row_ptr (8 B per row); and, for every row with a missing entry, the B-row (read) and the
Y-row (read and write).  C (K x R) is L2-resident and not counted.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from matcouply_b200 import _ops  # noqa: E402
from matcouply_b200._engine import AOADMMEngine, PackedMatrices, pack_mask_device  # noqa: E402
from matcouply_b200.decomposition import _parse_all_penalties  # noqa: E402

SHAPES = {
    "c1": dict(I=4096, J=(256, 256), K=512, R=16, kw=dict(non_negative=True)),
    "c2_slices": dict(I=1024, J=(256, 2048), K=1024, R=20, kw=dict(non_negative=True, parafac2=True,
                                                                   l1_penalty={2: 0.1})),
}
PATTERNS = [("random_1pct", 0.01, False), ("random_10pct", 0.10, False), ("random_30pct", 0.30, False),
            ("rows_10pct", 0.10, True)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in q.strip().split(",")[:2]]
    except Exception:  # noqa: BLE001 - the name from torch is enough when nvidia-smi is unavailable
        name, power = torch.cuda.get_device_name(), "not measured"
    return name, power


def make_data(shape, seed, dev):
    rs = np.random.RandomState(seed)
    lo, hi = shape["J"]
    Js = rs.randint(lo, hi + 1, size=shape["I"]) if hi > lo else np.full(shape["I"], lo)
    off = np.concatenate([[0], np.cumsum(Js)]).astype(np.int64)
    N, K = int(off[-1]), shape["K"]
    gen = torch.Generator(device=dev).manual_seed(seed)
    X = torch.zeros((N, _ops.padded_ld(K, torch.float64)), dtype=torch.float64, device=dev)
    X[:, :K] = torch.rand((N, K), dtype=torch.float64, device=dev, generator=gen)
    return PackedMatrices(X, off, K), gen


def make_mask(packed, frac, whole_rows, gen):
    N, K = packed.N, packed.K
    if whole_rows:
        rows = torch.rand(N, device=packed.X.device, generator=gen) >= frac
        return rows[:, None].expand(N, K).contiguous()
    return torch.rand((N, K), device=packed.X.device, generator=gen) >= frac


def make_engine(packed, shape, mask):
    regs = _parse_all_penalties(svd="truncated_svd", regs=None, dual_init="random_uniform",
                                aux_init="random_uniform", verbose=False, lower_bound=None, upper_bound=None,
                                l2_norm_bound=None, unimodal=None, tv_penalty=None, generalized_l2_penalty=None,
                                **{k: shape["kw"].get(k) for k in ("non_negative", "parafac2", "l1_penalty")})
    eng = AOADMMEngine(packed, shape["R"], regs, mask=mask)
    eng.load_state_device(seed=1)
    eng.prepare()
    eng.use_graph = eng.graph_auto()  # cmf_aoadmm's policy for n_iter_max >= 16
    for _ in range(2):  # the eager iterations before the steady state
        eng.outer_iteration()
        eng.diagnostics()
    return eng


def step(eng):
    launched = eng.graph_iteration(True) if eng.use_graph else None
    if launched is None:
        eng.outer_iteration()
        eng.diagnostics()
    else:
        eng._read_diagnostics(launched)


def time_steps(eng, n):
    step(eng)  # warm (captures the graph on first use)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        step(eng)  # every step ends in the device->host read of the scalar pack
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


def refill_bytes(m, packed, R):
    es = 8
    row_ptr, col = m.row_ptr, m.col.to(torch.int64)
    counts = torch.diff(row_ptr)
    rows = torch.repeat_interleave(torch.arange(packed.N, device=col.device), counts)
    sectors_per_row = (packed.X.shape[1] * es + 31) // 32
    sectors = torch.unique(rows * sectors_per_row + (col * es) // 32).numel()
    rows_with = int((counts > 0).sum())
    return dict(x_sectors=sectors, bytes=2 * 32 * sectors + 4 * m.n_missing + 8 * (packed.N + 1)
                + rows_with * R * es * 3, rows_with_missing=rows_with)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="c1,c2_slices")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_masked.py measures on a CUDA device; none found")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = card()
    lines = []
    for key in args.shapes.split(","):
        shape = SHAPES[key]
        packed, gen = make_data(shape, 0, dev)
        base = make_engine(packed, shape, None)
        for pname, frac, whole_rows in PATTERNS:
            mpacked = PackedMatrices(packed.X.clone(), packed.row_offsets, packed.K)
            mask = pack_mask_device(make_mask(mpacked, frac, whole_rows, gen), mpacked)
            eng = make_engine(mpacked, shape, mask)
            t_base, t_mask = [], []
            for _ in range(args.reps):  # alternate the arms
                t_base.append(time_steps(base, args.steps))
                t_mask.append(time_steps(eng, args.steps))
            m, R = eng.mask, shape["R"]
            Y = None if eng.fused_x1 else eng.Y
            out = torch.zeros(2, dtype=torch.float64, device=dev)
            # a refill with unchanged factors rewrites the same values: safe to repeat on the engine's state
            t_refill = event_time(lambda: _ops.mask_refill(mpacked.X, mpacked.N, mpacked.K, m.row_ptr, m.col, eng.gor,
                                                           eng.modes[0].x, eng.modes[1].x, eng.modes[2].x, Y, out,
                                                           eng.mask_ws), 20)
            Ytmp = torch.empty_like(eng.Y)
            t_y = event_time(lambda: _ops.xstream_y(mpacked.X, mpacked.N, mpacked.K, eng.modes[2].x, Ytmp, eng.ws,
                                                    eng.variant), 20)
            model = refill_bytes(m, mpacked, R)
            tb, tm = float(np.median(t_base)), float(np.median(t_mask))
            line = dict(shape=key, pattern=pname, card=name, power_limit=power, slices=shape["I"], rows=mpacked.N,
                        K=mpacked.K, R=R, n_missing=m.n_missing, graph=bool(eng.use_graph), fused_x1=eng.fused_x1,
                        step_unmasked_ms=tb * 1e3, step_masked_ms=tm * 1e3, step_ratio=tm / tb,
                        step_unmasked_ms_all=[t * 1e3 for t in t_base], step_masked_ms_all=[t * 1e3 for t in t_mask],
                        refill_ms=t_refill * 1e3, xstream_y_ms=t_y * 1e3, refill_over_xstream_y=t_refill / t_y,
                        refill_model_bytes=model["bytes"], refill_x_sectors=model["x_sectors"],
                        rows_with_missing=model["rows_with_missing"],
                        refill_model_gbps=model["bytes"] / t_refill / 1e9)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del eng, mpacked, mask
            torch.cuda.empty_cache()
        del base, packed
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=name, power_limit=power, steps=args.steps, reps=args.reps, results=lines), f, indent=1)


if __name__ == "__main__":
    main()
