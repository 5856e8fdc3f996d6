"""Batched grid search against the per-point loop (GridSearch.points vs GridSearch.point), one B200.

For each shape (N, T, D) of the UCI sizes the reference's find.py runs on and each grid size G, both paths evaluate the
same G seeded (w_std, b_std, eps) points on the same tests.synth.regression_data inputs.  The loop is synchronised
once at its end.  Warm-up: one full pass of each path; then CUDA events around `reps` passes.  Every row reports ms per
batch, points/s, the achieved TFLOP/s against the per-point model 2 (N^3/3 + N^2 (T + 1)) + recursion entries x layers,
and the largest relative difference between the two paths (mean and var relative to their largest magnitude, logdet
and quad relative to themselves).  The first line holds the card's name and power limit, read in the same run.

    python profiles/grid_batch_bench.py [--out FILE] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import smnngp_b200 as sm                                  # noqa: E402
from smnngp_b200 import device as dv                      # noqa: E402
from tests.synth import regression_data                   # noqa: E402

SHAPES = [(404, 52, 13), (824, 103, 8), (2048, 256, 8), (4096, 512, 8)]
GRIDS = [1, 11, 148, 1100]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (v.strip() for v in q[0].split(","))
    return dict(card=name, power_limit=power, max_sm_clock=clk, sms=torch.cuda.get_device_properties(0).multi_processor_count)


def hp_grid(g, seed=5):
    rng = np.random.default_rng(seed)
    w, b, e = rng.uniform(0.5, 2.0, g), rng.uniform(0.01, 1.0, g), 10.0 ** rng.uniform(-4, -2, g)
    return torch.stack([dv.make_hp(w[i], b[i], 1.0, e[i]) for i in range(g)])


def model_flop(n, t, n_act):
    recursion = (2 * n * (n + 1) // 2 + t * n) * n_act       # entries evaluated per point x layer applications
    return 2.0 * (n ** 3 / 3.0 + n * n * (t + 1)) + recursion


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        res = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps, res


def loop(gs, hps):
    return [gs.point(hps[i]) for i in range(hps.shape[0])]


RULE = dv._batch_wins            # what points() picks; the measurement times both paths at every workload


def batch(gs, hps):
    dv._batch_wins = lambda n, g: True
    try:
        return gs.points(hps)
    finally:
        dv._batch_wins = RULE


def max_rel_diff(rows, b):
    mean = torch.stack([r[0] for r in rows]); var = torch.stack([r[1] for r in rows])
    ld = torch.stack([r[2] for r in rows]); qd = torch.stack([r[3] for r in rows])
    return max(((b[0] - mean).abs().max() / mean.abs().max()).item(), ((b[1] - var).abs().max() / var.abs().max()).item(),
               ((b[2] - ld).abs() / ld.abs()).max().item(), ((b[3] - qd).abs() / qd.abs()).max().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="Boston shape only (rehearsal)")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    sm._lib.load()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    runs = [(s, "relu", 3) for s in SHAPES] + [(SHAPES[0], "erf", 3)]
    for (n, t, d), act, L in runs[:1] if a.quick else runs:
        x, y, xt, *_ = regression_data(n, d, t=t)
        spec = sm.StackSpec(L, act, "mlp")
        gs = dv.GridSearch(*(torch.from_numpy(v).cuda() for v in (x, y, xt)), spec=spec)
        for g in GRIDS:
            hps = hp_grid(g)
            reps = 3 if n * g <= 824 * 148 else 1
            t_loop, rows = timed(lambda: loop(gs, hps), reps)
            t_batch, b = timed(lambda: batch(gs, hps), reps)
            infos = torch.cat([r[4] for r in rows])
            flop = model_flop(n, t, L) * g
            row = dict(N=n, T=t, D=d, act=act, L=L, G=g, reps=reps, loop_ms=round(t_loop, 3), batch_ms=round(t_batch, 3),
                       loop_points_per_s=round(g / t_loop * 1e3, 1), batch_points_per_s=round(g / t_batch * 1e3, 1),
                       speedup=round(t_loop / t_batch, 2), loop_tflops=round(flop / t_loop * 1e-9, 4),
                       batch_tflops=round(flop / t_batch * 1e-9, 4), model_flop_per_point=model_flop(n, t, L),
                       max_rel_diff=max_rel_diff(rows, b), failed_points=int((infos != 0).sum().item()),
                       batch_info_equal=bool(torch.equal(infos, b[4])),
                       points_picks="batch" if RULE(n, g) else "loop")
            lines.append(row)
            print(json.dumps(row), flush=True)
        del gs
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
