"""Batched loss + gradient against the per-call loop (LossGradBatch.points vs lml_grad), one B200.

For each shape (N, D) of the UCI sizes the reference's train.py runs on and each batch size G, both paths evaluate the
same G seeded hyper-parameter points (Student-t) on the same tests.synth.regression_data inputs.  The loop is
synchronised once at its end.  Warm-up: one call of each path on the first point; then CUDA events around one pass
(three where a pass is short).  Every row reports ms per batch, points/s, the achieved TFLOP/s against the per-point
model N^3 + recursion entries x layers (N^3/3 flop each for the factorisation, its carried identity and the SYRK; the
value and the dual pass over the lower triangle), and the largest relative difference between the two
paths per component (each component relative to itself, with a floor of 1e-12 of the largest in its row).  The first
line holds the card's name and power limit, read in the same run.

    python profiles/grad_batch_bench.py [--out FILE] [--quick]
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

SHAPES = [(404, 13), (824, 8), (2048, 8), (4096, 8)]
BATCHES = [1, 11, 148, 1100]
COMPONENTS = ("log_p", "loss", "sum_log_L", "quad", "g_w_std", "g_b_std", "g_last_w_std", "g_eps", "g_alpha", "g_beta")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (v.strip() for v in q[0].split(","))
    return dict(card=name, power_limit=power, max_sm_clock=clk, sms=torch.cuda.get_device_properties(0).multi_processor_count)


def hp_rows(g, seed=5):
    rng = np.random.default_rng(seed)
    h = np.stack([rng.uniform(0.5, 2.0, g), rng.uniform(0.01, 1.0, g), rng.uniform(0.5, 1.5, g),
                  10.0 ** rng.uniform(-4, -2, g), rng.uniform(1.5, 4.0, g), rng.uniform(0.5, 3.0, g)], axis=1)
    return torch.from_numpy(np.ascontiguousarray(h)).cuda()


def model_flop(n, n_act):
    return float(n) ** 3 + 2.0 * (n * (n + 1) // 2) * n_act


def timed(fn, warm, reps):
    warm()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        res = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps, res


RULE = dv._grad_batch_wins       # what points() picks; the measurement times both paths at every workload


def loop(lgb, hps):
    rows = [dv.lml_grad(lgb.x, lgb.y, spec=lgb.spec, hp=hps[i], kind="student_t") for i in range(hps.shape[0])]
    return torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows]), torch.cat([r[2] for r in rows])


def batch(lgb, hps):
    dv._grad_batch_wins = lambda n, g: True
    try:
        return lgb.points(hps, "student_t")
    finally:
        dv._grad_batch_wins = RULE


def max_rel_diff(a, b):
    ref = torch.cat([a[0], a[1]], 1)
    got = torch.cat([b[0], b[1]], 1)
    floor = 1e-12 * ref.abs().amax(1, keepdim=True)
    d = ((got - ref).abs() / torch.maximum(ref.abs(), floor)).amax(0).cpu().numpy()
    return {k: float(v) for k, v in zip(COMPONENTS, d)}


def train_wall(restarts, rows, features, steps):
    """wall time of examples/regression_train.py at one setting, in its own process, start-up included (what a user
    waits for)"""
    import time
    ex = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "regression_train.py")
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, ex, "--rows", str(rows), "--features", str(features), "--max-steps", str(steps),
                        "--restarts", str(restarts)], capture_output=True, text=True)
    wall = time.perf_counter() - t0
    return dict(example="regression_train.py", rows=rows, features=features, max_steps=steps, restarts=restarts,
                wall_s=round(wall, 2), returncode=r.returncode, last_line=(r.stdout.strip().splitlines() or [""])[-1],
                stderr_tail=r.stderr.strip()[-300:] if r.returncode else "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="Boston shape only (rehearsal)")
    ap.add_argument("--train-steps", type=int, default=1000)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    sm._lib.load()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    runs = [(s, "relu", 3) for s in SHAPES] + [(SHAPES[0], "erf", 3)]
    for (n, d), act, L in runs[:1] if a.quick else runs:
        x, y, *_ = regression_data(n, d)
        spec = sm.StackSpec(L, act, "mlp")
        lgb = dv.LossGradBatch(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), spec=spec)
        for g in BATCHES:
            hps = hp_rows(g)
            reps = 3 if n * g <= 824 * 148 else 1
            t_loop, lo = timed(lambda: loop(lgb, hps), lambda: loop(lgb, hps[:1]), reps)
            t_batch, b = timed(lambda: batch(lgb, hps), lambda: batch(lgb, hps[:1]), reps)
            flop = model_flop(n, L) * g
            row = dict(N=n, D=d, act=act, L=L, G=g, reps=reps, loop_ms=round(t_loop, 3), batch_ms=round(t_batch, 3),
                       loop_points_per_s=round(g / t_loop * 1e3, 1), batch_points_per_s=round(g / t_batch * 1e3, 1),
                       speedup=round(t_loop / t_batch, 2), loop_tflops=round(flop / t_loop * 1e-9, 4),
                       batch_tflops=round(flop / t_batch * 1e-9, 4), model_flop_per_point=model_flop(n, L),
                       max_rel_diff=max_rel_diff(lo, b), failed_points=int((lo[2] != 0).sum().item()),
                       batch_info_equal=bool(torch.equal(lo[2], b[2])), points_picks="batch" if RULE(n, g) else "loop")
            lines.append(row)
            print(json.dumps(row), flush=True)
        del lgb
        torch.cuda.empty_cache()
    if not a.quick:
        for r in (1, 296):
            row = train_wall(r, 404, 13, a.train_steps)
            lines.append(row)
            print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
