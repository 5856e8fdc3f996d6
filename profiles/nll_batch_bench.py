"""Batched test NLL against the per-point loop (GridSearch.test_nll batched vs one test_nll call per point), one B200.

For each shape (N, T) of the UCI sizes the reference's train.py runs on and each batch size G, both paths evaluate the
same G seeded hyper-parameter points on the same tests.synth.regression_data inputs (Student-t; a Gaussian row and an
erf row at Boston size).  Each path is forced in turn by replacing device._batch_wins, so every workload times both.
One untimed pass of each path gives the launch count (smnngp_instr_launches) and the outputs compared; then CUDA events
around one pass (three where a pass is short), after a warm-up on the first point.  Every row reports ms per call,
points/s, the achieved TFLOP/s against the per-point model 2N^3/3 + N^2 (T + 2) flop (N^3/3 + N^2 (T + 1) under
Gaussian: no second factorisation) plus 2 flop per recursion entry and layer (two N(N+1)/2 Grams and the T x N cross
Gram; one Gram under Gaussian), the largest relative difference of nll, mean and var between the paths (mean and var
relative to their largest magnitude in the row), and the path the rule picks.

Then examples/regression_train.py's train_restarts at Boston size with 296 restarts, in this process: the rule forced
to the loop and to the batch, alternating, each run from the same starts; and the time of one validation (the
validation and test NLL of every restart) on each path.  The first line holds the card's name, power limit and SM count,
read in the same run.

    python profiles/nll_batch_bench.py [--out FILE] [--quick]
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
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import smnngp_b200 as sm                                  # noqa: E402
from smnngp_b200 import device as dv                      # noqa: E402
from tests.synth import regression_data                   # noqa: E402

SHAPES = [(404, 52, 13), (824, 103, 8), (2048, 256, 8), (4096, 512, 8)]
BATCHES = [1, 11, 148, 296, 1100]
RULE = dv._batch_wins            # what GridSearch.test_nll picks; the measurement times both paths at every workload
Y_MEAN, Y_STD = 0.37, 1.9


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


def model_flop(n, t, n_act, kind):
    tri = n * (n + 1) // 2
    if kind == "student_t":
        return 2.0 * n ** 3 / 3 + float(n) ** 2 * (t + 2) + 2.0 * (2 * tri + t * n) * n_act
    return float(n) ** 3 / 3 + float(n) ** 2 * (t + 1) + 2.0 * (tri + t * n) * n_act


def forced(batch):
    def set_rule():
        dv._batch_wins = (lambda n, g: True) if batch else (lambda n, g: False)
    return set_rule


def run(gs, hps, yt, kind, batch):
    forced(batch)()
    try:
        return gs.test_nll(hps, yt, Y_MEAN, Y_STD, kind)
    finally:
        dv._batch_wins = RULE


def timed(fn, warm, reps):
    warm()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def launches(fn):
    lib = sm._lib.load()
    torch.cuda.synchronize()
    lib.smnngp_instr_reset(0)
    res = fn()
    torch.cuda.synchronize()
    return res, int(lib.smnngp_instr_launches())


def max_rel_diff(a, b):
    nll = ((b[0] - a[0]).abs() / a[0].abs()).max().item()
    mean = ((b[1] - a[1]).abs().amax(1) / a[1].abs().amax(1)).max().item()
    var = ((b[2] - a[2]).abs().amax(1) / a[2].abs().amax(1)).max().item()
    return dict(nll=nll, mean=mean, var=var)


def workload(n, t, d, act, L, kind, g, gs, yt):
    hps = hp_rows(g)
    lo, loop_launches = launches(lambda: run(gs, hps, yt, kind, False))
    b, batch_launches = launches(lambda: run(gs, hps, yt, kind, True))
    reps = 3 if n * g <= 824 * 148 else 1
    t_loop = timed(lambda: run(gs, hps, yt, kind, False), lambda: run(gs, hps[:1], yt, kind, False), reps)
    t_batch = timed(lambda: run(gs, hps, yt, kind, True), lambda: run(gs, hps[:1], yt, kind, True), reps)
    flop = model_flop(n, t, L, kind) * g
    return dict(N=n, T=t, D=d, act=act, L=L, kind=kind, G=g, reps=reps, loop_ms=round(t_loop, 3),
                batch_ms=round(t_batch, 3), loop_points_per_s=round(g / t_loop * 1e3, 1),
                batch_points_per_s=round(g / t_batch * 1e3, 1), speedup=round(t_loop / t_batch, 2),
                loop_tflops=round(flop / t_loop * 1e-9, 4), batch_tflops=round(flop / t_batch * 1e-9, 4),
                model_flop_per_point=model_flop(n, t, L, kind), loop_launches=loop_launches,
                batch_launches=batch_launches, max_rel_diff=max_rel_diff(lo, b),
                failed_points=int((lo[3] != 0).sum().item()), batch_info_equal=bool(torch.equal(lo[3], b[3])),
                rule_picks="batch" if RULE(n, g) else "loop")


def training(steps, reps):
    """train_restarts of examples/regression_train.py, 296 restarts at Boston size, both paths alternating"""
    import regression_train as rt
    args = rt.parse(["--rows", "404", "--features", "13", "--restarts", "296", "--max-steps", str(steps)])
    (x, y), valid, test, (y_std, y_mean) = rt.make_data(args.rows, args.rows // 8, args.rows // 8, args.features,
                                                        args.seed)
    rows = []
    for rep in range(reps):
        for batch in (False, True):
            model = rt.build_multistart(args, x, y, y_mean, y_std)
            forced(batch)()
            try:
                model.test_nll(*valid)                   # warm-up of this path (module load, first workspace)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    model.test_nll(*valid).cpu()
                    model.test_nll(*test).cpu()
                val_ms = (time.perf_counter() - t0) / 3 * 1e3
                model = rt.build_multistart(args, x, y, y_mean, y_std)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                k, best = rt.train_restarts(model, args, valid, test, log=lambda *a, **kw: None)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
            finally:
                dv._batch_wins = RULE
            n_val = 1 + steps // args.valid_interval
            row = dict(example="regression_train.train_restarts", rows=404, features=13, restarts=296, max_steps=steps,
                       valid_interval=args.valid_interval, rep=rep, path="batch" if batch else "loop",
                       wall_s=round(wall, 3), validation_ms=round(val_ms, 2), validations=n_val,
                       validation_share=round(n_val * val_ms * 1e-3 / wall, 3), best_restart=k,
                       best=[best[0], best[1], best[2]])
            rows.append(row)
            print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="Boston shape only, short training (rehearsal)")
    ap.add_argument("--train-steps", type=int, default=200)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    sm._lib.load()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    runs = [(s, "relu", 3, "student_t") for s in SHAPES]
    runs += [(SHAPES[0], "relu", 3, "gauss"), (SHAPES[0], "erf", 3, "student_t")]
    for (n, t, d), act, L, kind in runs[:1] if a.quick else runs:
        x, y, xt, yt, *_ = regression_data(n, d, t=t)
        gs = dv.GridSearch(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(xt).cuda(),
                           spec=sm.StackSpec(L, act, "mlp"))
        ytd = torch.from_numpy(yt).cuda()
        for g in BATCHES[:2] if a.quick else BATCHES:
            row = workload(n, t, d, act, L, kind, g, gs, ytd)
            lines.append(row)
            print(json.dumps(row), flush=True)
        del gs
        torch.cuda.empty_cache()
    lines += training(20 if a.quick else a.train_steps, 1 if a.quick else 2)
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
