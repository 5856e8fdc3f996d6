"""Time the importance-sampling table of GridSearch.mixture (scale draws + one mixture launch) on the GPU against the
NumPy estimator on the host, and write one JSON line per shape.

The table has G * P * S * T log-density terms, each one FMA and one exp, plus G * P * S evidence terms; terms/s below is
that count (TERMS, kept here) over the time of the draw and mixture launches, taken with CUDA events after warm-up.  The
grid points come from GridSearch.points on synthetic UCI-shaped data; they are not part of the timed window.  The host
rate is measured on the first few grid points only (the whole table would take minutes in NumPy) and the parity column
compares the GPU table with the NumPy estimator on those points.

    python profiles/mixture_bench.py [--out profiles/r05_mixture.jsonl] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (N, T, G, P, S): Boston size (the reference's find.py grid: 1 100 points, a 10 x 10 prior table, 1 000 draws) and the
# largest N of the batched grid search with 148 points (one per SM)
SHAPES = [(404, 52, 1100, 100, 1000), (4096, 512, 148, 100, 1000)]
HOST_POINTS = 2


def TERMS(G, P, S, T):
    return G * P * S * (T + 1)


def card():
    import torch
    r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return torch.cuda.get_device_name(0), (r.stdout.strip() if r.returncode == 0 else "unknown")


def run(shape, reps):
    import torch
    import smnngp_b200 as sm
    from tests import mixture_ref as mr
    from tests.synth import regression_data
    n, t, g, p, s = shape
    x, y, xt, yt, ym, ys = regression_data(n, 13, t=t)
    dev = torch.device("cuda", 0)
    gs = sm.device.GridSearch(*(torch.from_numpy(v).to(dev) for v in (x, y, xt)), spec=sm.StackSpec(3, "relu", "mlp"))
    rng = np.random.default_rng(0)
    hps = torch.stack([sm.make_hp(w, b, 1.0, e, device=dev) for w, b, e in
                       zip(rng.uniform(0.5, 2.0, g), rng.uniform(0.01, 1.0, g), 10.0 ** rng.uniform(-4, -2, g))])
    mean, var, logdet, quad, info = gs.points(hps)
    scal = torch.stack([0.5 * logdet, quad], 1)
    a, b = np.meshgrid(np.linspace(0.5, 5.0, 10), np.linspace(0.5, 5.0, 10))   # a 10 x 10 (c, k) table
    params = torch.from_numpy(np.stack([a.ravel(), b.ravel()], 1)[:p].copy()).to(dev)
    ytd = torch.from_numpy(yt).to(dev)

    def table():
        draws = sm.device.scale_draws("burr12", params, s, seed=1)
        return sm.device.mixture_nll(scal, mean, var, ytd, n, draws, ym, ys)

    for _ in range(3):
        out = table()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        table()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    nll, lml, ess, _ = out
    draws = sm.device.scale_draws("burr12", params, s, seed=1).cpu().numpy()
    k = min(HOST_POINTS, g)
    t0 = time.perf_counter()
    rn, rl, re, _ = mr.mixture_nll(scal[:k].cpu().numpy(), mean[:k].cpu().numpy(), var[:k].cpu().numpy(), yt, n,
                                    draws, ym, ys)
    host_s = time.perf_counter() - t0
    diff = max(float(np.max(np.abs(a_[:k].cpu().numpy() - r_) / np.maximum(1.0, np.abs(r_))))
               for a_, r_ in ((nll, rn), (lml, rl), (ess, re)))
    terms = TERMS(g, p, s, t)
    return dict(N=n, T=t, G=g, P=p, S=s, terms=terms, gpu_ms=ms, gpu_terms_per_s=terms / (ms * 1e-3),
                host_points=k, host_s=host_s, host_terms_per_s=TERMS(k, p, s, t) / host_s,
                speedup=(terms / (ms * 1e-3)) / (TERMS(k, p, s, t) / host_s),
                max_rel_diff_vs_numpy=diff, failed_points=int((info != 0).sum()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_mixture.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mixture_bench needs a CUDA device")
    name, power = card()
    with open(args.out, "w") as f:
        for shape in SHAPES:
            rec = dict(run(shape, args.reps), gpu=name, power_limit=power, family="burr12")
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
