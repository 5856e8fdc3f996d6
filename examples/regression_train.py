"""The reference's regression training loop (experiments/regression/train.py:61-67, :126-228) on the B200 path:
same model construction, same Adam-on-softplus-variables loop, same NaN stop - every step is ONE fused CUDA call
(`SPR.loss_and_grad` -> smnngp_lml_grad_f64) instead of reverse-mode AD through JAX.

    python examples/regression_train.py --method tp --num-hiddens 3 --max-steps 200

On several GPUs (one process per GPU; every step is one smnngp_lml_grad_mg_f64 call per rank):

    torchrun --standalone --nproc-per-node 2 examples/regression_train.py --distributed --rows 20000 --max-steps 50

Many restarts at once (N <= 4096: every step evaluates all of them in one smnngp_lml_grad_batch_f64 launch):

    python examples/regression_train.py --rows 404 --features 13 --restarts 296 --restart-scale 0.5

Synthetic UCI-shaped data (no dataset download in this environment); swap `make_data` for the reference's
`get_dataset` / `split_dataset` (experiments/regression/data.py) to reproduce its runs."""
import argparse
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def make_data(n_train, n_valid, n_test, d, seed):
    from tests.synth import regression_data
    x, y, xr, yr, ym, ys = regression_data(n_train, d, t=n_valid + n_test, seed=seed)
    return (x, y), (xr[:n_valid], yr[:n_valid]), (xr[n_valid:], yr[n_valid:]), (ys, ym)


def build_model(args, x_train, y_train, y_mean, y_std):
    import smnngp_b200 as sm
    from smnngp_b200.spax import NNGPKernel, GaussianLikelihood, StudentTLikelihood, SPR
    base = {"mlp": sm.get_mlp_kernel, "resnet": sm.get_dense_resnet_kernel}[args.network]   # train.py:118-124

    def get_kernel_fn(w_std, b_std, last_w_std):
        return base(args.num_hiddens, act=args.activation, w_std=w_std, b_std=b_std, last_w_std=last_w_std)

    kernel = NNGPKernel(get_kernel_fn, args.w_std, args.b_std, args.last_w_std)            # train.py:126
    lik = StudentTLikelihood(args.alpha, args.beta) if args.method == "tp" else GaussianLikelihood()
    if getattr(args, "distributed", False):
        from smnngp_b200.spax import DistributedSPR
        return DistributedSPR(kernel, lik, x_train, y_train, y_mean, y_std, eps=args.epsilon)
    return SPR(kernel, lik, x_train, y_train, y_mean, y_std, eps=args.epsilon)             # train.py:137-142


def restart_starts(args):
    """[R, 6] safe values {w_std, b_std, last_w_std, eps, alpha, beta}: restart 0 is the command line, restart k > 0
    multiplies each of them by exp(s N(0, 1)), drawn from --seed."""
    base = np.array([args.w_std, args.b_std, args.last_w_std, args.epsilon, args.alpha, args.beta], dtype=np.float64)
    rng = np.random.default_rng(args.seed)
    starts = np.tile(base, (args.restarts, 1))
    starts[1:] *= np.exp(args.restart_scale * rng.standard_normal((args.restarts - 1, 6)))
    return starts


def build_multistart(args, x_train, y_train, y_mean, y_std):
    import smnngp_b200 as sm
    from smnngp_b200.spax import NNGPKernel, GaussianLikelihood, StudentTLikelihood, MultiStartSPR
    base = {"mlp": sm.get_mlp_kernel, "resnet": sm.get_dense_resnet_kernel}[args.network]

    def get_kernel_fn(w_std, b_std, last_w_std):
        return base(args.num_hiddens, act=args.activation, w_std=w_std, b_std=b_std, last_w_std=last_w_std)

    kernel = NNGPKernel(get_kernel_fn, args.w_std, args.b_std, args.last_w_std)
    lik = StudentTLikelihood(args.alpha, args.beta) if args.method == "tp" else GaussianLikelihood()
    return MultiStartSPR(kernel, lik, x_train, y_train, y_mean, y_std, starts=restart_starts(args))


def train_restarts(model, args, valid, test, log=print):
    """``train`` for every restart of a MultiStartSPR at once: one batched value + gradient call and one BatchAdam step
    per iteration.  A restart whose validation NLL is NaN is frozen (train.py:211's stop, per restart); the others go
    on.  Returns (best restart, (step, valid NLL, test NLL)) by validation NLL."""
    import torch
    from smnngp_b200.spax import BatchAdam
    opt = BatchAdam(model.raw, mask=model.mask)
    lr = args.learning_rate
    r = model.raw.shape[0]
    active = torch.ones(r, dtype=torch.bool, device=model.raw.device)
    valid_nll, test_nll = model.test_nll(*valid).cpu().numpy(), model.test_nll(*test).cpu().numpy()
    best = [(0, float(valid_nll[k]), float(test_nll[k])) for k in range(r)]
    log(f"[{0:5d}] {r} restarts  best NLL: {np.nanmin(valid_nll):.5f}")
    for i in range(1, args.max_steps + 1):
        loss, grad, _ = model.loss_and_grad()
        opt(lr, grad, active=active)
        if i % args.print_interval == 0:
            ls = loss.cpu().numpy()[active.cpu().numpy()]
            log(f"[{i:5d}] nll: {np.nanmin(ls) if ls.size else float('nan'):.5f} (best of {ls.size} active restarts)")
        if i % args.valid_interval == 0:
            valid_nll, test_nll = model.test_nll(*valid).cpu().numpy(), model.test_nll(*test).cpu().numpy()
            act = active.cpu().numpy()
            for k in np.flatnonzero(act):
                if math.isnan(valid_nll[k]):
                    act[k] = False
                elif not valid_nll[k] >= best[k][1]:
                    best[k] = (i, float(valid_nll[k]), float(test_nll[k]))
            active = torch.as_tensor(act, device=model.raw.device)
            log(f"[{i:5d}] NLL: {np.nanmin(valid_nll[act]) if act.any() else float('nan'):.5f}  "
                f"({int(act.sum())} of {r} restarts active)")
            if not act.any():
                break
    vals = np.array([b[1] for b in best])
    k = int(np.nanargmin(vals)) if np.isfinite(vals).any() else 0
    return k, best[k]


def train(model, args, valid, test, log=print):
    from smnngp_b200.spax import Adam
    opt = Adam(model.vars())
    lr = args.learning_rate
    valid_nll, test_nll = float(model.test_nll(*valid)), float(model.test_nll(*test))
    log(f"[{0:5d}] NLL: {valid_nll:.5f}  TEST: {test_nll:.5f}")
    best = (0, valid_nll, test_nll)
    for i in range(1, args.max_steps + 1):
        loss, grads = model.loss_and_grad()            # value + gradients w.r.t. the unconstrained variables
        opt(lr, grads)
        if i % args.print_interval == 0:
            ws, bs, ls = model.kernel.get_params()
            log(f"[{i:5d}] nll: {loss:.5f}  ws: {ws:.4f}  bs: {bs:.3E}  ls: {ls:.4f}  e: {model.eps.safe_value:.3E}")
        if i % args.valid_interval == 0:
            valid_nll, test_nll = float(model.test_nll(*valid)), float(model.test_nll(*test))
            log(f"[{i:5d}] NLL: {valid_nll:.5f}  TEST: {test_nll:.5f}")
            if math.isnan(valid_nll):                  # train.py:211: a non-PD kernel matrix yields NaN, never raises
                break
            if valid_nll < best[1]:
                best = (i, valid_nll, test_nll)
    return best


def parse(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("-m", "--method", choices=["gp", "tp"], default="tp")
    p.add_argument("-n", "--network", choices=["mlp", "resnet"], default="mlp")
    p.add_argument("-nh", "--num-hiddens", type=int, default=3)
    p.add_argument("-act", "--activation", choices=["relu", "erf"], default="relu")
    p.add_argument("-ws", "--w-std", type=float, default=1.0)
    p.add_argument("-bs", "--b-std", type=float, default=1e-8)
    p.add_argument("-ls", "--last-w-std", type=float, default=1.0)
    p.add_argument("-e", "--epsilon", type=float, default=1e-6)
    p.add_argument("-a", "--alpha", type=float, default=2.0)
    p.add_argument("-b", "--beta", type=float, default=2.0)
    p.add_argument("-lr", "--learning-rate", type=float, default=1e-2)
    p.add_argument("-t", "--max-steps", type=int, default=200)
    p.add_argument("-pi", "--print-interval", type=int, default=20)
    p.add_argument("-vi", "--valid-interval", type=int, default=50)
    p.add_argument("-s", "--seed", type=int, default=10)
    p.add_argument("--rows", type=int, default=4000)
    p.add_argument("--features", type=int, default=8)
    p.add_argument("--distributed", action="store_true", help="under torchrun: shard every step over the ranks' GPUs")
    p.add_argument("--restarts", type=int, default=1, help="train this many restarts at once (N <= 4096: one launch)")
    p.add_argument("--restart-scale", type=float, default=0.5, help="restart k > 0 scales each start by exp(s N(0,1))")
    return p.parse_args(argv)


def main(argv=None):
    args = parse(argv)
    (x, y), valid, test, (y_std, y_mean) = make_data(args.rows, args.rows // 8, args.rows // 8, args.features, args.seed)
    log = print
    if args.distributed:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
        dist.init_process_group("nccl", device_id=dev)
        to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        x, y, valid, test = to_dev(x), to_dev(y), tuple(map(to_dev, valid)), tuple(map(to_dev, test))
        if dist.get_rank() != 0:
            log = lambda *a, **k: None
    if args.restarts > 1:
        if args.distributed:
            raise SystemExit("--restarts runs on one GPU")
        model = build_multistart(args, x, y, y_mean, y_std)
        k, best = train_restarts(model, args, valid, test, log=log)
        log(f"best restart {k}: [{best[0]:5d}] NLL: {best[1]:.5f}  TEST: {best[2]:.5f}")
        return
    model = build_model(args, x, y, y_mean, y_std)
    best = train(model, args, valid, test, log=log)
    log(f"[{best[0]:5d}] NLL: {best[1]:.5f}  TEST: {best[2]:.5f}")
    if args.distributed:
        model.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
