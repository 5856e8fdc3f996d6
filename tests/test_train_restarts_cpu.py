"""Multi-start training on CPU: BatchAdam against spax.Adam, the example's --restarts loop with the device calls of
MultiStartSPR replaced by the oracle (test infrastructure only, as in test_train_loop_cpu), and the workspace size of the
batched loss + gradient."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import nngp_oracle as orc  # noqa: E402


def _example():
    import importlib.util
    spec = importlib.util.spec_from_file_location("regression_train", os.path.join(ROOT, "examples", "regression_train.py"))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    return ex


def _oracle_backed(model, kw_stack, poison=None):
    """patch the two device entry points of a MultiStartSPR with per-restart oracle evaluations (same contracts).
    poison: restarts whose loss, gradient and test NLL are NaN from the given step on (a non-PD kernel matrix)."""
    import torch
    calls = {"n": 0}

    def rows():
        return model.safe_values().cpu().numpy()

    def loss_and_grad():
        calls["n"] += 1
        h = rows()
        loss, grad = np.empty(len(h)), np.empty((len(h), 6))
        for r, v in enumerate(h):
            if poison and r in poison and calls["n"] >= poison[r]:
                loss[r], grad[r] = np.nan, np.nan
                continue
            loss[r], grad[r] = orc.spr_loss_grad(model.x_data.numpy(), model.y_data.numpy(), w_std=v[0], b_std=v[1],
                                                 last_w_std=v[2], eps=v[3], a=v[4], b=v[5], kind=model.kind, **kw_stack)
        g = torch.from_numpy(grad)
        g = torch.where(model.mask, g * torch.sigmoid(model.raw), torch.zeros_like(g))
        return torch.from_numpy(loss), g, torch.zeros(len(h), dtype=torch.int32)

    def test_nll(x, y):
        out = []
        for r, v in enumerate(rows()):
            if poison and r in poison and calls["n"] >= poison[r]:
                out.append(np.nan)
                continue
            out.append(orc.spr_test_nll(model.x_data.numpy(), model.y_data.numpy(), np.asarray(x), np.asarray(y),
                                        model.y_mean, model.y_std, w_std=v[0], b_std=v[1], last_w_std=v[2], eps=v[3],
                                        a=v[4], b=v[5], kind=model.kind, **kw_stack))
        return torch.tensor(out, dtype=torch.float64)

    model.loss_and_grad, model.test_nll = loss_and_grad, test_nll


def test_batch_adam_matches_adam_per_row():
    """Every element of a BatchAdam step is spax.Adam's on the same gradient sequence (to 1e-15), masked entries never
    move, and a NaN row stays in its row."""
    import torch
    from smnngp_b200.spax import Adam, BatchAdam, ConstraintTrainVar, positive
    rng = np.random.default_rng(3)
    r = 5
    starts = np.exp(rng.standard_normal((r, 6)))
    raw = torch.from_numpy(np.stack([[ConstraintTrainVar(v, constraint=positive()).value for v in row] for row in starts]))
    mask = np.array([True, True, True, True, False, False])            # Gaussian: alpha, beta are not variables
    opt = BatchAdam(raw, mask=mask)
    refs = [[ConstraintTrainVar(v, constraint=positive()) for v in row] for row in starts]
    ref_opts = [Adam({str(j): refs[i][j] for j in range(4)}) for i in range(r)]
    raw0 = raw.clone()
    for step in range(12):
        g = rng.standard_normal((r, 6)) * 10.0 ** rng.uniform(-8, 1, (r, 6))
        if step == 7:
            g[2, 1] = np.nan
        opt(0.05, torch.from_numpy(g))
        for i in range(r):
            ref_opts[i](0.05, {str(j): g[i, j] for j in range(4)})
    got = raw.numpy()
    for i in range(r):
        want = np.array([float(refs[i][j].value) for j in range(4)])
        if i == 2:
            assert np.isnan(got[i, :4]).sum() == 1 and np.isnan(got[i, 1]) and np.all(np.isnan(want) == np.isnan(got[i, :4]))
            ok = ~np.isnan(want)
            assert np.all(np.abs(got[i, :4][ok] - want[ok]) <= 1e-15 * np.maximum(1.0, np.abs(want[ok])))
        else:
            assert np.all(np.abs(got[i, :4] - want) <= 1e-15 * np.maximum(1.0, np.abs(want))), (i, got[i], want)
    assert np.array_equal(got[:, 4:], raw0.numpy()[:, 4:])              # masked columns never move
    # frozen rows keep their variables
    before = raw.clone()
    opt(0.05, torch.ones((r, 6), dtype=torch.float64), active=torch.tensor([True, False, True, True, False]))
    assert torch.equal(raw[1], before[1]) and torch.equal(raw[4], before[4]) and not torch.equal(raw[0], before[0])


@pytest.mark.parametrize("method", ["tp", "gp"])
def test_restart_loop_lowers_every_loss_and_reports_the_best(method):
    import torch
    ex = _example()
    args = ex.parse(["--method", method, "--rows", "60", "--features", "4", "--max-steps", "20", "--print-interval",
                     "10", "--valid-interval", "10", "--epsilon", "1e-3", "--b-std", "0.2", "-lr", "0.05",
                     "--restarts", "4", "--restart-scale", "0.3", "--num-hiddens", "2"])
    (x, y), valid, test, (y_std, y_mean) = ex.make_data(args.rows, 12, 12, args.features, args.seed)
    starts = ex.restart_starts(args)
    assert starts.shape == (4, 6)
    assert np.array_equal(starts[0], [args.w_std, args.b_std, args.last_w_std, args.epsilon, args.alpha, args.beta])
    assert np.all(starts[1:] != starts[0])
    model = ex.build_multistart(args, x, y, y_mean, y_std)
    assert model.raw.shape == (4, 6) and np.allclose(model.safe_values().numpy(), starts, rtol=1e-12)
    _oracle_backed(model, dict(num_hiddens=2, act="relu", arch="mlp"))
    l0, g0, _ = model.loss_and_grad()
    if method == "gp":
        assert torch.all(g0[:, 4:] == 0)
    lines = []
    k, best = ex.train_restarts(model, args, valid, test, log=lines.append)
    l1, _, _ = model.loss_and_grad()
    assert torch.all(l1 < l0), (l0, l1)
    if method == "gp":
        assert np.allclose(model.safe_values().numpy()[:, 4:], starts[:, 4:], rtol=1e-12)   # alpha, beta untouched
    assert 0 <= k < 4 and np.isfinite(best[1]) and best[0] % 10 == 0
    assert any("active" in s for s in lines)


def test_restart_loop_freezes_a_nan_restart():
    import torch
    ex = _example()
    args = ex.parse(["--rows", "60", "--features", "4", "--max-steps", "30", "--print-interval", "10",
                     "--valid-interval", "10", "--epsilon", "1e-3", "--b-std", "0.2", "-lr", "0.05", "--restarts", "3",
                     "--num-hiddens", "2"])
    (x, y), valid, test, (y_std, y_mean) = ex.make_data(args.rows, 12, 12, args.features, args.seed)
    model = ex.build_multistart(args, x, y, y_mean, y_std)
    _oracle_backed(model, dict(num_hiddens=2, act="relu", arch="mlp"), poison={1: 5})
    lines = []
    k, best = ex.train_restarts(model, args, valid, test, log=lines.append)
    raw = model.raw.numpy()
    assert np.all(np.isnan(raw[1]))                                   # its NaN gradient reached its own row only
    assert np.all(np.isfinite(raw[[0, 2]]))
    assert k != 1 and np.isfinite(best[1])
    # frozen at the first validation after the NaN; the other two go on to the last step
    assert [s for s in lines if "active)" in s] == [s for s in lines if "(2 of 3 restarts active)" in s] != []
    assert any(s.startswith("[   30] nll:") for s in lines)


@pytest.mark.parametrize("n,nh,arch", [(404, 3, 0), (1, 0, 0), (4096, 2, 1), (17, 64, 0)])
def test_lml_grad_batch_workspace_is_affine_in_slots(n, nh, arch):
    import smnngp_b200 as s
    lib = s._lib.load()
    one = lib.smnngp_lml_grad_batch_workspace_bytes(n, nh, arch, 1)
    assert one >= (2 * n + 1) * n * 8
    assert lib.smnngp_lml_grad_batch_workspace_bytes(n, nh, arch, 0) == 0
    for slots in (2, 7, 296):
        assert lib.smnngp_lml_grad_batch_workspace_bytes(n, nh, arch, slots) == slots * one
