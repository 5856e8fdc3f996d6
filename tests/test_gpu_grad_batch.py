"""Batched loss and gradient (smnngp_lml_grad_batch_f64 / LossGradBatch.points / MultiStartSPR): SPR.loss and its
six-scalar gradient at many points in one launch.  Parity with the oracle, the mpmath goldens and the per-call
lml_grad / lml, finite differences at N = 4096, bit-exact independence of a point from the rest of its batch, failure
isolation, argument checks, one launch, graph capture, the per-call fallback, and multi-start training.

Tolerances: against the oracle those of test_gpu_grad (loss 1e-8, every gradient component GRAD_TOL relative to itself
plus 1e-12 of the largest).  Against the per-call path AGREE_TOL: both factor the same matrix, with different blocking
and summation order, and the gradient contracts the explicit inverse of K + eps I, so both carry ~cond * 2^-53 relative
error (cond up to ~1e8 at eps = 1e-6); measured on a B200 the worst component differs by ~1e-10 (printed by the test)."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import nngp_oracle as orc
from tests.synth import regression_data, DEFAULT_HP

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOSS_TOL = 1e-8
GRAD_TOL = 1e-7
AGREE_TOL = 1e-8
NAMES = ("w_std", "b_std", "last_w_std", "eps", "alpha", "beta")
KIND = {"gauss": 0, "student_t": 1}
EINVAL, EWORKSPACE = 1, 3


@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


def _close(got, ref, tol):
    return np.abs(got - ref) <= tol * np.abs(ref) + 1e-12 * np.abs(ref).max()


def _hp_vec(hp):
    return np.array([hp[k] for k in NAMES], dtype=np.float64)


def _batch(sm, x, y, L, act, arch):
    import torch
    return sm.device.LossGradBatch(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), spec=sm.StackSpec(L, act, arch))


def _cabi(sm, lgb, hps, slots, kind):
    """smnngp_lml_grad_batch_f64 with a workspace of exactly `slots` slots -> host (out, grad, info)."""
    import torch
    lib = sm._lib.load()
    nh, act, arch = lgb.spec.ids()
    g, dev = hps.shape[0], lgb.y.device
    out = torch.empty((g, 4), dtype=torch.float64, device=dev)
    grad = torch.empty((g, 6), dtype=torch.float64, device=dev)
    info = torch.empty(g, dtype=torch.int32, device=dev)
    nbytes = lib.smnngp_lml_grad_batch_workspace_bytes(lgb.n, nh, arch, slots)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    rc = lib.smnngp_lml_grad_batch_f64(C.c_void_p(torch.cuda.current_stream().cuda_stream), lgb.k0dd.data_ptr(), lgb.ld0,
                                       lgb.q_d.data_ptr(), lgb.y.data_ptr(), lgb.n, g, nh, act, arch, hps.data_ptr(),
                                       KIND[kind], ws.data_ptr(), nbytes, out.data_ptr(), grad.data_ptr(),
                                       info.data_ptr())
    assert rc == 0, lib.smnngp_last_error()
    return _host((out, grad, info))


def _host(res):
    return tuple(r.cpu().numpy() for r in res)


def _same_bits(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def _rows(res, idx):
    return tuple(r[idx] for r in res)


def _random_hps(g, seed=5, kind_t=True):
    import torch
    rng = np.random.default_rng(seed)
    h = np.stack([rng.uniform(0.5, 2.0, g), rng.uniform(0.01, 1.0, g), rng.uniform(0.5, 1.5, g),
                  10.0 ** rng.uniform(-4, -2, g), rng.uniform(1.5, 4.0, g), rng.uniform(0.5, 3.0, g)], axis=1)
    return torch.from_numpy(np.ascontiguousarray(h)).cuda()


# ---- parity ---------------------------------------------------------------------------------------------------------
SHAPES = [(506, 13, 3, "relu", "mlp", "student_t", {}), (404, 8, 4, "erf", "mlp", "student_t", dict(b_std=0.3)),
          (1300, 8, 2, "relu", "resnet", "student_t", dict(b_std=0.2, w_std=1.3, last_w_std=0.8)),
          (700, 16, 1, "erf", "resnet", "gauss", dict(b_std=0.4)),
          (2600, 8, 3, "relu", "mlp", "student_t", dict(alpha=3.0, beta=1.5)),
          (77, 5, 2, "relu", "mlp", "gauss", dict(eps=1e-3)), (1, 4, 2, "relu", "mlp", "student_t", dict(eps=1e-2)),
          (129, 6, 0, "relu", "mlp", "student_t", dict(eps=1e-2)),
          (4096, 8, 3, "relu", "mlp", "student_t", dict(b_std=0.2, eps=1e-3))]


@pytest.mark.parametrize("n,d,L,act,arch,kind,over", SHAPES)
def test_batch_matches_oracle_and_lml_grad(sm, n, d, L, act, arch, kind, over):
    """A small (w_std, b_std, eps) grid around each shape of test_gpu_grad::test_grad_parity through the C-ABI: against
    the oracle, and every point against the per-call lml_grad (gradient) and lml (value)."""
    import torch
    x, y, *_ = regression_data(n, d)
    base = dict(DEFAULT_HP, **over)
    pts = []
    for w in (1.0, 1.25):
        for b in (1.0, 1.6):
            for e in (1.0, 10.0):
                pts.append(dict(base, w_std=base["w_std"] * w, b_std=base["b_std"] * b, eps=base["eps"] * e))
    if n >= 4096:
        pts = [pts[0], pts[3], pts[6]]
    elif n >= 1300:
        pts = pts[::2]
    hps = torch.from_numpy(np.stack([_hp_vec(h) for h in pts])).cuda()
    lgb = _batch(sm, x, y, L, act, arch)
    out, grad, info = _cabi(sm, lgb, hps, len(pts), kind)
    assert np.all(info == 0)
    spec = sm.StackSpec(L, act, arch)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    worst = np.zeros(6)
    worst_loss = 0.0
    for i, h in enumerate(pts):
        ref_loss, ref = orc.spr_loss_grad(x, y, num_hiddens=L, act=act, arch=arch, w_std=h["w_std"], b_std=h["b_std"],
                                          last_w_std=h["last_w_std"], eps=h["eps"], kind=kind, a=h["alpha"],
                                          b=h["beta"])
        assert abs(out[i, 1] - ref_loss) <= LOSS_TOL * abs(ref_loss), (i, out[i, 1], ref_loss)
        assert np.all(_close(grad[i], ref, GRAD_TOL)), (i, grad[i], ref)
        o1, g1, i1 = _host(sm.device.lml_grad(xd, yd, spec=spec, hp=hps[i], kind=kind))
        o0, i0 = _host(sm.device.lml(xd, yd, spec=spec, hp=hps[i], kind=kind))
        assert int(i1[0]) == 0 and int(i0[0]) == 0
        assert np.all(_close(out[i], o0, AGREE_TOL)), (i, out[i], o0)
        assert np.all(_close(grad[i], g1, AGREE_TOL)), (i, grad[i], g1)
        scale = 1e-12 * np.abs(g1).max()
        worst = np.maximum(worst, np.abs(grad[i] - g1) / np.maximum(np.abs(g1), scale))
        worst_loss = max(worst_loss, abs(out[i, 1] - o0[1]) / abs(o0[1]))
    print(f"\n[grad_batch] N={n} {act}/{arch}/L={L} {kind}: worst relative difference vs lml: loss {worst_loss:.2e}, "
          f"vs lml_grad: " + " ".join(f"{k} {v:.2e}" for k, v in zip(NAMES, worst)))


def test_batch_matches_mpmath_golden(sm):
    import torch
    gold = np.load(os.path.join(ROOT, "tests", "golden", "nngp_golden.npz"))
    x, y = gold["x"], gold["y"]
    for vi, s in enumerate(gold["variants"]):
        act, arch, L, w, b, v = str(s).split(",")
        hp = dict(w_std=float(w), b_std=float(b), last_w_std=float(v), eps=float(gold["eps"]), alpha=float(gold["a"]),
                  beta=float(gold["b"]))
        lgb = _batch(sm, x, y, int(L), act, arch)
        for kind, key in (("student_t", "t"), ("gauss", "g")):
            out, grad, info = _cabi(sm, lgb, torch.from_numpy(_hp_vec(hp)[None]).cuda(), 1, kind)
            assert info[0] == 0
            assert abs(out[0, 1] - float(gold[f"loss_{key}{vi}"])) <= 1e-9 * abs(out[0, 1])
            ref = gold[f"grad_{key}{vi}"]
            assert np.all(np.abs(grad[0] - ref) <= 1e-9 * np.abs(ref) + 1e-13 * np.abs(ref).max()), (s, kind, grad, ref)


def test_finite_differences_in_one_batch_at_4096(sm):
    """The centre point and its twelve central-difference neighbours (+-1e-4 relative in each scalar) in ONE batch: the
    analytic gradient must agree with the differences of the batch's own values."""
    import torch
    n, d = 4096, 16
    x, y, *_ = regression_data(n, d)
    hp = dict(w_std=1.3, b_std=0.4, last_w_std=0.8, eps=1e-2, alpha=2.5, beta=1.5)
    rows = [_hp_vec(hp)]
    for name in NAMES:
        for sgn in (1.0, -1.0):
            h = dict(hp)
            h[name] += sgn * 1e-4 * hp[name]
            rows.append(_hp_vec(h))
    lgb = _batch(sm, x, y, 3, "relu", "mlp")
    out, grad, info = _cabi(sm, lgb, torch.from_numpy(np.stack(rows)).cuda(), len(rows), "student_t")
    assert np.all(info == 0)
    for i, name in enumerate(NAMES):
        fd = (out[1 + 2 * i, 1] - out[2 + 2 * i, 1]) / (2e-4 * hp[name])
        assert abs(grad[0, i] - fd) <= 2e-5 * abs(fd) + 1e-9, f"{name}: analytic {grad[0, i]} vs central difference {fd}"


# ---- independence and reproducibility ------------------------------------------------------------------------------
def test_point_outputs_do_not_depend_on_the_batch(sm):
    import torch
    x, y, *_ = regression_data(404, 13)
    lgb = _batch(sm, x, y, 3, "relu", "mlp")
    hps = _random_hps(500)
    ref = _host(lgb.points(hps))
    assert np.all(ref[2] == 0)
    assert _same_bits(ref, _host(lgb.points(hps))), "two calls"
    for i in (0, 1, 36, 250, 499):
        assert _same_bits(_rows(ref, slice(i, i + 1)), _cabi(sm, lgb, hps[i:i + 1], 1, "student_t")), f"point {i} alone"
    assert _same_bits(_rows(ref, slice(0, 37)), _cabi(sm, lgb, hps[:37].contiguous(), 37, "student_t")), "batch of 37"
    perm = torch.from_numpy(np.random.default_rng(1).permutation(500)).cuda()
    got = _host(lgb.points(hps[perm]))
    inv = torch.argsort(perm).cpu().numpy()
    assert _same_bits(ref, _rows(got, inv)), "permuted batch"
    for slots in (1, 7):
        assert _same_bits(_rows(ref, slice(0, 37)), _cabi(sm, lgb, hps[:37].contiguous(), slots, "student_t")), slots
    assert _same_bits(ref, _cabi(sm, lgb, hps, 500, "student_t")), "one slot per point"


def test_failed_points_are_nan_and_isolated(sm):
    """eps = -2 makes K + eps I indefinite: info as lml_grad reports it, all-NaN out and grad, and the good neighbours
    are the same bits as in a batch without the failed points."""
    import torch
    x, y, *_ = regression_data(404, 13)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    lgb = _batch(sm, x, y, 3, "relu", "mlp")
    good = _random_hps(40, seed=9)
    bad_at = [0, 3, 4, 17, 41, 43]
    rows, k = [], 0
    for i in range(good.shape[0] + len(bad_at)):
        if i in bad_at:
            h = good[k % 40].clone()
            h[3] = -2.0
            rows.append(h)
        else:
            rows.append(good[k])
            k += 1
    mixed = torch.stack(rows)
    got = _cabi(sm, lgb, mixed, 296, "student_t")
    ref = _cabi(sm, lgb, good, 296, "student_t")
    ok = [i for i in range(mixed.shape[0]) if i not in bad_at]
    assert _same_bits(_rows(got, ok), ref)
    for i in bad_at:
        _, _, info1 = sm.device.lml_grad(xd, yd, spec=lgb.spec, hp=mixed[i], kind="student_t")
        assert int(got[2][i]) == int(info1.item()) != 0
        assert np.all(np.isnan(got[0][i])) and np.all(np.isnan(got[1][i]))


# ---- C-ABI ----------------------------------------------------------------------------------------------------------
def test_arguments_are_rejected_before_anything_is_enqueued(sm):
    import torch
    lib = sm._lib.load()
    x, y, *_ = regression_data(64, 5)
    lgb = _batch(sm, x, y, 2, "relu", "mlp")
    hps = _random_hps(4)
    out = torch.empty(4 * 10, dtype=torch.float64, device="cuda")
    info = torch.empty(4, dtype=torch.int32, device="cuda")
    nbytes = lib.smnngp_lml_grad_batch_workspace_bytes(64, 2, 0, 2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: t.data_ptr()
    good = dict(K0dd=p(lgb.k0dd), ld0=lgb.ld0, q_d=p(lgb.q_d), y=p(lgb.y), N=64, G=4, nh=2, act=0, arch=0, hp=p(hps),
                kind=1, ws=p(ws), nbytes=nbytes, out=p(out), grad=p(out) + 8 * 16, info=p(info))

    def call(**over):
        a = dict(good, **over)
        return lib.smnngp_lml_grad_batch_f64(s, a["K0dd"], a["ld0"], a["q_d"], a["y"], a["N"], a["G"], a["nh"], a["act"],
                                             a["arch"], a["hp"], a["kind"], a["ws"], a["nbytes"], a["out"], a["grad"],
                                             a["info"])

    cases = [(EWORKSPACE, dict(nbytes=nbytes // 2 - 1)), (EWORKSPACE, dict(nbytes=0)), (EWORKSPACE, dict(ws=None)),
             (EINVAL, dict(N=4097, ld0=4100)), (EINVAL, dict(N=0)), (EINVAL, dict(N=-3)), (EINVAL, dict(G=0)),
             (EINVAL, dict(ld0=63)), (EINVAL, dict(nh=65)), (EINVAL, dict(nh=-1)), (EINVAL, dict(act=2)),
             (EINVAL, dict(arch=2)), (EINVAL, dict(kind=2)), (EINVAL, dict(kind=-1))]
    cases += [(EINVAL, {k: None}) for k in ("K0dd", "q_d", "y", "hp", "out", "grad", "info")]
    for code, over in cases:
        lib.smnngp_instr_reset(0)
        assert call(**over) == code, over
        assert lib.smnngp_instr_launches() == 0, over
    lib.smnngp_instr_reset(0)
    assert call() == 0 and lib.smnngp_instr_launches() == 1


def test_one_launch_at_every_size(sm):
    import torch
    lib = sm._lib.load()
    for n, g in ((17, 1), (404, 37), (2000, 300)):
        x, y, *_ = regression_data(n, 6)
        lgb = _batch(sm, x, y, 3, "relu", "mlp")
        hps = _random_hps(g)
        torch.cuda.synchronize()
        lib.smnngp_instr_reset(0)
        _, _, info = _cabi(sm, lgb, hps, min(g, 296), "student_t")
        assert lib.smnngp_instr_launches() == 1, n
        assert np.all(info == 0)


def test_graph_capture_replays_with_new_scalars(sm):
    import torch
    lib = sm._lib.load()
    x, y, *_ = regression_data(404, 13)
    lgb = _batch(sm, x, y, 3, "relu", "mlp")
    g = 37
    hps = _random_hps(g, seed=2).clone()
    nh, act, arch = lgb.spec.ids()
    out = torch.empty((g, 4), dtype=torch.float64, device="cuda")
    grad = torch.empty((g, 6), dtype=torch.float64, device="cuda")
    info = torch.empty(g, dtype=torch.int32, device="cuda")
    nbytes = lib.smnngp_lml_grad_batch_workspace_bytes(lgb.n, nh, arch, g)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")

    def enqueue():
        rc = lib.smnngp_lml_grad_batch_f64(C.c_void_p(torch.cuda.current_stream().cuda_stream), lgb.k0dd.data_ptr(),
                                           lgb.ld0, lgb.q_d.data_ptr(), lgb.y.data_ptr(), lgb.n, g, nh, act, arch,
                                           hps.data_ptr(), 1, ws.data_ptr(), nbytes, out.data_ptr(), grad.data_ptr(),
                                           info.data_ptr())
        assert rc == 0

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        enqueue()                                      # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        enqueue()
    for seed in (3, 4):
        new = _random_hps(g, seed=seed)
        hps.copy_(new)
        graph.replay()
        torch.cuda.synchronize()
        assert _same_bits(_host((out, grad, info)), _cabi(sm, lgb, new, g, "student_t"))


@pytest.mark.parametrize("n,g", [(4100, 3), (404, 1)])
def test_points_fall_back_to_lml_grad(sm, n, g):
    """Above N = 4096, and where the measured crossover says the loop is faster, points() is the loop over lml_grad."""
    import torch
    assert not sm.device._grad_batch_wins(n, g)
    x, y, *_ = regression_data(n, 6)
    lgb = _batch(sm, x, y, 2, "relu", "mlp")
    hps = _random_hps(g)
    got = _host(lgb.points(hps, "student_t"))
    for i in range(g):
        one = _host(sm.device.lml_grad(lgb.x, lgb.y, spec=lgb.spec, hp=hps[i], kind="student_t"))
        assert _same_bits(_rows(got, slice(i, i + 1)), (one[0][None], one[1][None], one[2]))


# ---- multi-start training ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["tp", "gp"])
def test_multistart_restart_zero_is_spr(sm, method):
    """Restart 0 of a MultiStartSPR is SPR at the same values: loss and gradient within AGREE_TOL, and after 20 batched
    Adam steps its variables match a 20-step SPR + Adam run to 1e-7 relative.  Duplicate starts stay the same bits."""
    import torch
    sp = sm.spax
    x, y, *_ = regression_data(404, 13)
    ws, bs, ls, eps, a, b = 1.2, 0.3, 0.9, 1e-3, 2.5, 1.5

    def kern():
        return sp.NNGPKernel(lambda w_, b_, v_: sm.get_mlp_kernel(3, 1, "relu", w_, b_, v_), ws, bs, ls)

    lik = (lambda: sp.StudentTLikelihood(a, b)) if method == "tp" else sp.GaussianLikelihood
    rng = np.random.default_rng(0)
    starts = np.tile([ws, bs, ls, eps, a, b], (16, 1)) * np.exp(0.3 * rng.standard_normal((16, 6)))
    starts[0] = [ws, bs, ls, eps, a, b]
    starts[5] = starts[9] = starts[3]
    ms = sp.MultiStartSPR(kern(), lik(), torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), 0.0, 1.0,
                          starts=starts)
    assert sm.device._grad_batch_wins(404, 16)
    model = sp.SPR(kern(), lik(), x, y, 0.0, 1.0, eps=eps)
    loss, grads = model.loss_and_grad()
    mloss, mgrad, info = ms.loss_and_grad()
    assert np.all(info.cpu().numpy() == 0)
    names = ["kernel.w_std", "kernel.b_std", "kernel.last_w_std", "eps"] + (["likelihood.a", "likelihood.b"]
                                                                           if method == "tp" else [])
    want = np.array([grads[k] for k in names] + [0.0] * (6 - len(names)))
    got = mgrad[0].cpu().numpy()
    assert abs(float(mloss[0]) - loss) <= AGREE_TOL * abs(loss)
    assert np.all(_close(got, want, AGREE_TOL)), (got, want)
    if method == "gp":
        assert np.all(mgrad[:, 4:].cpu().numpy() == 0)
    opt = sp.Adam(model.vars())
    bopt = sp.BatchAdam(ms.raw, mask=ms.mask)
    for _ in range(20):
        _, grads = model.loss_and_grad()
        opt(0.01, grads)
        _, g, _ = ms.loss_and_grad()
        bopt(0.01, g)
    ref = np.array([float(model.vars()[k].value) for k in names])
    raw = ms.raw.cpu().numpy()
    assert np.all(np.abs(raw[0, :len(names)] - ref) <= 1e-7 * np.abs(ref)), (raw[0], ref)
    assert np.array_equal(raw[3].view(np.uint8), raw[5].view(np.uint8))
    assert np.array_equal(raw[3].view(np.uint8), raw[9].view(np.uint8))
    if method == "gp":
        assert np.allclose(ms.safe_values().cpu().numpy()[:, 4:], starts[:, 4:], rtol=1e-12)
