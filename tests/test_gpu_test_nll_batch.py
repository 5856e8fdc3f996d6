"""Batched test NLL (smnngp_test_nll_batch_f64 / GridSearch.test_nll / MultiStartSPR.test_nll): SPR.test_nll at many
hyper-parameter points in one launch.  Parity with the oracle and with the per-point test_nll, bit-exact independence of
a point from the rest of its batch and from the optional outputs, failure isolation of either factorisation, argument
checks, one launch, graph capture, the per-point fallback, and the multi-start model.

The targets are de-standardised with y_mean != 0 and y_std != 1 throughout, so that a wrong scale shows."""
import ctypes as C

import numpy as np
import pytest

from oracle import nngp_oracle as orc
from tests.synth import regression_data

LML_TOL = 1e-8
POINT_TOL = 1e-9        # batched vs per-point factorisations: same matrices, different blocking and summation order
YM, YS = 0.37, 1.9
KIND = {"gauss": 0, "student_t": 1}
EINVAL, EWORKSPACE = 1, 3


@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


def _data(n, t, d):
    import torch
    x, y, xt, yt, *_ = regression_data(n, d, t=t)
    return (x, y, xt, yt), tuple(torch.from_numpy(v).cuda() for v in (x, y, xt, yt))


def _random_hps(g, seed=5):
    """[G, 6] device rows {w_std, b_std, last_w_std, eps, alpha, beta}"""
    import torch
    rng = np.random.default_rng(seed)
    h = np.stack([rng.uniform(0.6, 1.7, g), rng.uniform(0.05, 0.9, g), rng.uniform(0.5, 1.5, g),
                  10.0 ** rng.uniform(-4, -2, g), rng.uniform(1.5, 4.0, g), rng.uniform(0.5, 3.0, g)], axis=1)
    return torch.from_numpy(np.ascontiguousarray(h)).cuda()


def _host(res):
    return tuple(r.cpu().numpy() for r in res)


def _same_bits(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def _rows(res, idx):
    return tuple(r[idx] for r in res)


def _cabi(sm, gs, hps, yt, slots, kind="student_t", outputs=True):
    """smnngp_test_nll_batch_f64 with a workspace of exactly `slots` slots -> host (nll, mean, var, logp, info); with
    outputs=False mean, var and logp are not asked for (returned as None)."""
    import torch
    lib = sm._lib.load()
    nh, act, arch = gs.spec.ids()
    g, t, dev = hps.shape[0], gs.t, gs.y.device
    nll = torch.empty(g, dtype=torch.float64, device=dev)
    info = torch.empty(g, dtype=torch.int32, device=dev)
    opt = [torch.empty((g, t), dtype=torch.float64, device=dev) for _ in range(3)] if outputs else [None] * 3
    nbytes = lib.smnngp_test_nll_batch_workspace_bytes(gs.n, t, nh, arch, slots)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    ptr = lambda v: v.data_ptr() if v is not None else None
    rc = lib.smnngp_test_nll_batch_f64(C.c_void_p(torch.cuda.current_stream().cuda_stream), gs.k0dd.data_ptr(), gs.ld0,
                                       gs.k0td.data_ptr(), gs.ld0, gs.q_d.data_ptr(), gs.q_t.data_ptr(), gs.y.data_ptr(),
                                       yt.data_ptr(), gs.n, t, g, nh, act, arch, hps.data_ptr(), KIND[kind], YM, YS,
                                       ws.data_ptr(), nbytes, nll.data_ptr(), *(ptr(v) for v in opt), info.data_ptr())
    assert rc == 0, lib.smnngp_last_error()
    torch.cuda.synchronize()
    return (nll.cpu().numpy(), *(v.cpu().numpy() if v is not None else None for v in opt), info.cpu().numpy())


# ---- parity -------------------------------------------------------------------------------------------------------
SHAPES = [(404, 52, 13, "relu", "mlp", 3), (900, 130, 8, "erf", "mlp", 2), (1500, 257, 16, "relu", "resnet", 2),
          (1, 4, 5, "relu", "mlp", 3), (17, 9, 4, "erf", "resnet", 1), (300, 1, 7, "relu", "mlp", 2),
          (250, 40, 6, "relu", "mlp", 0), (4096, 512, 8, "relu", "mlp", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["student_t", "gauss"])
@pytest.mark.parametrize("n,t,d,act,arch,L", SHAPES)
def test_batch_matches_oracle_and_test_nll(sm, n, t, d, act, arch, L, kind):
    """Six random points (three at N = 4096, where the oracle needs seconds per point) against the oracle at the
    project's tolerances, and every point against the per-point test_nll."""
    (x, y, xt, yt), (xd, yd, xtd, ytd) = _data(n, t, d)
    spec = sm.StackSpec(L, act, arch)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=spec)
    g = 3 if n >= 4096 else 6
    hps = _random_hps(g, seed=n + t)
    nll, mean, var, logp, info = _cabi(sm, gs, hps, ytd, g, kind)
    assert nll.shape == (g,) and mean.shape == (g, t) and var.shape == (g, t) and logp.shape == (g, t)
    assert np.all(info == 0)
    h = hps.cpu().numpy()
    worst = 0.0
    for i in range(g):
        kw = dict(num_hiddens=L, act=act, w_std=h[i, 0], b_std=h[i, 1], last_w_std=h[i, 2], arch=arch)
        ref, m_ref, v_ref = orc.spr_test_nll(x, y, xt, yt, YM, YS, eps=h[i, 3], kind=kind, a=h[i, 4], b=h[i, 5],
                                             return_parts=True, **kw)
        ktt = orc.nngp_diag(xt, **kw)
        assert abs(nll[i] - ref) <= LML_TOL * abs(ref), f"point {i}: nll {nll[i]} vs {ref}"
        assert np.abs(mean[i] - m_ref).max() <= LML_TOL * np.abs(m_ref).max(), f"point {i}: mean"
        assert np.all(np.abs(var[i] - v_ref) <= LML_TOL * np.abs(v_ref) + 1e-13 * ktt), f"point {i}: var"
        assert abs(-logp[i].mean() - nll[i]) <= 1e-12 * np.abs(logp[i]).mean(), f"point {i}: logp"
        n1, m1, v1, i1 = sm.device.test_nll(xd, yd, xtd, ytd, YM, YS, spec=spec, hp=hps[i], kind=kind)
        assert int(i1.item()) == 0
        m1, v1 = m1.cpu().numpy(), v1.cpu().numpy()
        errs = (abs(nll[i] - n1.item()) / abs(n1.item()), np.abs(mean[i] - m1).max() / max(np.abs(m1).max(), 1e-300),
                np.abs(var[i] - v1).max() / np.abs(v1).max())
        worst = max(worst, *errs)
    assert worst <= POINT_TOL, f"batched vs per-point: worst relative difference {worst:.3e}"
    print(f"\n[test_nll_batch] N={n} T={t} {act}/{arch}/L={L} {kind}: worst relative difference vs test_nll {worst:.3e}")


# ---- independence and reproducibility ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_point_outputs_do_not_depend_on_the_batch(sm):
    import torch
    _, (xd, yd, xtd, ytd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    hps = _random_hps(500)
    assert sm.device._batch_wins(404, 37)
    ref = _host(gs.test_nll(hps, ytd, YM, YS))
    assert np.all(ref[3] == 0)
    assert _same_bits(ref, _host(gs.test_nll(hps, ytd, YM, YS))), "two calls"
    full = _cabi(sm, gs, hps, ytd, 296)
    assert _same_bits(ref, (full[0], full[1], full[2], full[4])), "GridSearch.test_nll is the C-ABI call"
    for i in (0, 1, 36, 250, 499):
        assert _same_bits(_rows(full, slice(i, i + 1)), _cabi(sm, gs, hps[i:i + 1], ytd, 1)), f"point {i} alone"
    assert _same_bits(_rows(ref, slice(0, 37)), _host(gs.test_nll(hps[:37], ytd, YM, YS))), "batch of 37"
    perm = torch.from_numpy(np.random.default_rng(1).permutation(500)).cuda()
    got = _host(gs.test_nll(hps[perm], ytd, YM, YS))
    inv = torch.argsort(perm).cpu().numpy()
    assert _same_bits(ref, _rows(got, inv)), "permuted batch"
    for slots in (1, 7):
        assert _same_bits(_rows(full, slice(0, 37)), _cabi(sm, gs, hps[:37].contiguous(), ytd, slots)), f"{slots} slots"
    assert _same_bits(full, _cabi(sm, gs, hps, ytd, 500)), "one slot per point"
    bare = _cabi(sm, gs, hps, ytd, 296, outputs=False)
    assert _same_bits((full[0], full[4]), (bare[0], bare[4])), "nll without the optional outputs"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["student_t", "gauss"])
def test_failed_points_are_nan_and_isolated(sm, kind):
    """eps = -2 fails the predictive factorisation: every output NaN and info as test_nll reports it.  alpha / beta =
    -1e9 (shift 1e-6 alpha / beta = -1e3) fails only the Student-t factorisation, at pivot 1: mean and var finite, nll
    and logp NaN, info = 1 (under Gaussian that factorisation does not exist and the point is good).  The good
    neighbours are the same bits as in a batch without the failing points."""
    import torch
    _, (xd, yd, xtd, ytd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    good = _random_hps(40, seed=9)
    bad_eps, bad_lik = [0, 4, 41], [3, 17, 43]
    rows, k = [], 0
    for i in range(good.shape[0] + len(bad_eps) + len(bad_lik)):
        if i in bad_eps or i in bad_lik:
            h = good[k % 40].clone()
            if i in bad_eps:
                h[3] = -2.0
            else:
                h[4] = -1e9 * h[5]
            rows.append(h)
        else:
            rows.append(good[k])
            k += 1
    mixed = torch.stack(rows)
    got = _cabi(sm, gs, mixed, ytd, 296, kind)
    ref = _cabi(sm, gs, good, ytd, 296, kind)
    ok = [i for i in range(mixed.shape[0]) if i not in bad_eps + bad_lik]
    assert _same_bits(_rows(got, ok), ref)
    nll, mean, var, logp, info = got
    for i in bad_eps:
        _, _, _, info1 = sm.device.test_nll(xd, yd, xtd, ytd, YM, YS, spec=gs.spec, hp=mixed[i], kind=kind)
        assert int(info[i]) == int(info1.item()) != 0
        assert np.isnan(nll[i]) and np.all(np.isnan(mean[i])) and np.all(np.isnan(var[i])) and np.all(np.isnan(logp[i]))
    for i in bad_lik:
        assert np.all(np.isfinite(mean[i])) and np.all(np.isfinite(var[i]))
        if kind == "student_t":
            assert int(info[i]) == 1 and np.isnan(nll[i]) and np.all(np.isnan(logp[i]))
        else:
            assert int(info[i]) == 0 and np.isfinite(nll[i])


# ---- C-ABI ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_arguments_are_rejected_before_anything_is_enqueued(sm):
    import torch
    lib = sm._lib.load()
    _, (xd, yd, xtd, ytd) = _data(64, 8, 5)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(2, "relu", "mlp"))
    hps = _random_hps(4)
    out = torch.empty(4 + 3 * 4 * 8, dtype=torch.float64, device="cuda")
    info = torch.empty(4, dtype=torch.int32, device="cuda")
    nbytes = lib.smnngp_test_nll_batch_workspace_bytes(64, 8, 2, 0, 2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: t.data_ptr()
    good = dict(K0dd=p(gs.k0dd), ld0=gs.ld0, K0td=p(gs.k0td), ld0t=gs.ld0, q_d=p(gs.q_d), q_t=p(gs.q_t), y=p(gs.y),
                yt=p(ytd), N=64, T=8, G=4, nh=2, act=0, arch=0, hp=p(hps), kind=1, ws=p(ws), nbytes=nbytes, nll=p(out),
                mean=p(out) + 8 * 4, var=p(out) + 8 * 36, logp=p(out) + 8 * 68, info=p(info))

    def call(**over):
        a = dict(good, **over)
        return lib.smnngp_test_nll_batch_f64(s, a["K0dd"], a["ld0"], a["K0td"], a["ld0t"], a["q_d"], a["q_t"], a["y"],
                                             a["yt"], a["N"], a["T"], a["G"], a["nh"], a["act"], a["arch"], a["hp"],
                                             a["kind"], YM, YS, a["ws"], a["nbytes"], a["nll"], a["mean"], a["var"],
                                             a["logp"], a["info"])

    cases = [(EWORKSPACE, dict(nbytes=nbytes // 2 - 1)), (EWORKSPACE, dict(nbytes=0)), (EWORKSPACE, dict(ws=None)),
             (EINVAL, dict(N=4097, ld0=4100, ld0t=4100)), (EINVAL, dict(N=0)), (EINVAL, dict(N=-3)),
             (EINVAL, dict(T=0)), (EINVAL, dict(G=0)), (EINVAL, dict(ld0=63)), (EINVAL, dict(ld0t=63)),
             (EINVAL, dict(nh=65)), (EINVAL, dict(nh=-1)), (EINVAL, dict(act=2)), (EINVAL, dict(arch=2)),
             (EINVAL, dict(kind=2)), (EINVAL, dict(kind=-1))]
    cases += [(EINVAL, {k: None}) for k in ("K0dd", "K0td", "q_d", "q_t", "y", "yt", "hp", "nll", "info")]
    for code, over in cases:
        lib.smnngp_instr_reset(0)
        assert call(**over) == code, over
        assert lib.smnngp_instr_launches() == 0, over
    for over in ({}, dict(mean=None, var=None, logp=None)):
        lib.smnngp_instr_reset(0)
        assert call(**over) == 0 and lib.smnngp_instr_launches() == 1, over


@pytest.mark.gpu
def test_one_launch_at_every_size(sm):
    import torch
    lib = sm._lib.load()
    for n, g in ((17, 1), (404, 37), (2000, 300)):
        _, (xd, yd, xtd, ytd) = _data(n, 12, 6)
        gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
        hps = _random_hps(g)
        torch.cuda.synchronize()
        lib.smnngp_instr_reset(0)
        info = _cabi(sm, gs, hps, ytd, min(g, 296))[4]
        assert lib.smnngp_instr_launches() == 1, n
        assert np.all(info == 0)


@pytest.mark.gpu
def test_graph_capture_replays_with_new_scalars(sm):
    import torch
    lib = sm._lib.load()
    _, (xd, yd, xtd, ytd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    g, t = 37, gs.t
    hps = _random_hps(g, seed=2).clone()
    nh, act, arch = gs.spec.ids()
    nll = torch.empty(g, dtype=torch.float64, device="cuda")
    mean, var, logp = (torch.empty((g, t), dtype=torch.float64, device="cuda") for _ in range(3))
    info = torch.empty(g, dtype=torch.int32, device="cuda")
    nbytes = lib.smnngp_test_nll_batch_workspace_bytes(gs.n, t, nh, arch, g)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")

    def enqueue():
        rc = lib.smnngp_test_nll_batch_f64(C.c_void_p(torch.cuda.current_stream().cuda_stream), gs.k0dd.data_ptr(),
                                           gs.ld0, gs.k0td.data_ptr(), gs.ld0, gs.q_d.data_ptr(), gs.q_t.data_ptr(),
                                           gs.y.data_ptr(), ytd.data_ptr(), gs.n, t, g, nh, act, arch, hps.data_ptr(),
                                           1, YM, YS, ws.data_ptr(), nbytes, nll.data_ptr(), mean.data_ptr(),
                                           var.data_ptr(), logp.data_ptr(), info.data_ptr())
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
        assert _same_bits(_host((nll, mean, var, logp, info)), _cabi(sm, gs, new, ytd, g))


@pytest.mark.gpu
@pytest.mark.parametrize("n,g", [(4100, 3), (2048, 11)])
def test_falls_back_to_test_nll(sm, n, g):
    """Above N = 4096, and where the crossover says the loop is faster, GridSearch.test_nll is the test_nll loop."""
    assert not sm.device._batch_wins(n, g)
    _, (xd, yd, xtd, ytd) = _data(n, 8, 6)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(2, "relu", "mlp"))
    hps = _random_hps(g)
    got = _host(gs.test_nll(hps, ytd, YM, YS))
    for i in range(g):
        one = _host(sm.device.test_nll(xd, yd, xtd, ytd, YM, YS, spec=gs.spec, hp=hps[i]))
        assert _same_bits(_rows(got, slice(i, i + 1)), (one[0][None], one[1][None], one[2][None], one[3]))


# ---- multi-start model ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("method", ["tp", "gp"])
def test_multistart_test_nll_matches_test_nll(sm, method):
    import torch
    sp = sm.spax
    (x, y, xt, yt), (xd, yd, xtd, ytd) = _data(404, 50, 13)
    kind = "student_t" if method == "tp" else "gauss"
    kern = sp.NNGPKernel(lambda w_, b_, v_: sm.get_mlp_kernel(3, 1, "relu", w_, b_, v_), 1.0, 0.1, 1.0)
    lik = sp.StudentTLikelihood(2.0, 2.0) if method == "tp" else sp.GaussianLikelihood()
    rng = np.random.default_rng(0)
    starts = np.tile([1.0, 0.1, 1.0, 1e-3, 2.0, 2.0], (16, 1)) * np.exp(0.3 * rng.standard_normal((16, 6)))
    ms = sp.MultiStartSPR(kern, lik, xd, yd, YM, YS, starts=starts)
    assert sm.device._batch_wins(404, 16)
    got = ms.test_nll(xt, yt).cpu().numpy()
    assert got.shape == (16,)
    hps = ms.safe_values()
    for r in range(16):
        ref = sm.device.test_nll(xd, yd, xtd, ytd, YM, YS, spec=ms.spec, hp=hps[r], kind=kind)[0].item()
        assert abs(got[r] - ref) <= POINT_TOL * abs(ref), (r, got[r], ref)


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,t,nh,arch", [(404, 52, 3, 0), (1, 1, 0, 0), (4096, 512, 2, 1), (17, 300, 64, 0)])
def test_test_nll_batch_workspace_is_affine_in_slots(n, t, nh, arch):
    import smnngp_b200 as s
    lib = s._lib.load()
    one = lib.smnngp_test_nll_batch_workspace_bytes(n, t, nh, arch, 1)
    assert one >= (n + t + 1) * n * 8
    assert lib.smnngp_test_nll_batch_workspace_bytes(n, t, nh, arch, 0) == 0
    for slots in (2, 7, 296):
        assert lib.smnngp_test_nll_batch_workspace_bytes(n, t, nh, arch, slots) == slots * one
