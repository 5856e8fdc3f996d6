"""The scale mixture (csrc/mixture.cu): scale draws against the CPU replica of their Philox stream, draw for draw; the
importance-sampling table against the NumPy estimator on the same draws, against the Gaussian path for a point mass
and against the Student-t closed forms for inverse-gamma draws; edge draws, failure isolation, bit-identical pairs in
any batch, one launch per call, graph replay and the spax likelihood."""
import ctypes as C

import numpy as np
import pytest

from oracle import nngp_oracle as orc
from tests import mixture_ref as mr
from tests.synth import regression_data, DEFAULT_HP

SMNNGP_EINVAL = 1
FAMILY = {"invgamma": 0, "burr12": 1}
EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


def _params(family, P, seed):
    """[P, 2] prior rows: inverse gamma a on both sides of 1, Burr XII c and k over two decades; for P >= 3 row 1 is
    not a valid prior"""
    rng = np.random.default_rng(seed)
    if family == "invgamma":
        prm = np.stack([10.0 ** rng.uniform(np.log10(0.3), np.log10(40.0), P), rng.uniform(0.5, 3.0, P)], 1)
    else:
        prm = np.stack([10.0 ** rng.uniform(np.log10(0.5), 1.0, P), 10.0 ** rng.uniform(-1.0, np.log10(2.0), P)], 1)
    if P >= 3:
        prm[1] = (-1.0, 2.0) if family == "invgamma" else (np.inf, 0.5)
    return prm


DRAW_CASES = [("invgamma", 1, 1, 0), ("burr12", 1, 255, 2**64 - 1), ("invgamma", 3, 4097, 2**32 + 7),
              ("burr12", 3, 1000, 1234), ("invgamma", 100, 255, 2**40 + 3), ("burr12", 100, 4097, 2**32 + 7),
              ("invgamma", 100, 1000, 2**64 - 1), ("burr12", 100, 1, 5), ("invgamma", 3, 1, 2**33)]


@pytest.mark.gpu
@pytest.mark.parametrize("family,P,S,seed", DRAW_CASES, ids=["%s-P%d-S%d-seed%d" % c for c in DRAW_CASES])
def test_scale_draws_match_replica(sm, family, P, S, seed):
    import torch
    prm = _params(family, P, seed=P * 7 + S)
    got = sm.device.scale_draws(family, torch.from_numpy(prm).cuda(), S, seed=seed).cpu().numpy()
    ref, margin = mr.scale_draws(family, prm, S, seed)
    assert got.shape == (P, S)
    valid = np.array([a > 0 and b > 0 and np.isfinite(a) and np.isfinite(b) for a, b in prm])
    assert np.isnan(got[~valid]).all() and not np.isnan(got[valid]).any()
    # a few ulp of fp64 libm between CUDA and NumPy; the Burr exponent log(expm1(.)) / c carries an absolute rounding
    # of its own size into the relative error of s
    with np.errstate(divide="ignore"):
        size = np.maximum(1.0, np.abs(np.log(np.abs(ref))))
    tol = (1e-14 if family == "burr12" else 1e-13) * size
    near = margin < 1e-10                          # gamma accept decisions within rounding of the threshold
    with np.errstate(invalid="ignore"):
        rel = np.where(got[valid] == ref[valid], 0.0, np.abs(got[valid] - ref[valid]) / np.abs(ref[valid]))
    bad = (rel > tol[valid]) & ~near[valid]
    print(f"{family} P={P} S={S}: worst relative difference {rel[~near[valid]].max(initial=0):.3e}, "
          f"{int(near.sum())} draws near a decision")
    assert not bad.any(), f"{int(bad.sum())} draws differ, first at {np.argwhere(bad)[0]}"


@pytest.mark.gpu
def test_scale_draws_do_not_reuse_the_posterior_draw_stream(sm):
    """same seed: the scale stream's counters (j, p, 0xFFFFFFFF) are not sample_f_iid's (s, t, c < 2^31)"""
    import torch
    prm = torch.tensor([[1.0, 1.0]], dtype=torch.float64, device="cuda")
    s1 = sm.device.scale_draws("burr12", prm, 64, seed=3).cpu().numpy()
    s2 = sm.device.scale_draws("burr12", prm, 64, seed=2**32 + 3).cpu().numpy()
    assert not np.any(s1 == s2)
    assert s1.shape == (1, 64) and np.all(s1 > 0)


def _points(sm, n, t, d, act, arch, L, g, seed=5):
    import torch
    x, y, xt, yt, ym, ys = regression_data(n, d, t=t)
    xd, yd, xtd = (torch.from_numpy(v).cuda() for v in (x, y, xt))
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(L, act, arch))
    rng = np.random.default_rng(seed)
    hps = torch.stack([sm.make_hp(rng.uniform(0.5, 2.0), rng.uniform(0.01, 1.0), 1.0, 10.0 ** rng.uniform(-4, -2))
                       for _ in range(g)])
    return gs, hps, yt, ym, ys


def _ell_scale(scal, draws, n):
    """largest |max_j l_j| over the table: l_j is rounded at this size on either side, and logp, nll and ess are
    differences and ratios of its exponentials"""
    tops = [np.max(mr._mixture_ell(d, n, q)[0]) for q in np.asarray(scal)[:, 1] for d in np.asarray(draws)]
    return max([abs(t) for t in tops if np.isfinite(t)] + [1.0])


def _assert_close(got, ref, ell, what):
    """1e-12 relative, plus 8 ulp of l_j carried into the result"""
    both_nan = np.isnan(got) & np.isnan(ref)
    same = (got == ref) | both_nan
    err = np.where(same, 0.0, np.abs(got - ref))
    mag = np.abs(np.where(np.isfinite(ref), ref, 0.0))
    tol = 1e-12 * mag + 1e-12 + 8 * EPS * ell * np.maximum(1.0, mag)
    print(f"{what}: worst abs {err.max(initial=0):.3e}")
    assert np.all(err <= tol), f"{what} off at {np.argwhere(err > tol)[:5]}: {got[err > tol][:3]} vs {ref[err > tol][:3]}"


MIX_SHAPES = [(404, 52, 13, "relu", "mlp", 3, 11), (900, 130, 8, "erf", "mlp", 2, 5), (17, 9, 4, "erf", "resnet", 1, 4),
              (1, 4, 5, "relu", "mlp", 3, 3), (300, 1, 7, "relu", "mlp", 2, 6), (4100, 20, 6, "relu", "mlp", 2, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["invgamma", "burr12"])
@pytest.mark.parametrize("n,t,d,act,arch,L,g", MIX_SHAPES, ids=["N%d-T%d-%s" % (s[0], s[1], s[3]) for s in MIX_SHAPES])
def test_mixture_matches_oracle_on_the_same_draws(sm, family, n, t, d, act, arch, L, g):
    """GridSearch.mixture (batched points, or the point loop for N > 4096) and mixture_nll with logp against
    oracle.mixture_nll on the GPU's points and draws (the draws are checked against the replica above)"""
    import torch
    gs, hps, yt, ym, ys = _points(sm, n, t, d, act, arch, L, g)
    P, S = 4, 777
    prm = _params(family, P, seed=n)
    prm[1] = prm[0] if family == "invgamma" else (1.7, 0.6)             # every row a valid prior here
    nll, lml, ess = (r.cpu().numpy() for r in
                     gs.mixture(hps, torch.from_numpy(yt).cuda(), ym, ys, family=family, params=prm, num_samples=S,
                                seed=n))
    mean, var, logdet, quad, info = gs.points(hps)
    assert int(info.abs().sum()) == 0
    draws = sm.device.scale_draws(family, torch.from_numpy(prm).cuda(), S, seed=n)
    scal = torch.stack([0.5 * logdet, quad], 1)
    nll2, lml2, ess2, logp = sm.device.mixture_nll(scal, mean, var, torch.from_numpy(yt).cuda(), n, draws, ym, ys,
                                                   logp=True)
    for a, b in ((nll, nll2), (lml, lml2), (ess, ess2)):
        assert np.array_equal(a, b.cpu().numpy())
    rn, rl, re, rp = mr.mixture_nll(scal.cpu().numpy(), mean.cpu().numpy(), var.cpu().numpy(), yt, n,
                                     draws.cpu().numpy(), ym, ys)
    assert np.isfinite(nll).all() and np.isfinite(lml).all()
    assert np.all(ess >= 1.0 - 1e-12) and np.all(ess <= S * (1.0 + 1e-12))
    ell = _ell_scale(scal.cpu().numpy(), draws.cpu().numpy(), n)
    _assert_close(nll, rn, ell, "nll")
    _assert_close(lml, rl, ell, "lml")
    _assert_close(ess, re, ell, "ess")
    _assert_close(logp.cpu().numpy(), rp, ell, "logp")


@pytest.mark.gpu
def test_point_mass_is_the_gaussian_path(sm):
    """draws all equal to 1: lml is the Gaussian evidence of K + eps I (from the pieces of lml(kind="gauss")), nll the
    Gaussian test NLL of the same predictive, ess = S"""
    import torch
    n, t, d, G, S = 404, 52, 13, 7, 1000
    gs, hps, yt, ym, ys = _points(sm, n, t, d, "relu", "mlp", 3, G)
    mean, var, _, _, _ = gs.points(hps)
    x, y, *_ = regression_data(n, d, t=t)
    outs = torch.stack([sm.device.lml(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), spec=gs.spec, hp=hps[i],
                                      kind="gauss")[0] for i in range(G)])
    draws = torch.ones((2, S), dtype=torch.float64, device="cuda")
    nll, lml, ess, _ = sm.device.mixture_nll(outs[:, 2:4].contiguous(), mean, var, torch.from_numpy(yt).cuda(), n,
                                             draws, ym, ys)
    nll, lml, ess = (r.cpu().numpy() for r in (nll, lml, ess))
    ref_lml = outs[:, 0].cpu().numpy()[:, None]
    ref_nll = gs.test_nll(hps, torch.from_numpy(yt).cuda(), ym, ys, kind="gauss")[0].cpu().numpy()[:, None]
    assert np.all(ess == S)
    assert np.all(np.abs(lml - ref_lml) <= 1e-12 * np.abs(ref_lml)), (lml, ref_lml)
    assert np.all(np.abs(nll - ref_nll) <= 1e-12 * np.abs(ref_nll)), (nll, ref_nll)


@pytest.mark.gpu
def test_inverse_gamma_converges_to_student_t(sm):
    """IG(a, b) draws, S = 2^20, N = 17: lml within 5 standard errors of lml(kind="student_t") and nll of
    test_nll(kind="student_t") at eps = 1e-6 a / b, where both regularisers coincide"""
    import torch
    n, t, d = 17, 9, 4
    a, b = 2.0, 2.0
    x, y, xt, yt, ym, ys = regression_data(n, d, t=t)
    xd, yd, xtd, ytd = (torch.from_numpy(v).cuda() for v in (x, y, xt, yt))
    spec = sm.StackSpec(2, "relu", "mlp")
    hp = sm.make_hp(1.0, 0.1, 1.0, 1e-6 * a / b, a, b)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=spec)
    mean, var, logdet, quad, _ = gs.points(hp[None])
    S = 2**20
    draws = sm.device.scale_draws("invgamma", torch.tensor([[a, b]], dtype=torch.float64, device="cuda"), S, seed=11)
    nll, lml, ess, logp = sm.device.mixture_nll(torch.stack([0.5 * logdet, quad], 1), mean, var, ytd, n, draws, ym,
                                                ys, logp=True)
    ref_lml = float(sm.device.lml(xd, yd, spec=spec, hp=hp, kind="student_t")[0][0])
    ref_nll = float(sm.device.test_nll(xd, yd, xtd, ytd, ym, ys, spec=spec, hp=hp, kind="student_t")[0])
    se_lml, _, se_nll = mr.mixture_se(draws.cpu().numpy()[0], float(0.5 * logdet[0]), float(quad[0]), n,
                                       mean.cpu().numpy()[0], var.cpu().numpy()[0], yt, ym, ys)
    got_lml, got_nll = float(lml[0, 0]), float(nll[0, 0])
    print(f"lml {got_lml} vs {ref_lml} (se {se_lml:.2e}); nll {got_nll} vs {ref_nll} (se {se_nll:.2e}); "
          f"ess {float(ess[0, 0]):.0f}")
    assert abs(got_lml - ref_lml) <= 5 * se_lml
    assert abs(got_nll - ref_nll) <= 5 * se_nll


@pytest.mark.gpu
def test_edge_draws_and_failures_stay_confined(sm):
    import torch
    n, t, G, S = 30, 6, 4, 64
    rng = np.random.default_rng(8)
    scal = np.stack([rng.uniform(-5, 5, G), rng.uniform(10, 60, G)], 1)
    mean, var, yt = rng.standard_normal((G, t)), rng.uniform(0.1, 2.0, (G, t)), rng.standard_normal(t)
    ok = 10.0 ** rng.uniform(-1, 1, S)
    edge = ok.copy()
    edge[:8] = [0.0, 1e-300, 1e300, np.inf, 0.0, 1e-300, 1e300, np.inf]
    zero = np.resize([0.0, np.inf], S)
    nanrow = ok.copy()
    nanrow[17] = np.nan
    draws = np.stack([ok, edge, zero, nanrow])
    bad_scal = scal.copy()
    bad_scal[2] = np.nan                                             # a failed factorisation at point 2

    def run(sc, dr_):
        r = sm.device.mixture_nll(torch.from_numpy(sc).cuda(), torch.from_numpy(mean).cuda(),
                                  torch.from_numpy(var).cuda(), torch.from_numpy(yt).cuda(), n,
                                  torch.from_numpy(dr_).cuda(), 0.3, 1.7, logp=True)
        return [x.cpu().numpy() for x in r]

    nll, lml, ess, logp = run(scal, draws)
    assert np.isfinite(nll[:, :2]).all() and np.isfinite(lml[:, :2]).all() and np.isfinite(logp[:, :2]).all()
    assert np.all(ess[:, 2] == 0.0) and np.all(lml[:, 2] == -np.inf) and np.isnan(nll[:, 2]).all()
    assert np.isnan(logp[:, 2]).all()
    assert np.isnan(nll[:, 3]).all() and np.isnan(lml[:, 3]).all() and np.isnan(ess[:, 3]).all()
    assert np.isnan(logp[:, 3]).all()
    rn, rl, re, rp = mr.mixture_nll(scal, mean, var, yt, n, draws[:2], 0.3, 1.7)
    ell = _ell_scale(scal, draws[:1], n)
    _assert_close(nll[:, :2], rn, ell, "nll")
    _assert_close(lml[:, :2], rl, ell, "lml")
    _assert_close(ess[:, :2], re, ell, "ess")
    _assert_close(logp[:, :2], rp, ell, "logp")
    nll2, lml2, ess2, logp2 = run(bad_scal, draws)
    for a, b in ((nll, nll2), (lml, lml2), (ess, ess2), (logp, logp2)):
        assert np.isnan(b[2]).all()
        keep = np.array([0, 1, 3])
        assert np.array_equal(a[keep].view(np.uint64), b[keep].view(np.uint64))


@pytest.mark.gpu
def test_pair_outputs_are_the_same_bits_in_any_batch(sm):
    import torch
    n, t, G, P, S = 50, 37, 5, 4, 1000
    rng = np.random.default_rng(9)
    scal = np.stack([rng.uniform(-5, 5, G), rng.uniform(20, 80, G)], 1)
    mean, var, yt = rng.standard_normal((G, t)), rng.uniform(0.1, 2.0, (G, t)), rng.standard_normal(t)
    prm = _params("burr12", P, 1)
    prm[1] = (1.7, 0.6)
    draws = sm.device.scale_draws("burr12", torch.from_numpy(prm).cuda(), S, seed=4)
    draws = draws.cpu().numpy()

    def run(gi, pi, logp=True):
        r = sm.device.mixture_nll(torch.from_numpy(scal[gi]).cuda(), torch.from_numpy(mean[gi]).cuda(),
                                  torch.from_numpy(var[gi]).cuda(), torch.from_numpy(yt).cuda(), n,
                                  torch.from_numpy(draws[pi]).cuda(), 0.1, 2.0, logp=logp)
        return [None if x is None else x.cpu().numpy() for x in r]

    full = run(np.arange(G), np.arange(P))
    assert np.isfinite(full[0]).all()
    perm_g, perm_p = rng.permutation(G), rng.permutation(P)
    perm = run(perm_g, perm_p)
    for k in range(4):
        assert np.array_equal(perm[k], full[k][perm_g][:, perm_p])
    nolog = run(np.arange(G), np.arange(P), logp=False)
    assert nolog[3] is None
    for k in range(3):
        assert np.array_equal(nolog[k], full[k])
    split = [run(np.arange(G), np.arange(0, 1)), run(np.arange(G), np.arange(1, P))]
    for k in range(4):
        assert np.array_equal(np.concatenate([split[0][k], split[1][k]], axis=1), full[k])
    for g, p in ((0, 0), (4, 3), (2, 1)):
        one = run(np.array([g]), np.array([p]))
        for k in range(4):
            assert np.array_equal(one[k][0, 0], full[k][g, p])


def _ptr(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


@pytest.mark.gpu
def test_one_launch_per_call_and_none_when_rejected(sm):
    import torch
    lib = sm._lib.load()
    f64 = dict(dtype=torch.float64, device="cuda")
    G, P, S, T, N = 3, 2, 100, 5, 20
    prm = torch.tensor([[2.0, 2.0], [1.0, 3.0]], **f64)
    draws = torch.empty((P, S), **f64)
    scal = torch.tensor([[1.0, 20.0]] * G, **f64)
    mean, var, yt = torch.zeros((G, T), **f64), torch.ones((G, T), **f64), torch.zeros(T, **f64)
    out = [torch.empty((G, P), **f64) for _ in range(3)]
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.smnngp_instr_reset(0)
    assert lib.smnngp_scale_draws_f64(s, 0, _ptr(prm), P, S, 1, _ptr(draws)) == 0
    assert lib.smnngp_instr_launches() == 1
    lib.smnngp_instr_reset(0)
    assert lib.smnngp_mixture_nll_f64(s, _ptr(scal), _ptr(mean), _ptr(var), T, _ptr(yt), N, T, G, _ptr(draws), P, S,
                                      0.0, 1.0, *(_ptr(o) for o in out), None) == 0
    assert lib.smnngp_instr_launches() == 1
    lib.smnngp_instr_reset(0)
    assert lib.smnngp_mixture_nll_f64(s, _ptr(scal), None, None, 0, None, N, 0, G, _ptr(draws), P, S, 0.0, 1.0, None,
                                      _ptr(out[1]), _ptr(out[2]), None) == 0
    assert lib.smnngp_instr_launches() == 1
    lib.smnngp_instr_reset(0)
    assert lib.smnngp_scale_draws_f64(s, 2, _ptr(prm), P, S, 1, _ptr(draws)) == SMNNGP_EINVAL
    assert lib.smnngp_mixture_nll_f64(s, _ptr(scal), _ptr(mean), _ptr(var), T, _ptr(yt), N, T, G, _ptr(draws), P, S,
                                      0.0, 0.0, *(_ptr(o) for o in out), None) == SMNNGP_EINVAL
    assert lib.smnngp_instr_launches() == 0
    torch.cuda.synchronize()
    assert np.isfinite(out[1].cpu().numpy()).all()


@pytest.mark.gpu
def test_graph_replay_with_new_params(sm):
    import torch
    n, t, G, P, S = 40, 8, 3, 2, 500
    rng = np.random.default_rng(12)
    f64 = dict(dtype=torch.float64, device="cuda")
    scal = torch.from_numpy(np.stack([rng.uniform(-5, 5, G), rng.uniform(20, 60, G)], 1)).cuda()
    mean, var = torch.from_numpy(rng.standard_normal((G, t))).cuda(), torch.from_numpy(rng.uniform(0.1, 2, (G, t))).cuda()
    yt = torch.from_numpy(rng.standard_normal(t)).cuda()
    prm = torch.tensor([[1.5, 0.7], [3.0, 2.0]], **f64)
    lib = sm._lib.load()
    draws = torch.empty((P, S), **f64)
    outs = [torch.empty((G, P), **f64) for _ in range(3)]

    def enqueue():
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        assert lib.smnngp_scale_draws_f64(st, 1, _ptr(prm), P, S, 21, _ptr(draws)) == 0
        assert lib.smnngp_mixture_nll_f64(st, _ptr(scal), _ptr(mean), _ptr(var), t, _ptr(yt), n, t, G, _ptr(draws), P,
                                          S, 0.2, 1.3, *(_ptr(o) for o in outs), None) == 0

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        enqueue()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        enqueue()
    for new in ([[1.5, 0.7], [3.0, 2.0]], [[0.8, 1.9], [5.0, 0.3]]):
        prm.copy_(torch.tensor(new, **f64))
        graph.replay()
        torch.cuda.synchronize()
        got = [o.cpu().numpy().copy() for o in outs]
        d = sm.device.scale_draws("burr12", torch.tensor(new, **f64), S, seed=21)
        ref = sm.device.mixture_nll(scal, mean, var, yt, n, d, 0.2, 1.3)
        for a, b in zip(got, ref[:3]):
            assert np.array_equal(a, b.cpu().numpy())


@pytest.mark.gpu
def test_spr_burr12_likelihood(sm):
    import torch
    from smnngp_b200 import spax as sp
    n, t, d = 120, 20, 5
    x, y, xt, yt, ym, ys = regression_data(n, d, t=t)
    kern = sp.NNGPKernel(lambda w, b, v: sm.get_mlp_kernel(3, 1, "relu", w, b, v), w_std=1.2, b_std=0.3,
                         last_w_std=0.9)
    lik = sp.BurrXIILikelihood(1.7, 0.6, num_samples=3000, seed=77)
    eps = 1e-4
    kw = dict(num_hiddens=3, act="relu", w_std=kern.w_std.safe_value, b_std=kern.b_std.safe_value,
              last_w_std=kern.last_w_std.safe_value, arch="mlp")
    mean, var, logdet, quad = orc.find_grid_point(x, y, xt, eps, kernel_kwargs=kw)
    draws, _ = mr.scale_draws("burr12", [[lik.c.safe_value, lik.k.safe_value]], 3000, 77)
    rn, rl, _, _ = mr.mixture_nll([[0.5 * logdet, quad]], mean[None], var[None], yt, n, draws, ym, ys)
    for host in (False, True):
        xs, yy = (x, y) if host else (torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
        model = sp.SPR(kern, lik, xs, yy, ym, ys, eps=eps)
        loss = float(model.loss())
        nll = float(model.test_nll(xt if host else torch.from_numpy(xt).cuda(),
                                   yt if host else torch.from_numpy(yt).cuda()))
        assert abs(loss + rl[0, 0] / n) <= 1e-9 * abs(rl[0, 0] / n), (loss, -rl[0, 0] / n)
        assert abs(nll - rn[0, 0]) <= 1e-8 * abs(rn[0, 0]), (nll, rn[0, 0])
        with pytest.raises(TypeError):
            model.loss_and_grad()
    with pytest.raises(TypeError):
        sp.MultiStartSPR(kern, lik, torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), ym, ys,
                         starts=np.ones((2, 6)))
    other = sp.SPR(sp.NNGPKernel(lambda w, b, v: (lambda x1, x2=None, get="nngp": None)), lik, x, y, ym, ys)
    with pytest.raises(TypeError):
        other.loss()
