"""The NNGP layer recursion outside the O(1) range of standardised inputs: layer variances u far from 1 (tiny or huge
inputs, deep ReLU stacks that halve u at every layer, small weights), every angle between two rows, and the gradient
in the same regimes - plus exact identities of the gradient that need no oracle, up to the full BASELINE config 3
size.

The ReLU step phi(k; u1, u2) is positively homogeneous (phi(c k; c u1, c u2) = c phi), so its error is measured
relative to sqrt(u1 u2) and a ReLU stack with b_std = 0 is exactly scale-equivariant: K(c X) = c^2 K(X)."""
import json
import math
import os

import mpmath as mp
import numpy as np
import pytest

from oracle import nngp_oracle as orc
from tests.golden.make_golden import act_off
from tests.synth import regression_data, pixel_data, DEFAULT_HP

pytestmark = pytest.mark.gpu

GRAM_TOL = 1e-10
LML_TOL = 1e-8
GRAD_TOL = 1e-7
IDENTITY_TOL = 1e-8
SMNNGP_EINVAL = 1                           # include/smnngp.h
NAMES = ("w_std", "b_std", "last_w_std", "eps", "alpha", "beta")
# input scales 2^e: exact in binary, and u1 u2 (down to 2^-800, up to 2^800) stays a normal double
SCALE_EXPS = (-200, -100, -40, -24, -12, 0, 12, 40, 100, 200)


@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


def _hpd(sm, hp):
    return sm.make_hp(*(hp[k] for k in NAMES))


def _kw(hp, L, act, arch):
    return dict(num_hiddens=L, act=act, w_std=hp["w_std"], b_std=hp["b_std"], last_w_std=hp["last_w_std"], arch=arch)


def _cuda(*arrays):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays)


# ---- a. one ReLU step at every angle and at radii 2^-200 .. 2^200, against 50-digit mpmath -------------------------
def _row_angles():
    """angles of the rows: exact axis directions, both sides of the swap at pi/4 and 3 pi/4 (s = |k|) and of the
    tan(pi/8) switch of the atan polynomial (pi/8, 3 pi/8, 5 pi/8, 7 pi/8), and near-(anti)parallel pairs"""
    pi = math.pi
    ang = [0.0, pi / 2, pi, 1e-8, 1e-4, pi - 1e-8, pi / 2 + 1e-9, 1.0, 2.0]
    for c in (pi / 8, pi / 4, 3 * pi / 8, 5 * pi / 8, 3 * pi / 4, 7 * pi / 8):
        for d in (1e-12, 1e-6):
            ang += [c - d, c + d]
    return ang


def _unit(phi):
    """sqrt(2) (cos phi, sin phi) with the axis directions exact, so that q0 = ||x||^2 / 2 ~ 1"""
    exact = {0.0: (1.0, 0.0), math.pi / 2: (0.0, 1.0), math.pi: (-1.0, 0.0)}
    c, s = exact.get(phi, (math.cos(phi), math.sin(phi)))
    return math.sqrt(2.0) * c, math.sqrt(2.0) * s


def test_relu_step_every_angle_and_scale_vs_mpmath(sm):
    """L = 1, relu, w = v = 1, b = 0, D = 2: K_ij = phi(k_ij; q_i, q_j) with q_i = r_i^2, k_ij = r_i r_j cos(phi_i -
    phi_j).  Every pair of rows: all angle differences, equal and different radii.  The reference evaluates the step in
    50 digits on the exact float inputs; each entry is held to 1e-15 sqrt(q_i q_j) (the step itself is good to
    2.5e-16, the rest covers the rounding of k in X.X^T / D)."""
    units = [_unit(p) for p in _row_angles()]
    x = np.array([[math.ldexp(a, e), math.ldexp(b, e)] for e in SCALE_EXPS for a, b in units])
    n = len(x)
    hp = dict(w_std=1.0, b_std=0.0, last_w_std=1.0, eps=1e-6, alpha=2.0, beta=2.0)
    (xd,) = _cuda(x)
    k = sm.device.gram(xd, spec=sm.StackSpec(1, "relu", "mlp"), hp=_hpd(sm, hp)).cpu().numpy()
    ref = np.empty((n, n))
    with mp.workdps(50):
        xm = [[mp.mpf(float(v)) for v in row] for row in x]
        q = [(r[0] * r[0] + r[1] * r[1]) / 2 for r in xm]
        for i in range(n):
            for j in range(i + 1):
                kij = (xm[i][0] * xm[j][0] + xm[i][1] * xm[j][1]) / 2
                ref[i, j] = ref[j, i] = float(act_off(kij, q[i], q[j], "relu"))
        scale = np.array([[float(mp.sqrt(q[i] * q[j])) for j in range(n)] for i in range(n)])
    err = np.abs(k - ref) / scale
    i, j = np.unravel_index(np.argmax(err), err.shape)
    assert err.max() <= 1e-15, (f"max |K - phi| / sqrt(q_i q_j) = {err.max():.3e} at radii 2^{SCALE_EXPS[i // len(units)]},"
                                f" 2^{SCALE_EXPS[j // len(units)]}: K {k[i, j]!r} vs {ref[i, j]!r}")


# ---- b. scale equivariance of every ReLU Gram path ---------------------------------------------------------------
@pytest.mark.parametrize("d", [13, 16])                     # odd D: cp.async-fed GEMM; D = 16: TMA-fed
@pytest.mark.parametrize("arch,L", [("mlp", 3), ("resnet", 2)])
def test_relu_gram_scale_equivariance(sm, d, arch, L):
    """relu with b_std = 0: K(c X) = c^2 K(X) for the symmetric Gram (full, and lower-only with eps_abs = c^2 eps), the
    cross Gram, nngp_diag and the grid search's recursion over a cached base Gram, at c = 2^-200 .. 2^200; entries
    within 1e-14 c^2 sqrt(K_ii K_jj)."""
    x, _, xt, *_ = regression_data(300, d, t=70, seed=d)
    hp = dict(w_std=1.2, b_std=0.0, last_w_std=0.9, eps=1e-3, alpha=2.0, beta=2.0)
    spec = sm.StackSpec(L, "relu", arch)
    kw = _kw(hp, L, "relu", arch)
    xd, xtd = _cuda(x, xt)
    hpd = _hpd(sm, hp)
    k1 = sm.device.gram(xd, spec=spec, hp=hpd).cpu().numpy()
    assert np.abs(k1 - orc.nngp_gram(x, **kw)).max() <= GRAM_TOL * np.abs(k1).max()
    kl1 = sm.device.gram(xd, spec=spec, hp=hpd, shift="eps_abs", lower_only=True).cpu().numpy()
    kx1 = sm.device.gram(xd, xtd, spec=spec, hp=hpd).cpu().numpy()
    q1 = sm.device.nngp_diag(xd, spec=spec, hp=hpd).cpu().numpy()
    qt1 = sm.device.nngp_diag(xtd, spec=spec, hp=hpd).cpu().numpy()
    assert np.abs(q1 - np.diag(k1)).max() <= 1e-14 * q1.max()
    sc = np.sqrt(np.outer(q1, q1))
    scx = np.sqrt(np.outer(q1, qt1))
    for e in SCALE_EXPS:
        c = 2.0 ** e
        c2 = c * c
        hpc = dict(hp, eps=hp["eps"] * c2)
        xc, xtc = _cuda(x * c, xt * c)
        hpcd = _hpd(sm, hpc)
        kc = sm.device.gram(xc, spec=spec, hp=hpcd).cpu().numpy()
        err = (np.abs(kc - c2 * k1) / (c2 * sc)).max()
        assert err <= 1e-14, f"c = 2^{e}: symmetric Gram, max |K(cX) - c^2 K(X)| / (c^2 sqrt(K_ii K_jj)) = {err:.3e}"
        assert np.array_equal(kc, kc.T)
        klc = sm.device.gram(xc, spec=spec, hp=hpcd, shift="eps_abs", lower_only=True).cpu().numpy()
        assert np.all(np.triu(klc, 1) == 0.0)
        err = (np.abs(klc - c2 * kl1) / (c2 * sc)).max()
        assert err <= 1e-14, f"c = 2^{e}: lower-only Gram + eps_abs, error {err:.3e}"
        kxc = sm.device.gram(xc, xtc, spec=spec, hp=hpcd).cpu().numpy()
        err = (np.abs(kxc - c2 * kx1) / (c2 * scx)).max()
        assert err <= 1e-14, f"c = 2^{e}: cross Gram, error {err:.3e}"
        qc = sm.device.nngp_diag(xc, spec=spec, hp=hpcd).cpu().numpy()
        assert (np.abs(qc - c2 * q1) / (c2 * q1)).max() <= 1e-14, f"c = 2^{e}: nngp_diag"


@pytest.mark.parametrize("arch,L,d", [("mlp", 3, 13), ("resnet", 2, 16)])
def test_relu_grid_search_and_predict_scale_equivariance(sm, arch, L, d):
    """The same homogeneity end to end: the grid search on its cached base Gram (gram_from_base) and from scratch, and
    predict with the relative regulariser eps tr(K) / N.  mean(c X) = mean(X), var(c X) = c^2 var(X); with the absolute
    jitter scaled as well, log det(c^2 A) = log det(A) + N log c^2 and quad(c^2 A) = quad(A) / c^2.  Runs Gram, Cholesky
    and finalize at pivots down to 2^-400."""
    import torch
    n, t = 300, 60
    x, y, xt, *_ = regression_data(n, d, t=t, seed=7)
    hp = dict(w_std=1.3, b_std=0.0, last_w_std=0.8, eps=1e-3, alpha=2.0, beta=2.0)
    spec = sm.StackSpec(L, "relu", arch)
    kw = _kw(hp, L, "relu", arch)
    xd, yd, xtd = _cuda(x, y, xt)
    hpd = _hpd(sm, hp)
    mean_ref, cov_ref = orc.nt_predict(x, y, xt, hp["eps"], kernel_kwargs=kw)
    m1, v1, info = sm.device.predict(xd, yd, xtd, spec=spec, hp=hpd)
    m1, v1 = m1.cpu().numpy()[:, 0], v1.cpu().numpy()
    assert int(info.item()) == 0
    assert np.abs(m1 - mean_ref[:, 0]).max() <= LML_TOL * np.abs(mean_ref).max()
    ktt = orc.nngp_diag(xt, **kw)
    assert np.all(np.abs(v1 - np.diag(cov_ref)) <= LML_TOL * np.abs(np.diag(cov_ref)) + 1e-13 * ktt)
    _, _, ld1, qd1, _ = sm.device.grid_point(xd, yd, xtd, spec=spec, hp=hpd)
    ld1, qd1 = float(ld1.item()), float(qd1.item())
    for e in SCALE_EXPS:
        c = 2.0 ** e
        c2 = c * c
        xc, xtc = _cuda(x * c, xt * c)
        hp_rel = hpd                                           # relative regulariser: eps stays
        hp_abs = _hpd(sm, dict(hp, eps=hp["eps"] * c2))        # absolute jitter scales with K
        mc, vc, info = sm.device.predict(xc, yd, xtc, spec=spec, hp=hp_rel)
        assert int(info.item()) == 0
        mc, vc = mc.cpu().numpy()[:, 0], vc.cpu().numpy()
        assert np.abs(mc - m1).max() <= LML_TOL * np.abs(m1).max(), f"c = 2^{e}: predictive mean"
        assert np.all(np.abs(vc - c2 * v1) <= LML_TOL * c2 * np.abs(v1) + 1e-13 * c2 * ktt), f"c = 2^{e}: variance"
        gs = sm.device.GridSearch(xc, yd, xtc, spec=spec)
        gm, gv, _, _, info = gs.point(hp_rel)
        assert int(info.item()) == 0
        assert np.abs(gm.cpu().numpy() - m1).max() <= LML_TOL * np.abs(m1).max(), f"c = 2^{e}: grid mean"
        assert np.all(np.abs(gv.cpu().numpy() - c2 * v1) <= LML_TOL * c2 * np.abs(v1) + 1e-13 * c2 * ktt)
        _, _, gld, gq, info = gs.point(hp_abs)
        _, _, sld, sq, info2 = sm.device.grid_point(xc, yd, xtc, spec=spec, hp=hp_abs)      # from scratch
        assert int(info.item()) == 0 and int(info2.item()) == 0
        shift = n * math.log(c2)
        for what, ld, q in (("grid search", gld, gq), ("from scratch", sld, sq)):
            ld, q = float(ld.item()), float(q.item())
            assert abs(ld - (ld1 + shift)) <= LML_TOL * (abs(ld1) + n), f"c = 2^{e}, {what}: log det {ld} vs {ld1 + shift}"
            assert abs(q * c2 - qd1) <= LML_TOL * abs(qd1), f"c = 2^{e}, {what}: quad {q * c2} vs {qd1}"
        del gs
        torch.cuda.synchronize()


# ---- c. deep stacks and small weights against the oracle -------------------------------------------------------
DEPTH_CASES = (
    # relu mlp: u shrinks by w^2 / 2 per layer (w = 1: halves; b = 1e-8 settles it near 2e-16)
    [("relu", "mlp", L, w, b) for L in (16, 32, 48, 64) for w in (0.5, 1.0, math.sqrt(2.0)) for b in (0.0, 1e-8)]
    + [("relu", "resnet", L, w, b) for L in (16, 64) for w in (0.5, 1.0, math.sqrt(2.0)) for b in (0.0, 1e-8)]
    + [("relu", arch, 3, w, b) for arch in ("mlp", "resnet") for w in (0.03, 0.01) for b in (0.0, 1e-8)]
    # erf: the control (its step has no floor).  w <= 1 only: at w^2 = 2 the erf recursion is in its chaotic phase and
    # amplifies rounding at every layer - one ulp of relative change in X moves the exact L = 64 mlp Gram by ~1e-10 of
    # max |K|, so no evaluation (the oracle's included) is good to GRAM_TOL there
    + [("erf", arch, L, w, 1e-8) for arch in ("mlp", "resnet") for L in (16, 64) for w in (0.5, 1.0)]
    + [("erf", "mlp", 3, 0.01, 0.0)]
)


@pytest.mark.parametrize("act,arch,L,w,b", DEPTH_CASES)
def test_gram_deep_and_small_weights_vs_oracle(sm, act, arch, L, w, b):
    x, *_ = regression_data(200, 13, seed=L)
    x[7] = x[3]                                           # a duplicate pair: s = 0 at every layer
    hp = dict(DEFAULT_HP, w_std=w, b_std=b, last_w_std=1.1)
    ref = orc.nngp_gram(x, **_kw(hp, L, act, arch))
    (xd,) = _cuda(x)
    k = sm.device.gram(xd, spec=sm.StackSpec(L, act, arch), hp=_hpd(sm, hp)).cpu().numpy()
    err = np.abs(k - ref).max() / np.abs(ref).max()
    assert err <= GRAM_TOL, f"gram err {err:.3e} (max |K| {np.abs(ref).max():.3e})"
    q = sm.device.nngp_diag(xd, spec=sm.StackSpec(L, act, arch), hp=_hpd(sm, hp)).cpu().numpy()
    qref = orc.nngp_diag(x, **_kw(hp, L, act, arch))
    assert np.abs(q - qref).max() <= 1e-12 * np.abs(qref).max()


def test_more_than_64_hidden_layers_rejected(sm):
    x, *_ = regression_data(20, 4)
    (xd,) = _cuda(x)
    hpd = _hpd(sm, DEFAULT_HP)
    sm.device.gram(xd, spec=sm.StackSpec(64, "relu", "mlp"), hp=hpd)
    with pytest.raises(RuntimeError, match=rf"\(status {SMNNGP_EINVAL}\)"):
        sm.device.gram(xd, spec=sm.StackSpec(65, "relu", "mlp"), hp=hpd)


# ---- d. the gradient in the same regimes ----------------------------------------------------------------------------
def _grad(sm, x, y, hp, L, act, arch, kind):
    import torch
    xd, yd = _cuda(x, y)
    out, grad, info = sm.device.lml_grad(xd, yd, spec=sm.StackSpec(L, act, arch),
                                         hp=torch.tensor([hp[k] for k in NAMES], dtype=torch.float64).cuda(), kind=kind)
    return out.cpu().numpy(), grad.cpu().numpy(), int(info.item())


def _assert_grad_close(grad, ref, what):
    tol = GRAD_TOL * np.abs(ref) + 1e-12 * np.abs(ref).max()
    assert np.all(np.abs(grad - ref) <= tol), f"{what}: grad {grad} vs {ref}: err {np.abs(grad - ref)} tol {tol}"


@pytest.mark.parametrize("e", SCALE_EXPS)
@pytest.mark.parametrize("arch,L,kind", [("mlp", 3, "student_t"), ("resnet", 2, "gauss")])
def test_grad_scaled_inputs_vs_oracle(sm, e, arch, L, kind):
    """inputs c X with the jitter c^2 eps: the same conditioning as the unscaled problem, so the same tolerance.
    Compared as theta * d loss / d theta: g_eps grows like c^-4 in the Gaussian case, the others like c^-2, and the
    absolute floor of the tolerance (relative to the largest component) must not swallow them."""
    x, y, *_ = regression_data(300, 13, seed=5)
    c = 2.0 ** e
    xc = x * c
    hp = dict(w_std=1.2, b_std=0.0, last_w_std=0.9, eps=1e-4 * c * c, alpha=2.5, beta=1.5)
    ref_loss, ref = orc.spr_loss_grad(xc, y, kind=kind, eps=hp["eps"], a=hp["alpha"], b=hp["beta"],
                                      **_kw(hp, L, "relu", arch))
    out, grad, info = _grad(sm, xc, y, hp, L, "relu", arch, kind)
    assert info == 0
    assert abs(out[1] - ref_loss) <= LML_TOL * abs(ref_loss)
    theta = np.array([hp[k] for k in NAMES])
    _assert_grad_close(theta * grad, theta * ref, f"c = 2^{e}")


@pytest.mark.parametrize("kind", ["student_t", "gauss"])
def test_grad_deep_relu_vs_oracle(sm, kind):
    """L = 48 at the reference's defaults (w_std = 1, b_std = 1e-8): the layer variance is ~4e-15 at the last layer"""
    x, y, *_ = regression_data(300, 13, seed=6)
    hp = dict(DEFAULT_HP)
    ref_loss, ref = orc.spr_loss_grad(x, y, kind=kind, eps=hp["eps"], a=hp["alpha"], b=hp["beta"],
                                      **_kw(hp, 48, "relu", "mlp"))
    out, grad, info = _grad(sm, x, y, hp, 48, "relu", "mlp", kind)
    assert info == 0
    assert abs(out[1] - ref_loss) <= LML_TOL * abs(ref_loss)
    _assert_grad_close(grad, ref, "L = 48")


def _assert_identity(lhs, rhs, terms, what):
    scale = max(abs(t) for t in terms)
    assert abs(lhs - rhs) <= IDENTITY_TOL * scale, f"{what}: {lhs!r} vs {rhs!r} (largest term {scale:.3e})"


def _check_identities(grad, out, hp, n, L, act, arch, kind):
    """exact identities of d loss / d (w_std, b_std, last_w_std, eps, alpha, beta):
    - K is homogeneous of degree 2 in last_w_std and the likelihood depends on (b/a)(K + eps I) (Student-t) or K + eps I
      (Gaussian), so scaling v^2, eps (and 1/beta) together gives (v/2) g_v + eps g_eps = beta g_beta (Student-t),
      = (N - quad) / (2 N) (Gaussian, quad = y^T (K + eps I)^-1 y = out[3]);
    - with b_std = 0, K depends on b_std only through b_std^2: g_b = 0 exactly;
    - relu mlp with b_std = 0: K is homogeneous of degree 2L in w_std, so w g_w = L v g_v."""
    w, v, eps, beta = hp["w_std"], hp["last_w_std"], hp["eps"], hp["beta"]
    tv, te = 0.5 * v * grad[2], eps * grad[3]
    if kind == "student_t":
        _assert_identity(tv + te, beta * grad[5], (tv, te, beta * grad[5]), "(v/2) g_v + eps g_eps = beta g_beta")
    else:
        _assert_identity(tv + te, (n - out[3]) / (2 * n), (tv, te, 0.5, out[3] / (2 * n)),
                         "(v/2) g_v + eps g_eps = (N - quad) / (2 N)")
    if hp["b_std"] == 0.0:
        assert grad[1] == 0.0, f"g_b = {grad[1]!r} with b_std = 0"
        if act == "relu" and arch == "mlp":
            _assert_identity(w * grad[0], L * v * grad[2], (w * grad[0], L * v * grad[2]), "w g_w = L v g_v")


@pytest.mark.parametrize("b_std", [0.0, 0.3])
@pytest.mark.parametrize("kind", ["student_t", "gauss"])
@pytest.mark.parametrize("act,arch,L", [("relu", "mlp", 3), ("relu", "resnet", 2), ("erf", "mlp", 3),
                                        ("erf", "resnet", 2), ("relu", "mlp", 48)])
def test_grad_exact_identities(sm, act, arch, L, kind, b_std):
    n = 1500
    x, y, *_ = regression_data(n, 16, seed=9)
    hp = dict(w_std=1.3, b_std=b_std, last_w_std=0.8, eps=1e-4, alpha=2.5, beta=1.5)
    out, grad, info = _grad(sm, x, y, hp, L, act, arch, kind)
    assert info == 0 and np.all(np.isfinite(grad))
    _check_identities(grad, out, hp, n, L, act, arch, kind)


# ---- 3. the value and gradient at BASELINE config 3 size -------------------------------------------------------------
def test_c3_full_size_gradient(sm):
    """N = 60 000, D = 784 (what bench.py's value_and_gradient line measures): the value against the recorded oracle,
    the exact identities, g_alpha and g_beta against their closed forms in 50 digits from the device's own quad, and
    bitwise reproducibility of the gradient.  lml_grad needs 16 N^2 bytes of workspace."""
    import torch
    path = os.path.join(os.path.dirname(__file__), "golden", "c3_full.json")
    with open(path) as f:
        g = json.load(f)
    if g.get("oracle_loss") is None:
        pytest.skip("tests/golden/c3_full.json holds no oracle value yet")
    if torch.cuda.get_device_properties(0).total_memory < 80e9:
        pytest.skip("needs 80 GB of device memory")
    n = g["n"]
    x, y, *_ = pixel_data(n, g["d"], seed=g["seed"])
    xd, yd = _cuda(x, y)
    del x
    hp = dict(g["hp"])
    spec = sm.StackSpec(3, "relu", "mlp")

    def call(h):
        hd = _hpd(sm, h)
        out, grad, info = sm.device.lml_grad(xd, yd, spec=spec, hp=hd)
        return out.cpu().numpy(), grad.cpu().numpy(), int(info.item()), hd

    sm.device.release_workspaces()
    torch.cuda.empty_cache()
    try:
        out, grad, info, hd = call(hp)
        assert info == 0
        assert abs(out[1] - g["oracle_loss"]) <= LML_TOL * abs(g["oracle_loss"]), (out[1], g["oracle_loss"])
        out_v, info_v = sm.device.lml(xd, yd, spec=spec, hp=hd)
        assert int(info_v.item()) == 0 and np.array_equal(out_v.cpu().numpy(), out)
        _check_identities(grad, out, hp, n, 3, "relu", "mlp", "student_t")
        with mp.workdps(50):
            a, b, quad = mp.mpf(hp["alpha"]), mp.mpf(hp["beta"]), mp.mpf(float(out[3]))
            t = a + mp.mpf(n) / 2
            g_alpha = float(-(-mp.log1p(quad / (2 * b)) + mp.digamma(t) - mp.digamma(a)) / n)
            g_beta = float(-(t * quad / (b * (2 * b + quad)) - mp.mpf(n) / (2 * b)) / n)
        assert abs(grad[4] - g_alpha) <= 1e-12 * abs(g_alpha), (grad[4], g_alpha)
        assert abs(grad[5] - g_beta) <= 1e-11 * abs(g_beta), (grad[5], g_beta)
        _, grad2, info2, _ = call(hp)
        assert info2 == 0 and np.array_equal(grad2, grad), (grad2, grad)
        hp0 = dict(hp, b_std=0.0)
        out0, grad0, info0, _ = call(hp0)
        assert info0 == 0
        _check_identities(grad0, out0, hp0, n, 3, "relu", "mlp", "student_t")
    finally:
        del xd, yd
        sm.device.release_workspaces()
        torch.cuda.empty_cache()
