"""The scale mixture without a GPU: the replica's scale draws against scipy, the quadrature against the inverse-gamma
closed form, the NumPy estimator against both, the point mass against the Gaussian densities, and the argument checks
of the two C entry points."""
import ctypes as C

import numpy as np
import pytest
import scipy.stats as st

from tests import mixture_ref as mr

SMNNGP_EINVAL = 1


@pytest.mark.parametrize("c,k", [(0.5, 0.5), (1.7, 0.6), (3.0, 2.0), (10.0, 0.1)])
def test_replica_burr12_draws_are_burr12(c, k):
    s, margin = mr.scale_draws("burr12", [[c, k]], 50000, seed=20261022)
    assert np.all(margin == np.inf) and np.all(s >= 0)
    assert st.kstest(s[0], st.burr12(c, k).cdf).pvalue > 1e-3


@pytest.mark.parametrize("a", [0.3, 1.0, 2.5, 40.0])
def test_replica_invgamma_draws_are_invgamma(a):
    b = 1.7
    s, _ = mr.scale_draws("invgamma", [[a, b]], 50000, seed=20261022)
    assert np.all(s > 0)
    assert st.kstest(s[0], st.invgamma(a, scale=b).cdf).pvalue > 1e-3


def test_replica_rows_are_independent_streams_and_invalid_rows_are_nan():
    prm = [[1.7, 0.6], [1.7, 0.6], [0.0, 1.0], [np.inf, 1.0], [1.0, np.nan]]
    s, _ = mr.scale_draws("burr12", prm, 100, seed=3)
    assert not np.any(s[0] == s[1])
    assert np.isnan(s[2:]).all()
    s2, _ = mr.scale_draws("burr12", prm[:1], 100, seed=3)
    assert np.array_equal(s2[0], s[0])


def _problem(n, t, seed=0):
    """A = X X^T / n + I / 2, y, and a predictive (m, v) at t test points"""
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n, n))
    a = x @ x.T / n + 0.5 * np.eye(n)
    y = rng.normal(size=n)
    logdet = np.log(np.diag(np.linalg.cholesky(a))).sum()
    quad = float(y @ np.linalg.solve(a, y))
    return a, y, logdet, quad, rng.normal(size=t), rng.uniform(0.2, 1.0, t), rng.normal(size=t)


YM, YS = 0.37, 1.9


@pytest.mark.parametrize("n", [6, 17])
@pytest.mark.parametrize("a,b", [(2.0, 2.0), (0.7, 3.0)])
def test_quadrature_is_the_invgamma_closed_form(n, a, b):
    A, y, logdet, quad, m, v, yt = _problem(n, 3)
    cl, cp = mr.invgamma_mixture_closed_form(a, b, logdet, quad, n, m, v, yt, YM, YS)
    ql, qp = mr.mixture_quadrature(lambda s: st.invgamma(a, scale=b).logpdf(s), logdet, quad, n, m, v, yt, YM, YS)
    assert abs(ql - cl) <= 1e-10 * abs(cl)
    assert np.all(np.abs(qp - cp) <= 1e-10 * np.abs(cp))
    # the closed form is the multivariate t of the reference's Student-t prior
    assert abs(cl - st.multivariate_t(loc=np.zeros(n), shape=(b / a) * A, df=2 * a).logpdf(y)) <= 1e-12 * abs(cl)


@pytest.mark.parametrize("n", [6, 17])
@pytest.mark.parametrize("family", ["invgamma", "burr12"])
def test_estimator_converges_to_the_exact_values(n, family):
    """2^20 prior draws: lml, logp and nll within 5 delta-method standard errors of the closed form (inverse gamma) or
    of the quadrature (Burr XII)"""
    A, y, logdet, quad, m, v, yt = _problem(n, 4, seed=n)
    if family == "invgamma":
        a, b = 2.0, 2.0
        draws = st.invgamma(a, scale=b).rvs(size=2**20, random_state=n)
        xl, xp = mr.invgamma_mixture_closed_form(a, b, logdet, quad, n, m, v, yt, YM, YS)
    else:
        c, k = 1.7, 0.6
        draws = st.burr12(c, k).rvs(size=2**20, random_state=n)
        xl, xp = mr.mixture_quadrature(lambda s: st.burr12(c, k).logpdf(s), logdet, quad, n, m, v, yt, YM, YS)
    nll, lml, ess, logp = mr.mixture_nll([[logdet, quad]], m[None], v[None], yt, n, draws[None], YM, YS)
    se_lml, se_logp, se_nll = mr.mixture_se(draws, logdet, quad, n, m, v, yt, YM, YS)
    assert 1.0 < ess[0, 0] <= 2**20
    assert abs(lml[0, 0] - xl) <= 5 * se_lml, (lml[0, 0], xl, se_lml)
    assert np.all(np.abs(logp[0, 0] - xp) <= 5 * se_logp), (logp[0, 0], xp, se_logp)
    assert abs(nll[0, 0] + xp.mean()) <= 5 * se_nll, (nll[0, 0], -xp.mean(), se_nll)


@pytest.mark.parametrize("s0", [1.0, 0.37, 12.5])
def test_point_mass_is_the_gaussian_of_the_scaled_covariance(s0):
    n, S = 9, 1000
    A, y, logdet, quad, m, v, yt = _problem(n, 5, seed=3)
    nll, lml, ess, logp = mr.mixture_nll([[logdet, quad]], m[None], v[None], yt, n, np.full((1, S), s0), YM, YS)
    ref_lml = st.multivariate_normal(np.zeros(n), s0 * A).logpdf(y)
    ref_logp = st.norm.logpdf(yt * YS + YM, m * YS + YM, np.sqrt(s0 * v) * YS)
    assert ess[0, 0] == S
    assert abs(lml[0, 0] - ref_lml) <= 1e-13 * abs(ref_lml)
    assert np.all(np.abs(logp[0, 0] - ref_logp) <= 1e-13 * np.maximum(1.0, np.abs(ref_logp)))
    assert abs(nll[0, 0] + ref_logp.mean()) <= 1e-13 * abs(ref_logp.mean())


def test_estimator_edge_draws():
    n = 8
    A, y, logdet, quad, m, v, yt = _problem(n, 3, seed=4)
    draws = np.array([[0.0, 1e-300, 1e300, np.inf, 1.0, 2.0], [0.0, np.inf, 0.0, np.inf, 0.0, np.inf],
                      [1.0, 2.0, np.nan, 1.0, 1.0, 1.0]])
    with np.errstate(all="ignore"):
        nll, lml, ess, logp = mr.mixture_nll([[logdet, quad], [np.nan, quad]], np.stack([m, m]), np.stack([v, v]),
                                             yt, n, draws, YM, YS)
    assert np.isfinite([nll[0, 0], lml[0, 0], ess[0, 0]]).all() and np.isfinite(logp[0, 0]).all()
    assert ess[0, 1] == 0.0 and lml[0, 1] == -np.inf and np.isnan(nll[0, 1]) and np.isnan(logp[0, 1]).all()
    assert np.isnan([nll[0, 2], lml[0, 2], ess[0, 2]]).all()
    assert np.isnan(nll[1]).all() and np.isnan(lml[1]).all() and np.isnan(ess[1]).all() and np.isnan(logp[1]).all()


# ---- the C-ABI's argument checks (they run before anything touches a device) -----------------------------------
@pytest.fixture(scope="module")
def lib():
    import smnngp_b200 as sm
    assert "smnngp_scale_draws_f64" in sm._lib.EXPORTS and "smnngp_mixture_nll_f64" in sm._lib.EXPORTS
    return sm._lib.load()


def _check_rejects(lib, name, call, cases):
    for over in cases:
        lib.smnngp_lml_host_f64(None, None, 0, 0, 0, 0, 0, None, 0, None, None)     # leaves another call's message
        assert name.encode() not in lib.smnngp_last_error()
        lib.smnngp_instr_reset(0)
        assert call(**over) == SMNNGP_EINVAL, (name, over)
        assert lib.smnngp_instr_launches() == 0, (name, over)
        assert name.encode() in lib.smnngp_last_error(), (name, over, lib.smnngp_last_error())


PTR = C.c_void_p(256)                  # never dereferenced: every case below is rejected first


def test_scale_draws_rejects_bad_arguments(lib):
    good = dict(family=1, params=PTR, P=3, S=100, out=PTR)

    def call(**over):
        a = dict(good, **over)
        return lib.smnngp_scale_draws_f64(None, a["family"], a["params"], a["P"], a["S"], 7, a["out"])

    _check_rejects(lib, "smnngp_scale_draws_f64", call, [
        dict(P=0), dict(S=0), dict(P=-1), dict(S=-4), dict(P=2**31), dict(S=2**31), dict(family=2), dict(family=-1),
        dict(params=None), dict(out=None)])


def test_mixture_nll_rejects_bad_arguments(lib):
    good = dict(scal=PTR, mean=PTR, var=PTR, ld=5, yt=PTR, N=10, T=5, G=3, draws=PTR, P=2, S=100, y_std=1.0,
                nll=PTR, lml=PTR, ess=PTR)

    def call(**over):
        a = dict(good, **over)
        return lib.smnngp_mixture_nll_f64(None, a["scal"], a["mean"], a["var"], a["ld"], a["yt"], a["N"], a["T"],
                                          a["G"], a["draws"], a["P"], a["S"], 0.0, a["y_std"], a["nll"], a["lml"],
                                          a["ess"], None)

    _check_rejects(lib, "smnngp_mixture_nll_f64", call, [
        dict(N=0), dict(G=0), dict(P=0), dict(S=0), dict(N=-1), dict(T=-1), dict(ld=4), dict(y_std=0.0),
        dict(y_std=-1.0), dict(y_std=float("inf")), dict(y_std=float("nan")), dict(scal=None), dict(draws=None),
        dict(lml=None), dict(ess=None), dict(mean=None), dict(var=None), dict(yt=None), dict(nll=None),
        dict(G=2**40, P=2**40), dict(P=2**40, S=2**40), dict(G=2**31, P=2**31, T=8, ld=8), dict(G=4, ld=2**62)])
