"""Reference for the scale mixture (``csrc/mixture.cu``), NumPy / SciPy only, FP64.  TEST INFRASTRUCTURE ONLY, like
``oracle/``, on which it builds:

* ``scale_draws`` replicates ``smnngp_scale_draws_f64`` with the generator of ``oracle/draws_ref.py``: draw j of prior
  row p uses the counter (j, p, 0xFFFFFFFF, n); s = b / gamma(a) (inverse gamma) or, from one uniform u,
  s = exp(log(expm1(-log u / k)) / c) (Burr XII);
* ``mixture_nll`` is the importance-sampling estimator of ``smnngp_mixture_nll_f64`` (``scipy.special.logsumexp``);
* ``mixture_quadrature`` and ``invgamma_mixture_closed_form`` are exact values it converges to, and ``mixture_se`` its
  delta-method standard errors.
"""
from __future__ import annotations

import numpy as np
from scipy.special import gammaln

from oracle.draws_ref import _Cells
from oracle.nngp_oracle import _t_logpdf

__all__ = ["scale_draws", "mixture_nll", "mixture_quadrature", "invgamma_mixture_closed_form", "mixture_se"]


SCALE_FAMILIES = ("invgamma", "burr12")


def scale_draws(family, params, S, seed):
    """The draws of ``smnngp_scale_draws_f64``: params [P, 2] ((a, b) for "invgamma", (c, k) for "burr12").

    Returns (draws, margin), each [P, S]: the scales and the smallest |margin| of each draw's gamma decisions (inf for
    Burr XII draws, which take none).  A row with a parameter <= 0 or not finite gives NaN draws."""
    if family not in SCALE_FAMILIES:
        raise ValueError(f"unknown family {family!r}")
    params = np.asarray(params, dtype=np.float64).reshape(-1, 2)
    P, S = params.shape[0], int(S)
    draws = np.full((P, S), np.nan)
    margin = np.full((P, S), np.inf)
    j = np.arange(S, dtype=np.int64)
    idx = np.arange(S)
    for p, (a, b) in enumerate(params):
        if not (a > 0.0 and b > 0.0 and np.isfinite(a) and np.isfinite(b)):
            continue
        cells = _Cells(seed, j, np.full(S, p), np.full(S, 0xFFFFFFFF))
        if family == "invgamma":
            g, margin[p] = cells.gamma(float(a), idx)
            with np.errstate(divide="ignore"):
                draws[p] = b / g
        else:
            u = cells.uniform(idx)
            with np.errstate(divide="ignore", over="ignore"):
                draws[p] = np.exp(np.log(np.expm1(-np.log(u) / b)) / a)
    return draws, margin


# ----------------------------------------------------------------------------------------------------------
# scale mixture of the output scale by importance sampling (find.py:163-191, smnngp_mixture_nll_f64):
# y | s ~ N(0, s A), f_t | y, s ~ N(m_t, s v_t), scale draws s_j from the prior
# ----------------------------------------------------------------------------------------------------------
def _mixture_ell(s, n, quad):
    """l_j = -(n/2) log s_j - quad / (2 s_j), -inf for s_j = 0 or +inf (NaN stays NaN)"""
    s = np.asarray(s, dtype=np.float64)
    edge = (s == 0.0) | (s == np.inf)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        ell = -0.5 * n * np.log(s) - quad / (2.0 * s)
    return np.where(edge, -np.inf, ell), edge


def mixture_nll(scal, mean, var, y_test, n, draws, y_mean, y_std):
    """The importance-sampling estimator of the scale mixture at every (grid point g, draw row p): scal [G, 2] =
    {sum log L_ii, y^T A^-1 y} of A = K + eps I, mean / var [G, T] the predictive (standardised), y_test [T]
    (standardised), n training rows, draws [P, S].  Returns (nll, lml, ess) [G, P] and logp [G, P, T]; with T = 0
    (y_test None) nll and logp are None."""
    from scipy.special import logsumexp
    scal = np.asarray(scal, dtype=np.float64).reshape(-1, 2)
    draws = np.asarray(draws, dtype=np.float64)
    G, (P, S) = scal.shape[0], draws.shape
    T = 0 if y_test is None else len(y_test)
    lml, ess = np.empty((G, P)), np.empty((G, P))
    nll = np.empty((G, P)) if T else None
    logp = np.empty((G, P, T)) if T else None
    if T:
        yt = np.asarray(y_test, dtype=np.float64) * y_std + y_mean
        mt = np.asarray(mean, dtype=np.float64).reshape(G, T) * y_std + y_mean
        vt = np.asarray(var, dtype=np.float64).reshape(G, T) * y_std ** 2
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for g in range(G):
            logdet, quad = scal[g]
            for p in range(P):
                ell, edge = _mixture_ell(draws[p], n, quad)
                lse = logsumexp(ell)
                lml[g, p] = lse - np.log(S) - logdet - 0.5 * n * np.log(2 * np.pi)
                top = np.max(ell)
                w = np.exp(ell - top)
                ess[g, p] = 0.0 if top == -np.inf else w.sum() ** 2 / (w * w).sum()
                if T:
                    sv = draws[p][:, None] * vt[g][None, :]                                    # [S, T]
                    lnorm = -0.5 * np.log(2 * np.pi * sv) - (yt - mt[g]) ** 2 / (2.0 * sv)
                    term = np.where(edge[:, None], -np.inf, ell[:, None] + lnorm)
                    logp[g, p] = logsumexp(term, axis=0) - lse
                    nll[g, p] = -np.mean(logp[g, p])
                if np.isnan(logdet) or np.isnan(quad):
                    lml[g, p] = ess[g, p] = np.nan
                    if T:
                        logp[g, p] = nll[g, p] = np.nan
    return nll, lml, ess, logp


def mixture_quadrature(log_prior, logdet, quad, n, mean=None, var=None, y_test=None, y_mean=0.0, y_std=1.0):
    """Exact lml and logp [T] of the scale mixture with prior density exp(log_prior(s)): 1-D adaptive quadrature over
    u = log s (integrand pi(s) s exp(l(s))), centred at log(quad / n) and scaled by the integrand's maximum."""
    from scipy import integrate
    c = np.log(quad / n)
    lo, hi = c - 40.0, c + 40.0

    def f(u):
        s = np.exp(u)
        return log_prior(s) + u - 0.5 * n * u - quad / (2.0 * s)

    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        grid = np.linspace(lo, hi, 8001)
        vals = np.array([f(u) for u in grid])
        top = np.nanmax(vals)
        u0 = grid[np.nanargmax(vals)]
        opts = dict(limit=500, epsabs=0.0, epsrel=1e-13, points=[c, u0])
        Z = integrate.quad(lambda u: np.exp(f(u) - top), lo, hi, **opts)[0]
        lml = np.log(Z) + top - logdet - 0.5 * n * np.log(2 * np.pi)
        if y_test is None:
            return lml, None
        yt = np.asarray(y_test, dtype=np.float64) * y_std + y_mean
        mt = np.asarray(mean, dtype=np.float64) * y_std + y_mean
        vt = np.asarray(var, dtype=np.float64) * y_std ** 2
        logp = np.empty(len(yt))
        for t in range(len(yt)):
            def ft(u, t=t):
                sv = np.exp(u) * vt[t]
                return np.exp(f(u) - top - 0.5 * np.log(2 * np.pi * sv) - (yt[t] - mt[t]) ** 2 / (2.0 * sv))
            logp[t] = np.log(integrate.quad(ft, lo, hi, **opts)[0] / Z)
    return lml, logp


def invgamma_mixture_closed_form(a, b, logdet, quad, n, mean=None, var=None, y_test=None, y_mean=0.0, y_std=1.0):
    """The scale mixture under an inverse-gamma IG(a, b) prior in closed form: y is multivariate t_{2a} with shape
    (b / a) A, and f_t | y is t_{2a + n}(m~_t, v~_t (2b + quad) / (2a + n)).  Returns (lml, logp [T] or None)."""
    lml = (gammaln(a + 0.5 * n) - gammaln(a) + a * np.log(b) - (a + 0.5 * n) * np.log(b + 0.5 * quad) - logdet
           - 0.5 * n * np.log(2 * np.pi))
    if y_test is None:
        return lml, None
    yt = np.asarray(y_test, dtype=np.float64) * y_std + y_mean
    mt = np.asarray(mean, dtype=np.float64) * y_std + y_mean
    vt = np.asarray(var, dtype=np.float64) * y_std ** 2
    df = 2.0 * a + n
    return lml, _t_logpdf(yt, df, mt, np.sqrt(vt * (2.0 * b + quad) / df))


def mixture_se(draws, logdet, quad, n, mean=None, var=None, y_test=None, y_mean=0.0, y_std=1.0):
    """Delta-method standard errors of the estimator of ``mixture_nll`` for one (g, p): (se of lml, se of logp [T],
    se of nll).  lml = log mean(w) + const has se sd(w) / (sqrt(S) mean(w)); logp_t = log(mean(w f_t) / mean(w)) is a
    ratio estimator with se sd(w f_t / mean(w f_t) - w / mean(w)) / sqrt(S)."""
    draws = np.asarray(draws, dtype=np.float64)
    S = draws.size
    ell, edge = _mixture_ell(draws, n, quad)
    w = np.exp(ell - ell.max())
    se_lml = w.std() / (np.sqrt(S) * w.mean())
    if y_test is None:
        return se_lml, None, None
    yt = np.asarray(y_test, dtype=np.float64) * y_std + y_mean
    mt = np.asarray(mean, dtype=np.float64) * y_std + y_mean
    vt = np.asarray(var, dtype=np.float64) * y_std ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        sv = draws[:, None] * vt[None, :]
        lf = -0.5 * np.log(2 * np.pi * sv) - (yt - mt) ** 2 / (2.0 * sv)
        lf = np.where(edge[:, None], -np.inf, lf)
    wf = w[:, None] * np.exp(lf - lf.max(axis=0))                       # [S, T], a constant factor per t cancels
    z = wf / wf.mean(axis=0) - (w / w.mean())[:, None]
    se_logp = z.std(axis=0) / np.sqrt(S)
    se_nll = z.mean(axis=1).std() / np.sqrt(S)
    return se_lml, se_logp, se_nll
