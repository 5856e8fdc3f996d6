"""Likelihoods with the interface of spax/likelihoods.py:18-65 (prior_logpdf / logpdf / require)."""
import math

import torch

from .base import Module, ConstraintTrainVar
from .bijectors import positive
from .utils import multivariate_t_logpdf, multivariate_normal_logpdf
from .. import device as _dev

__all__ = ["Likelihood", "GaussianLikelihood", "StudentTLikelihood", "BurrXIILikelihood"]


def _diag(cov):
    return cov if cov.ndim == 1 else torch.diagonal(cov)


class Likelihood(Module):
    kind = None


class GaussianLikelihood(Likelihood):
    require = None
    kind = "gauss"

    def prior_logpdf(self, x, cov):
        return multivariate_normal_logpdf(x, 0.0, cov)                       # likelihoods.py:25-28

    def logpdf(self, x, mean, cov, aux=None):
        sigma = torch.sqrt(_diag(cov))                                       # likelihoods.py:30-33
        z = (x - mean) / sigma
        return -0.5 * math.log(2 * math.pi) - torch.log(sigma) - 0.5 * z * z


class StudentTLikelihood(Likelihood):
    require = ["cov_data", "y_data"]
    kind = "student_t"

    def __init__(self, alpha, beta):
        self.a = ConstraintTrainVar(alpha, constraint=positive())
        self.b = ConstraintTrainVar(beta, constraint=positive())

    def prior_logpdf(self, x, cov):
        a, b = self.a.safe_value, self.b.safe_value                          # likelihoods.py:45-50
        return multivariate_t_logpdf(x, 0.0, (b / a) * cov, 2 * a)

    def logpdf(self, x, mean, cov, aux):
        a, b = self.a.safe_value, self.b.safe_value                          # likelihoods.py:52-65
        cov_data, y_data = aux
        num_data = cov_data.shape[-1]
        df = 2 * a
        cond_df = df + num_data
        # y^T ((b/a) cov_data + 1e-6 I)^-1 y through a Cholesky solve instead of the reference's LU inverse
        _, quad, _ = _dev.cov_solve(cov_data, y_data, scale=b / a, shift=1e-6)
        d = df + quad
        sigma = torch.sqrt(d / cond_df * b / a * _diag(cov))
        z = (x - mean) / sigma
        norm = (math.lgamma(cond_df / 2) + 0.5 * math.log(cond_df) + 0.5 * torch.log(sigma * sigma * math.pi)
                - math.lgamma((cond_df + 1) / 2))
        return -(norm + (cond_df + 1) / 2 * torch.log1p(z * z / cond_df))


class BurrXIILikelihood(Likelihood):
    """Scale mixture of NNGPs with a Burr Type XII prior on the output scale (CDF 1 - (1 + s^c)^-k): y | s ~ N(0, s A).
    The prior has no conjugate form, so ``SPR.loss`` and ``SPR.test_nll`` importance-sample the scale over
    ``num_samples`` prior draws (``device.scale_draws`` with a fixed ``seed``: every evaluation sees the same draws).
    Only the fused path of an smnngp ``KernelFn`` evaluates it, and there is no gradient."""
    require = None
    kind = "burr12"

    def __init__(self, c, k, *, num_samples=1000, seed=0):
        self.c = ConstraintTrainVar(c, constraint=positive())
        self.k = ConstraintTrainVar(k, constraint=positive())
        self.num_samples = int(num_samples)
        self.seed = int(seed)

    def draws(self, device):
        """[1, num_samples] scale draws of the current (c, k)"""
        params = torch.tensor([[self.c.safe_value, self.k.safe_value]], dtype=torch.float64, device=device)
        return _dev.scale_draws("burr12", params, self.num_samples, seed=self.seed)
