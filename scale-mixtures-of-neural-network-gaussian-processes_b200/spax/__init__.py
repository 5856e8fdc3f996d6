from .kernels import NNGPKernel
from .likelihoods import Likelihood, GaussianLikelihood, StudentTLikelihood
from .models import SPR, DistributedSPR, MultiStartSPR
from .utils import jitter, multivariate_t_logpdf, multivariate_normal_logpdf
from .base import Module, TrainVar, ConstraintTrainVar
from .bijectors import positive
from .priors import Prior, GaussianPrior, InverseGammaPrior
from .optimizer import Adam, BatchAdam
