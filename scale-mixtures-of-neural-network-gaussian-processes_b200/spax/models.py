"""SPR with the interface of spax/models.py:81-120.  When the kernel closure is an smnngp ``KernelFn`` and the
likelihood is one of ours, ``loss`` and ``test_nll`` are single fused C-ABI calls (Gram never leaves the
device, solves fused into the factorisation); otherwise they compose K / prior_logpdf / predict / logpdf
exactly like the reference does - every piece still on the CUDA path."""
import numpy as np
import torch

from .base import Module, ConstraintTrainVar
from .bijectors import positive
from .utils import jitter
from .. import device as _dev
from ..nt_kernels import KernelFn

__all__ = ["SPR", "DistributedSPR", "MultiStartSPR"]


class SPR(Module):
    def __init__(self, kernel, likelihood, x_data, y_data, y_mean, y_std, *, eps: float = 1e-6):
        self.kernel = kernel
        self.likelihood = likelihood
        self.x_data = x_data
        self.y_data = y_data
        self.y_mean = y_mean
        self.y_std = y_std
        self.num_data = x_data.shape[0]
        self.eps = ConstraintTrainVar(eps, constraint=positive())

    def _hp_args(self):
        lik = self.likelihood
        a = lik.a.safe_value if hasattr(lik, "a") else 2.0
        b = lik.b.safe_value if hasattr(lik, "b") else 2.0
        return dict(eps=self.eps.safe_value, alpha=a, beta=b)

    def _fused(self, kernel_fn):
        return isinstance(kernel_fn, KernelFn) and getattr(self.likelihood, "kind", None) in _dev.KIND

    def _mixture(self, kernel_fn):
        """Whether the likelihood is an importance-sampled scale mixture (BurrXIILikelihood); it needs the fused path"""
        if getattr(self.likelihood, "kind", None) != "burr12":
            return False
        if not isinstance(kernel_fn, KernelFn):
            raise TypeError("BurrXIILikelihood needs a kernel_fn built by smnngp nt_kernels")
        return True

    def _mixture_pieces(self, kernel_fn):
        """(x, y, hp, scal [1, 2], draws [1, S]) on the device: {sum log L_ii, y^T A^-1 y} of A = K + eps I from the
        Gaussian LML and the likelihood's scale draws"""
        x = _dev._f64(self.x_data, "cuda" if not isinstance(self.x_data, torch.Tensor) else None)
        y = _dev._f64(self.y_data, x.device)
        hp = kernel_fn.hp(x.device, **self._hp_args())
        out, _ = _dev.lml(x, y, spec=kernel_fn.spec, hp=hp, kind="gauss")
        return x, y, hp, out[2:4].reshape(1, 2), self.likelihood.draws(x.device)

    def loss(self):
        kernel_fn = self.kernel.get_kernel_fn()
        if self._mixture(kernel_fn):
            x, _, _, scal, draws = self._mixture_pieces(kernel_fn)
            _, lml, _, _ = _dev.mixture_nll(scal, None, None, None, self.num_data, draws, 0.0, 1.0)
            loss = -lml[0, 0] / self.num_data
            return float(loss) if isinstance(self.x_data, np.ndarray) else loss
        if self._fused(kernel_fn):
            host = isinstance(self.x_data, np.ndarray)
            hp = kernel_fn.hp_host(**self._hp_args()) if host else kernel_fn.hp(self.x_data.device, **self._hp_args())
            out, _ = _dev.lml(self.x_data, self.y_data, spec=kernel_fn.spec, hp=hp, kind=self.likelihood.kind)
            return float(out[1]) if host else out[1]
        eps = self.eps.safe_value
        cov = self.kernel.K(kernel_fn, self.x_data) + jitter(self.num_data, eps=eps, device=self.x_data.device)
        log_prob = self.likelihood.prior_logpdf(self.y_data, cov)
        return -log_prob / self.num_data

    def loss_and_grad(self):
        """(loss, grads): the pair ``objax.GradValues(model.loss, model.vars())`` returns in the reference's train
        step (experiments/regression/train.py:62-66), as one fused call.  ``grads`` maps the names of
        ``self.vars()`` to d loss / d (unconstrained variable value) - the softplus chain rule
        (spax/base.py:23-25, spax/bijectors.py:51-53) is applied here.  Scalars the likelihood does not own
        (Gaussian: alpha, beta) are absent."""
        kernel_fn = self.kernel.get_kernel_fn()
        if getattr(self.likelihood, "kind", None) == "burr12":
            raise TypeError("loss_and_grad: the importance-sampled scale mixture (BurrXIILikelihood) has no gradient")
        if not self._fused(kernel_fn):
            raise TypeError("loss_and_grad needs a kernel_fn built by smnngp nt_kernels and a spax likelihood")
        host = isinstance(self.x_data, np.ndarray)
        hp = kernel_fn.hp_host(**self._hp_args()) if host else kernel_fn.hp(self.x_data.device, **self._hp_args())
        out, grad, _ = _dev.lml_grad(self.x_data, self.y_data, spec=kernel_fn.spec, hp=hp, kind=self.likelihood.kind)
        g = grad if host else grad.cpu().numpy()
        loss = float(out[1])
        slots = {"kernel.w_std": (self.kernel.w_std, 0), "kernel.b_std": (self.kernel.b_std, 1),
                 "kernel.last_w_std": (self.kernel.last_w_std, 2), "eps": (self.eps, 3)}
        if hasattr(self.likelihood, "a"):
            slots["likelihood.a"] = (self.likelihood.a, 4)
            slots["likelihood.b"] = (self.likelihood.b, 5)
        grads = {name: float(g[i]) * float(var.constraint.grad(var.value)) for name, (var, i) in slots.items()}
        return loss, grads

    def test_nll(self, x, y):
        kernel_fn = self.kernel.get_kernel_fn()
        if self._mixture(kernel_fn):
            xd, yd, hp, scal, draws = self._mixture_pieces(kernel_fn)
            xt, yt = _dev._f64(x, xd.device), _dev._f64(y, xd.device)
            mean, var, _ = _dev.predict(xd, yd, xt, spec=kernel_fn.spec, hp=hp, shift="eps_rel")
            nll, _, _, _ = _dev.mixture_nll(scal, mean.reshape(1, -1), var.reshape(1, -1), yt, self.num_data, draws,
                                            float(self.y_mean), float(self.y_std))
            return float(nll[0, 0]) if isinstance(self.x_data, np.ndarray) else nll[0, 0]
        if self._fused(kernel_fn):
            host = isinstance(self.x_data, np.ndarray)
            hp = kernel_fn.hp_host(**self._hp_args()) if host else kernel_fn.hp(self.x_data.device, **self._hp_args())
            nll, _, _, _ = _dev.test_nll(self.x_data, self.y_data, x, y, float(self.y_mean), float(self.y_std),
                                         spec=kernel_fn.spec, hp=hp, kind=self.likelihood.kind)
            return nll
        eps = self.eps.safe_value
        mean, cov = self.kernel.predict(kernel_fn, self.x_data, self.y_data[:, None], x, eps=eps)
        require = self.likelihood.require
        if require:
            aux_dict = dict(y_data=self.y_data)
            if "cov_data" in require:
                aux_dict["cov_data"] = self.kernel.K(kernel_fn, self.x_data)      # models.py:107, no jitter
            aux = tuple(aux_dict[k] for k in require)
        else:
            aux = None
        log_prob = self.likelihood.logpdf((y * self.y_std) + self.y_mean, (mean.flatten() * self.y_std) + self.y_mean,
                                          cov * self.y_std ** 2, aux)
        return -torch.mean(log_prob)



class DistributedSPR(SPR):
    """SPR whose device work is sharded over the ranks of a torch.distributed process group (one process per GPU,
    launched with torchrun): the same methods, every rank passes the same data and obtains the same numbers.

        loss / loss_and_grad -> smnngp_lml_grad_mg_f64  (distributed.DistributedGrad)
        test_nll             -> smnngp_test_nll_mg_f64  (distributed.DistributedPredict)

    x_data / y_data must be torch CUDA tensors on this rank's device.  The solvers are created on first use (they own
    the rank's row shard and the NVLink-visible buffers) and re-used by every later step - the reference evaluates the
    same shapes for 30 000 steps (experiments/regression/train.py:178).  ``solvers=`` injects ready-made ones (tests)."""

    def __init__(self, kernel, likelihood, x_data, y_data, y_mean, y_std, *, eps: float = 1e-6, group=None, block=None,
                 solvers=None):
        super().__init__(kernel, likelihood, x_data, y_data, y_mean, y_std, eps=eps)
        self.group, self.block = group, block
        self._grad_solver = (solvers or {}).get("grad")
        self._predict_solvers = dict((solvers or {}).get("predict", {}))

    def _spec_hp(self):
        kernel_fn = self.kernel.get_kernel_fn()
        if not self._fused(kernel_fn):
            raise TypeError("DistributedSPR needs a kernel_fn built by smnngp nt_kernels and a spax likelihood")
        return kernel_fn.spec, kernel_fn.hp(self.x_data.device, **self._hp_args())

    def loss_and_grad(self):
        from ..distributed import DistributedGrad
        spec, hp = self._spec_hp()
        if self._grad_solver is None:
            self._grad_solver = DistributedGrad(self.num_data, self.x_data.shape[1], spec, self.x_data.device,
                                                group=self.group, block=self.block)
        out, grad, _ = self._grad_solver.lml_grad(self.x_data, self.y_data, hp, kind=self.likelihood.kind)
        g = grad.cpu().numpy()
        slots = {"kernel.w_std": (self.kernel.w_std, 0), "kernel.b_std": (self.kernel.b_std, 1),
                 "kernel.last_w_std": (self.kernel.last_w_std, 2), "eps": (self.eps, 3)}
        if hasattr(self.likelihood, "a"):
            slots["likelihood.a"] = (self.likelihood.a, 4)
            slots["likelihood.b"] = (self.likelihood.b, 5)
        grads = {name: float(g[i]) * float(var.constraint.grad(var.value)) for name, (var, i) in slots.items()}
        return float(out[1]), grads

    def loss(self):
        return self.loss_and_grad()[0]

    def test_nll(self, x, y):
        from ..distributed import DistributedPredict
        spec, hp = self._spec_hp()
        t = int(x.shape[0])
        solver = self._predict_solvers.get(t)
        if solver is None:
            solver = DistributedPredict(self.num_data, self.x_data.shape[1], t, 1, spec, self.x_data.device,
                                        group=self.group, block=self.block)
            self._predict_solvers[t] = solver
        nll, _, _, _ = solver.test_nll(self.x_data, self.y_data, x, y, float(self.y_mean), float(self.y_std), hp,
                                       kind=self.likelihood.kind)
        return nll[0]

    def close(self):
        for s in [self._grad_solver, *self._predict_solvers.values()]:
            if s is not None and hasattr(s, "close"):
                s.close()
        self._grad_solver, self._predict_solvers = None, {}


def _softplus(x):
    return torch.logaddexp(x, torch.zeros_like(x))                                    # bijectors.Softplus on a tensor


def _softplus_inverse(x):
    return torch.where(x < 20.0, torch.log(torch.expm1(torch.clamp(x, max=20.0))), x)


class MultiStartSPR:
    """R copies of an SPR over the same data, trained together: multi-start restarts of the six non-convex scalars.
    ``starts`` [R, 6] holds the safe values {w_std, b_std, last_w_std, eps, alpha, beta} of every restart; the stack
    comes from ``kernel.get_kernel_fn()`` and the kind from the likelihood (their own variables are not used).  The
    unconstrained variables are one device tensor ``raw`` [R, 6] (softplus, spax/bijectors.py), stepped by
    ``BatchAdam``.  Under a Gaussian likelihood alpha and beta are not variables (``mask`` is False there): their
    gradient is 0 and they are never updated."""

    def __init__(self, kernel, likelihood, x_data, y_data, y_mean, y_std, *, starts):
        kernel_fn = kernel.get_kernel_fn()
        if getattr(likelihood, "kind", None) == "burr12":
            raise TypeError("MultiStartSPR: the importance-sampled scale mixture (BurrXIILikelihood) has no gradient")
        if not (isinstance(kernel_fn, KernelFn) and getattr(likelihood, "kind", None) in _dev.KIND):
            raise TypeError("MultiStartSPR needs a kernel_fn built by smnngp nt_kernels and a spax likelihood")
        self.spec, self.kind = kernel_fn.spec, likelihood.kind
        if isinstance(x_data, torch.Tensor):
            dev = x_data.device
        else:
            dev = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        to_dev = lambda a: a.to(dev, torch.float64) if isinstance(a, torch.Tensor) else torch.as_tensor(
            np.ascontiguousarray(a, dtype=np.float64), device=dev)
        self.x_data, self.y_data = to_dev(x_data), to_dev(y_data)
        self.y_mean, self.y_std = float(y_mean), float(y_std)
        self.num_data = self.x_data.shape[0]
        starts = to_dev(starts)
        if starts.ndim != 2 or starts.shape[1] != 6:
            raise ValueError("starts must be [R, 6]")
        self.raw = _softplus_inverse(starts).contiguous()
        self.mask = torch.ones(6, dtype=torch.bool, device=dev)
        if self.kind != "student_t":
            self.mask[4:] = False
        self._batch = None

    def safe_values(self):
        """[R, 6] constrained values {w_std, b_std, last_w_std, eps, alpha, beta}."""
        return _softplus(self.raw)

    def loss_and_grad(self):
        """(loss [R], grad_raw [R, 6], info [R]) in one ``LossGradBatch.points`` call: loss = SPR.loss of every
        restart, grad_raw = d loss / d raw (the softplus chain rule applied on the device, zero where ``mask`` is
        False)."""
        if self._batch is None:
            self._batch = _dev.LossGradBatch(self.x_data, self.y_data, spec=self.spec)
        out, grad, info = self._batch.points(self.safe_values(), self.kind)
        g = torch.where(self.mask, grad * torch.sigmoid(self.raw), torch.zeros_like(grad))
        return out[:, 1], g, info

    def test_nll(self, x, y):
        """[R] SPR.test_nll of every restart.  Where one launch for every restart is faster (``device._batch_wins``,
        never for N > 4096) the bases of (x_data, x) are computed once and ``GridSearch.test_nll`` evaluates all the
        restarts in one smnngp_test_nll_batch_f64 launch; elsewhere one fused call per restart."""
        x = torch.as_tensor(x, dtype=torch.float64, device=self.x_data.device)
        y = torch.as_tensor(y, dtype=torch.float64, device=self.x_data.device)
        hps = self.safe_values()
        if _dev._batch_wins(self.num_data, hps.shape[0]):
            gs = _dev.GridSearch(self.x_data, self.y_data, x, spec=self.spec)
            return gs.test_nll(hps, y, self.y_mean, self.y_std, self.kind)[0]
        rows = [_dev.test_nll(self.x_data, self.y_data, x, y, self.y_mean, self.y_std, spec=self.spec, hp=hps[r],
                              kind=self.kind)[0] for r in range(hps.shape[0])]
        return torch.stack(rows)
