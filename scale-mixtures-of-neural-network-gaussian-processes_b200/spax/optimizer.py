"""Adam on the (host-resident, scalar) unconstrained variables of a spax Module - the role objax.optimizer.Adam plays
in the reference's train step (experiments/regression/train.py:61-67, :151).  The six trainable scalars live on the
host; the device work of a step is the single fused value+gradient call behind ``SPR.loss_and_grad``."""
import math

import numpy as np

__all__ = ["Adam", "BatchAdam"]


class Adam:
    def __init__(self, vc, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8, skip_nan: bool = False):
        """vc: dict name -> TrainVar, as returned by ``Module.vars()`` (possibly filtered).
        skip_nan=True (a deviation from objax, opt-in): a step whose gradient holds a NaN (non-PD kernel matrix) is
        dropped instead of poisoning every variable."""
        self.vars = dict(vc)
        self.beta1, self.beta2, self.eps = beta1, beta2, eps
        self.skip_nan = skip_nan
        self.step = 0
        self.m = {k: np.zeros_like(v.value, dtype=np.float64) for k, v in self.vars.items()}
        self.v = {k: np.zeros_like(v.value, dtype=np.float64) for k, v in self.vars.items()}

    def __call__(self, lr: float, grads):
        """grads: dict name -> d loss / d (unconstrained value) (what ``SPR.loss_and_grad`` returns).  Variables
        without a gradient entry are left untouched.  The update is objax.optimizer.Adam's,
        ``p -= lr_t * m * rsqrt(v + eps)`` - eps sits INSIDE the square root, so a scalar whose gradient is ~1e-8
        (b_std at the reference defaults) moves by ~lr * 1e-4 per step instead of ~lr.  NaN gradients propagate
        into the variables like they do in the reference (the training loop stops on a NaN validation loss,
        regression/train.py:211) unless ``skip_nan`` was requested."""
        if self.skip_nan and any(math.isnan(float(g)) for g in grads.values()):
            return
        self.step += 1
        lr_t = lr * math.sqrt(1.0 - self.beta2 ** self.step) / (1.0 - self.beta1 ** self.step)
        for k, var in self.vars.items():
            if k not in grads:
                continue
            g = np.asarray(grads[k], dtype=np.float64)
            self.m[k] = self.beta1 * self.m[k] + (1.0 - self.beta1) * g
            self.v[k] = self.beta2 * self.v[k] + (1.0 - self.beta2) * g * g
            var.assign(var.value - lr_t * self.m[k] / np.sqrt(self.v[k] + self.eps))


class BatchAdam:
    """``Adam`` on R models at once: the unconstrained variables of every restart are one [R, 6] tensor (``raw``, updated
    in place on its device), and one step applies objax's update elementwise, ``p -= lr_t * m * rsqrt(v + eps)`` with eps
    inside the square root, exactly like ``Adam``.  Rows never mix: a NaN gradient poisons only its own row.
    mask: [6] (or [R, 6]) booleans, False for entries that are not variables (Gaussian likelihood: alpha, beta); those
    are never updated."""

    def __init__(self, raw, mask=None, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8):
        import torch
        self.raw = raw
        self.mask = None if mask is None else torch.as_tensor(mask, dtype=torch.bool, device=raw.device)
        self.beta1, self.beta2, self.eps = beta1, beta2, eps
        self.step = 0
        self.m = torch.zeros_like(raw)
        self.v = torch.zeros_like(raw)

    def __call__(self, lr: float, grad, active=None):
        """grad: [R, 6] d loss / d raw (what ``MultiStartSPR.loss_and_grad`` returns).  active: optional [R] booleans;
        rows that are False (frozen restarts) keep their variables."""
        import torch
        self.step += 1
        lr_t = lr * math.sqrt(1.0 - self.beta2 ** self.step) / (1.0 - self.beta1 ** self.step)
        self.m = self.beta1 * self.m + (1.0 - self.beta1) * grad
        self.v = self.beta2 * self.v + (1.0 - self.beta2) * grad * grad
        new = self.raw - lr_t * self.m / torch.sqrt(self.v + self.eps)
        keep = torch.zeros_like(self.raw, dtype=torch.bool)
        if self.mask is not None:
            keep |= ~self.mask
        if active is not None:
            keep |= ~torch.as_tensor(active, dtype=torch.bool, device=self.raw.device)[:, None]
        self.raw.copy_(torch.where(keep, self.raw, new))
