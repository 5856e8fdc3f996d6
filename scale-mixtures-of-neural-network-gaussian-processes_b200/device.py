"""Device-level ops: thin, allocation-aware wrappers over the C-ABI (include/smnngp.h).

PyTorch is used for device memory and streams only.  Inputs may be torch CUDA tensors (device entry points,
enqueue-only on the current stream) or NumPy arrays (host entry points: copies included, synchronous).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib

ACT = {"relu": 0, "erf": 1}
ARCH = {"mlp": 0, "resnet": 1}
KIND = {"gauss": 0, "student_t": 1}
SHIFT = {"none": 0, "eps_abs": 1, "eps_rel": 2, "lik": 3}


@dataclass(frozen=True)
class StackSpec:
    """The layer stack of experiments/nt_kernels.py:21-31 (mlp) / :83-103 (resnet)."""
    num_hiddens: int
    act: str = "relu"
    arch: str = "mlp"

    def ids(self):
        if self.act not in ACT:
            raise KeyError("Unsupported act '{}'".format(self.act))      # nt_kernels.py:18
        if self.arch not in ARCH:
            raise ValueError(f"Unsupported network '{self.arch}'")       # regression/train.py:124
        return int(self.num_hiddens), ACT[self.act], ARCH[self.arch]


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("smnngp: no CUDA device - this path has no CPU fallback")


_ws_cache: dict = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Cached scratch buffer per (device, stream): calls enqueued on different streams never share (and so never
    corrupt) a workspace, and a buffer that has to grow is released to torch's caching allocator, which only hands it
    out again in the order of the stream it was allocated on (the stream the earlier call was enqueued on)."""
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    key = (idx, torch.cuda.current_stream(idx).cuda_stream)
    cur = _ws_cache.get(key)
    if cur is None or cur.numel() < nbytes:
        _ws_cache[key] = None
        cur = torch.empty(int(nbytes), dtype=torch.uint8, device=torch.device("cuda", idx))
        _ws_cache[key] = cur
    return cur


def release_workspaces():
    _ws_cache.clear()
    _lib.load().smnngp_host_release()


def _on_device_of_first_arg(fn):
    """Run ``fn`` with the first tensor argument's device current.  The library resolves the device from the stream
    it is handed, but torch's default stream is the legacy stream (handle 0), which belongs to whatever device is
    current - so the Python layer pins the device as well."""
    import functools

    @functools.wraps(fn)
    def wrapped(x, *a, **k):
        if isinstance(x, torch.Tensor) and x.is_cuda:
            with torch.cuda.device(x.device):
                return fn(x, *a, **k)
        return fn(x, *a, **k)
    return wrapped


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f64(x, device=None):
    t = torch.as_tensor(x, dtype=torch.float64, device=device) if not isinstance(x, torch.Tensor) else x
    if t.dtype != torch.float64:
        t = t.to(torch.float64)
    return t.contiguous()


def make_hp(w_std, b_std, last_w_std, eps=1e-6, alpha=2.0, beta=2.0, device="cuda"):
    """Device operand {w_std, b_std, last_w_std, eps, alpha, beta} (safe values)."""
    vals = [float(v) for v in (w_std, b_std, last_w_std, eps, alpha, beta)]
    return torch.tensor(vals, dtype=torch.float64, device=device)


def _np_hp(w_std, b_std, last_w_std, eps=1e-6, alpha=2.0, beta=2.0):
    return np.ascontiguousarray([w_std, b_std, last_w_std, eps, alpha, beta], dtype=np.float64)


# ---------------------------------------------------------------------------------------------------------
@_on_device_of_first_arg
def gram(x, x2=None, *, spec: StackSpec, hp, shift="none", lower_only=False, out=None):
    """K = kernel_fn(x, x2, get="nngp") (spax/kernels.py:23-27).  Device tensors in, device tensor out."""
    _require_cuda()
    lib = _lib.load()
    nh, act, arch = spec.ids()
    x = _f64(x)
    sym = x2 is None or x2 is x
    x2t = None if sym else _f64(x2, x.device)
    n, d = x.shape
    m = n if sym else x2t.shape[0]
    if not sym and x2t.shape[1] != d:
        raise ValueError("feature dimensions differ")
    if out is None:
        out = torch.empty((n, m), dtype=torch.float64, device=x.device)
        if lower_only:
            out.zero_()
    ws_bytes = lib.smnngp_gram_workspace_bytes(n, m, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    rc = lib.smnngp_gram_f64(_stream(x.device), _p(x), _p(x2t), n, m, d, nh, act, arch, _p(hp), SHIFT[shift],
                             1 if lower_only else 0, _p(out), out.stride(0), _p(ws), ws_bytes)
    _lib.check(rc, "gram")
    return out


@_on_device_of_first_arg
def nngp_diag(x, *, spec: StackSpec, hp):
    _require_cuda()
    lib = _lib.load()
    nh, act, arch = spec.ids()
    x = _f64(x)
    n, d = x.shape
    q = torch.empty(n, dtype=torch.float64, device=x.device)
    ws_bytes = lib.smnngp_gram_workspace_bytes(n, n, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    _lib.check(lib.smnngp_nngp_diag_f64(_stream(x.device), _p(x), n, d, nh, act, arch, _p(hp), _p(q), _p(ws),
                                        ws_bytes), "nngp_diag")
    return q


@_on_device_of_first_arg
def potrf_(a: torch.Tensor, n_cols=None):
    """In-place lower Cholesky of the leading n_cols x n_cols of the row-major a [M, >=n_cols]; extra rows become
    rows * L^-T.  Returns (sum log L_ii [device scalar], info [device int])."""
    _require_cuda()
    lib = _lib.load()
    assert a.dtype == torch.float64 and a.is_cuda and a.stride(1) == 1
    m = a.shape[0]
    n = a.shape[1] if n_cols is None else n_cols
    info = torch.zeros(1, dtype=torch.int32, device=a.device)
    logdet = torch.zeros(1, dtype=torch.float64, device=a.device)
    ws_bytes = lib.smnngp_potrf_workspace_bytes(max(m, n))       # rows: sizes the panel buffer of the fused solve
    ws = _workspace(ws_bytes, a.device)
    rc = lib.smnngp_potrf_trapezoid_f64(_stream(a.device), _p(a), m, n, a.stride(0), _p(logdet), _p(info), _p(ws),
                                        ws_bytes)
    _lib.check(rc, "potrf")
    return logdet, info


@_on_device_of_first_arg
def cov_solve(cov, y, *, scale=1.0, shift=0.0):
    """(sum log L_ii, ||L^-1 y||^2, info) for L = chol(scale * cov + shift I); cov is left untouched."""
    _require_cuda()
    lib = _lib.load()
    cov = _f64(cov)
    y = _f64(y, cov.device)
    n = cov.shape[0]
    out = torch.empty(2, dtype=torch.float64, device=cov.device)
    info = torch.zeros(1, dtype=torch.int32, device=cov.device)
    ws_bytes = lib.smnngp_cov_solve_workspace_bytes(n)
    ws = _workspace(ws_bytes, cov.device)
    rc = lib.smnngp_cov_solve_f64(_stream(cov.device), _p(cov), n, cov.stride(0), _p(y), float(scale), float(shift),
                                  _p(ws), ws_bytes, _p(out), _p(info))
    _lib.check(rc, "cov_solve")
    return out[0], out[1], info


@_on_device_of_first_arg
def lml(x, y, *, spec: StackSpec, hp, kind="student_t"):
    """Fused SPR.loss pieces (spax/models.py:93-98).  Device inputs -> (out[4] device tensor, info);
    NumPy inputs -> host entry point, returns (np.ndarray[4], int).
    out = [log p(y), -log p(y)/N, sum log L_ii, ||L^-1 y||^2]."""
    lib = _lib.load()
    nh, act, arch = spec.ids()
    if isinstance(x, np.ndarray):
        _require_cuda()
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        hp = np.ascontiguousarray(hp, dtype=np.float64)
        out = np.empty(4, dtype=np.float64)
        info = C.c_int(0)
        rc = lib.smnngp_lml_host_f64(x.ctypes.data, y.ctypes.data, x.shape[0], x.shape[1], nh, act, arch,
                                     hp.ctypes.data, KIND[kind], out.ctypes.data, C.byref(info))
        _lib.check(rc, "lml_host")
        return out, info.value
    _require_cuda()
    x = _f64(x)
    y = _f64(y, x.device)
    n, d = x.shape
    out = torch.empty(4, dtype=torch.float64, device=x.device)
    info = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws_bytes = lib.smnngp_lml_workspace_bytes(n, d, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    rc = lib.smnngp_lml_f64(_stream(x.device), _p(x), _p(y), n, d, nh, act, arch, _p(hp), KIND[kind], _p(ws),
                            ws_bytes, _p(out), _p(info))
    _lib.check(rc, "lml")
    return out, info


@_on_device_of_first_arg
def lml_grad(x, y, *, spec: StackSpec, hp, kind="student_t"):
    """SPR.loss and d loss / d {w_std, b_std, last_w_std, eps, alpha, beta} in one call - the value/gradient pair
    objax.GradValues(model.loss, vars) produces in regression/train.py:62-66 (before the softplus chain rule).
    Device inputs -> (out[4], grad[6], info) device tensors; NumPy inputs -> host entry point."""
    lib = _lib.load()
    nh, act, arch = spec.ids()
    if isinstance(x, np.ndarray):
        _require_cuda()
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        hp = np.ascontiguousarray(hp, dtype=np.float64)
        out = np.empty(4, dtype=np.float64)
        grad = np.empty(6, dtype=np.float64)
        info = C.c_int(0)
        rc = lib.smnngp_lml_grad_host_f64(x.ctypes.data, y.ctypes.data, x.shape[0], x.shape[1], nh, act, arch,
                                          hp.ctypes.data, KIND[kind], out.ctypes.data, grad.ctypes.data,
                                          C.byref(info))
        _lib.check(rc, "lml_grad_host")
        return out, grad, info.value
    _require_cuda()
    x = _f64(x)
    y = _f64(y, x.device)
    n, d = x.shape
    out = torch.empty(4, dtype=torch.float64, device=x.device)
    grad = torch.empty(6, dtype=torch.float64, device=x.device)
    info = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws_bytes = lib.smnngp_lml_grad_workspace_bytes(n, d, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    rc = lib.smnngp_lml_grad_f64(_stream(x.device), _p(x), _p(y), n, d, nh, act, arch, _p(hp), KIND[kind], _p(ws),
                                 ws_bytes, _p(out), _p(grad), _p(info))
    _lib.check(rc, "lml_grad")
    return out, grad, info


class LmlGraph:
    """The fused LML call captured once into a CUDA graph and replayed - the analogue of wrapping SPR.loss in
    objax.Jit (regression/train.py:61-67): the training loop evaluates the same shapes tens of thousands of
    times, and for N <~ 20k the ~1700 dependent small launches of the factorisation are launch-latency bound.
    Inputs are copied into static buffers; hyper-parameters stay a device operand, so they may change between
    replays without re-capturing."""

    def __init__(self, n, d, *, spec: StackSpec, kind="student_t", device="cuda"):
        _require_cuda()
        self.lib = _lib.load()
        self.spec, self.kind = spec, kind
        nh, act, arch = spec.ids()
        dev = torch.device(device)
        self.x = torch.zeros((n, d), dtype=torch.float64, device=dev)
        self.y = torch.zeros(n, dtype=torch.float64, device=dev)
        self.hp = torch.ones(6, dtype=torch.float64, device=dev)
        self.out = torch.zeros(4, dtype=torch.float64, device=dev)
        self.info = torch.zeros(1, dtype=torch.int32, device=dev)
        self.ws_bytes = self.lib.smnngp_lml_workspace_bytes(n, d, nh, arch)
        self.ws = torch.empty(int(self.ws_bytes), dtype=torch.uint8, device=dev)
        self.graph = None

    def _enqueue(self):
        nh, act, arch = self.spec.ids()
        n, d = self.x.shape
        rc = self.lib.smnngp_lml_f64(_stream(self.x.device), _p(self.x), _p(self.y), n, d, nh, act, arch, _p(self.hp),
                                     KIND[self.kind], _p(self.ws), self.ws_bytes, _p(self.out), _p(self.info))
        _lib.check(rc, "lml (graph)")

    def __call__(self, x, y, hp):
        with torch.cuda.device(self.x.device):
            return self._call(x, y, hp)

    def _call(self, x, y, hp):
        self.x.copy_(x, non_blocking=True)
        self.y.copy_(y, non_blocking=True)
        self.hp.copy_(hp, non_blocking=True)
        if self.graph is None:
            s = torch.cuda.Stream(device=self.x.device)
            s.wait_stream(torch.cuda.current_stream(self.x.device))
            with torch.cuda.stream(s):
                self._enqueue()                       # warm-up: function attributes, lazy module loading
            torch.cuda.current_stream(self.x.device).wait_stream(s)
            torch.cuda.synchronize(self.x.device)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._enqueue()
        self.graph.replay()
        return self.out, self.info


@_on_device_of_first_arg
def predict(x, y, x_test, *, spec: StackSpec, hp, shift="eps_rel", full_cov=False):
    """NNGPKernel.predict (spax/kernels.py:29-32): returns (mean [T,C], var [T] = diag(cov), info); with
    full_cov=True (device inputs) the second element is the full [T,T] posterior covariance."""
    lib = _lib.load()
    nh, act, arch = spec.ids()
    if isinstance(x, np.ndarray):
        _require_cuda()
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if y.ndim == 1:
            y = y[:, None]
        xt = np.ascontiguousarray(x_test, dtype=np.float64)
        hp = np.ascontiguousarray(hp, dtype=np.float64)
        n, d = x.shape
        t, c = xt.shape[0], y.shape[1]
        mean = np.empty((t, c), dtype=np.float64)
        var = np.empty(t, dtype=np.float64)
        info = C.c_int(0)
        rc = lib.smnngp_predict_host_f64(x.ctypes.data, y.ctypes.data, xt.ctypes.data, n, t, c, d, nh, act, arch,
                                         hp.ctypes.data, SHIFT[shift], mean.ctypes.data, var.ctypes.data,
                                         C.byref(info))
        _lib.check(rc, "predict_host")
        return mean, var, info.value
    _require_cuda()
    x = _f64(x)
    y = _f64(y, x.device)
    if y.ndim == 1:
        y = y[:, None].contiguous()
    xt = _f64(x_test, x.device)
    n, d = x.shape
    t, c = xt.shape[0], y.shape[1]
    mean = torch.empty((t, c), dtype=torch.float64, device=x.device)
    var = torch.empty(t, dtype=torch.float64, device=x.device)
    info = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws_bytes = lib.smnngp_predict_workspace_bytes(n, t, c, d, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    if full_cov:
        cov = torch.empty((t, t), dtype=torch.float64, device=x.device)
        rc = lib.smnngp_predict_cov_f64(_stream(x.device), _p(x), _p(y), _p(xt), n, t, c, d, nh, act, arch, _p(hp),
                                        SHIFT[shift], _p(ws), ws_bytes, _p(mean), _p(var), _p(cov), cov.stride(0),
                                        _p(info))
        _lib.check(rc, "predict_cov")
        return mean, cov, info
    rc = lib.smnngp_predict_f64(_stream(x.device), _p(x), _p(y), _p(xt), n, t, c, d, nh, act, arch, _p(hp),
                                SHIFT[shift], _p(ws), ws_bytes, _p(mean), _p(var), _p(info))
    _lib.check(rc, "predict")
    return mean, var, info


@_on_device_of_first_arg
def test_nll(x, y, x_test, y_test, y_mean, y_std, *, spec: StackSpec, hp, kind="student_t"):
    """Fused SPR.test_nll (spax/models.py:100-120).  Returns (nll, mean [T], var [T], info)."""
    lib = _lib.load()
    nh, act, arch = spec.ids()
    if isinstance(x, np.ndarray):
        _require_cuda()
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        xt = np.ascontiguousarray(x_test, dtype=np.float64)
        yt = np.ascontiguousarray(y_test, dtype=np.float64)
        hp = np.ascontiguousarray(hp, dtype=np.float64)
        n, d = x.shape
        t = xt.shape[0]
        nll = np.empty(1, dtype=np.float64)
        mean = np.empty(t, dtype=np.float64)
        var = np.empty(t, dtype=np.float64)
        info = C.c_int(0)
        rc = lib.smnngp_test_nll_host_f64(x.ctypes.data, y.ctypes.data, xt.ctypes.data, yt.ctypes.data, n, t, d, nh,
                                          act, arch, hp.ctypes.data, KIND[kind], float(y_mean), float(y_std),
                                          nll.ctypes.data, mean.ctypes.data, var.ctypes.data, C.byref(info))
        _lib.check(rc, "test_nll_host")
        return float(nll[0]), mean, var, info.value
    _require_cuda()
    x = _f64(x)
    y = _f64(y, x.device)
    xt = _f64(x_test, x.device)
    yt = _f64(y_test, x.device)
    n, d = x.shape
    t = xt.shape[0]
    nll = torch.empty(1, dtype=torch.float64, device=x.device)
    mean = torch.empty(t, dtype=torch.float64, device=x.device)
    var = torch.empty(t, dtype=torch.float64, device=x.device)
    info = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws_bytes = lib.smnngp_predict_workspace_bytes(n, t, 1, d, nh, arch)
    ws = _workspace(ws_bytes, x.device)
    rc = lib.smnngp_test_nll_f64(_stream(x.device), _p(x), _p(y), _p(xt), _p(yt), n, t, d, nh, act, arch, _p(hp),
                                 KIND[kind], float(y_mean), float(y_std), _p(ws), ws_bytes, _p(nll), _p(mean),
                                 _p(var), C.c_void_p(0), _p(info))
    _lib.check(rc, "test_nll")
    return nll[0], mean, var, info


@_on_device_of_first_arg
def grid_point(x, y, x_test, *, spec: StackSpec, hp):
    """The device work of ONE point (w_std, b_std, eps) of the reference's grid search
    (experiments/regression/find.py:134-160): the predictive with the RELATIVE regulariser (``predict(eps)``,
    find.py:75-77) and, for the absolute one, ``log det(K + eps I)`` and ``y^T (K + eps I)^-1 y``
    (find.py:149-156, there through an explicit inverse and ``multivariate_normal.logpdf``).  The (alpha, beta)
    importance-sampling table that follows (find.py:163-186) is host arithmetic on these outputs.
    Returns (mean [T], var [T], logdet, quad, info) with logdet = log det(K + eps I)."""
    mean, var, info1 = predict(x, y, x_test, spec=spec, hp=hp, shift="eps_rel")
    out, info2 = lml(x, y, spec=spec, hp=hp, kind="gauss")
    if isinstance(x, np.ndarray):
        return mean[:, 0], var, 2.0 * float(out[2]), float(out[3]), max(int(info1), int(info2))
    return mean[:, 0], var, 2.0 * out[2], out[3], torch.maximum(info1, info2)


GRID_BATCH_MAX_N = 4096


def _batch_wins(n, g):
    """Whether ``GridSearch.points`` evaluates G points of N training rows in one batched launch rather than one
    point after the other.  Up to the resident slots the batch costs what one CTA needs for one point; that is
    3.2, 8.9, 38 and 130 times a ``point`` call at N = 404, 824, 2048 and 4096 (profiles/r03_grid_batch.jsonl, B200 at
    1000 W), ~3.2 (N / 404)^1.6.  Past the slots the batch runs in waves of at least 148 points, which still beats the
    loop wherever one wave does.  ``GridSearch.test_nll`` uses the same rule: a batched test-NLL point costs about a
    batched grid point (the same two factorisations) and a ``test_nll`` call about a ``point`` call
    (profiles/nll_batch_bench.py times both paths)."""
    return n <= GRID_BATCH_MAX_N and g >= 3.2 * (n / 404.0) ** 1.6


class GridSearch:
    """The reference's hyper-parameter grid search (experiments/regression/find.py:134-199) with the base Gram cached:
    X.X^T / D, Xt.X^T / D and the input variances are computed once; every ``point(hp)`` is recursion-only passes over
    the cached bases plus the two factorisations - the same outputs as ``grid_point`` without touching X again."""

    def __init__(self, x, y, x_test, *, spec: StackSpec):
        _require_cuda()
        self.lib = _lib.load()
        self.spec = spec
        x = _f64(x)
        self.y = _f64(y, x.device)
        xt = _f64(x_test, x.device)
        self.x, self.x_test = x, xt                  # for the per-point test_nll loop
        self.n, d = x.shape
        self.t = xt.shape[0]
        dev = x.device
        self.ld0 = (self.n + 15) // 16 * 16
        self.k0dd = torch.empty((self.n, self.ld0), dtype=torch.float64, device=dev)
        self.k0td = torch.empty((self.t, self.ld0), dtype=torch.float64, device=dev)
        self.q_d = torch.empty(self.n, dtype=torch.float64, device=dev)
        self.q_t = torch.empty(self.t, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = self.lib.smnngp_grid_base_f64(_stream(dev), _p(x), _p(xt), self.n, self.t, d, _p(self.k0dd), self.ld0,
                                               _p(self.k0td), self.ld0, _p(self.q_d), _p(self.q_t))
        _lib.check(rc, "grid_base")

    def point(self, hp):
        """(mean [T], var [T], logdet, quad, info) for the scalars in ``hp`` (device operand, see make_hp)."""
        nh, act, arch = self.spec.ids()
        dev = self.y.device
        mean = torch.empty(self.t, dtype=torch.float64, device=dev)
        var = torch.empty(self.t, dtype=torch.float64, device=dev)
        out = torch.empty(2, dtype=torch.float64, device=dev)
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        ws_bytes = self.lib.smnngp_grid_workspace_bytes(self.n, self.t, nh, arch)
        with torch.cuda.device(dev):
            ws = _workspace(ws_bytes, dev)
            rc = self.lib.smnngp_grid_point_f64(_stream(dev), _p(self.k0dd), self.ld0, _p(self.k0td), self.ld0,
                                                _p(self.q_d), _p(self.q_t), _p(self.y), self.n, self.t, nh, act, arch,
                                                _p(hp), _p(ws), ws_bytes, _p(mean), _p(var), _p(out), _p(info))
        _lib.check(rc, "grid_point")
        return mean, var, 2.0 * out[0], out[1], info

    def points(self, hps):
        """Every row of ``hps`` [G, 6] (device operand rows, e.g. ``torch.stack`` of make_hp) at once:
        (mean [G, T], var [G, T], logdet [G], quad [G], info [G]), row g what ``point(hps[g])`` returns.  Where one
        launch for the whole grid is faster (``_batch_wins``) a CTA evaluates each point in its own workspace slot
        (smnngp_grid_batch_f64); elsewhere, and always for N > 4096, the points run one after the other."""
        dev = self.y.device
        hps = _f64(hps, dev)
        if hps.ndim != 2 or hps.shape[1] != 6:
            raise ValueError("hps must be [G, 6]")
        g = hps.shape[0]
        if not _batch_wins(self.n, g):
            rows = [self.point(hps[i]) for i in range(g)]
            return tuple(torch.stack([r[k] for r in rows]) for k in range(4)) + (torch.cat([r[4] for r in rows]),)
        nh, act, arch = self.spec.ids()
        mean = torch.empty((g, self.t), dtype=torch.float64, device=dev)
        var = torch.empty((g, self.t), dtype=torch.float64, device=dev)
        out = torch.empty((g, 2), dtype=torch.float64, device=dev)
        info = torch.empty(g, dtype=torch.int32, device=dev)
        # every slot a CTA the device keeps resident (grid_batch_kernel: two per SM); more would only wait
        slots = min(g, 2 * torch.cuda.get_device_properties(dev).multi_processor_count)
        ws_bytes = self.lib.smnngp_grid_batch_workspace_bytes(self.n, self.t, nh, arch, slots)
        with torch.cuda.device(dev):
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            rc = self.lib.smnngp_grid_batch_f64(_stream(dev), _p(self.k0dd), self.ld0, _p(self.k0td), self.ld0,
                                                _p(self.q_d), _p(self.q_t), _p(self.y), self.n, self.t, g, nh, act,
                                                arch, _p(hps), _p(ws), ws_bytes, _p(mean), _p(var), _p(out), _p(info))
        _lib.check(rc, "grid_batch")
        return mean, var, 2.0 * out[:, 0], out[:, 1], info

    def test_nll(self, hps, y_test, y_mean, y_std, kind="student_t"):
        """``SPR.test_nll`` on the test rows at every row of ``hps`` [G, 6] (device operand rows, see make_hp):
        (nll [G], mean [G, T], var [G, T], info [G]), row g what ``test_nll(x, y, x_test, y_test, y_mean, y_std,
        hp=hps[g], kind=kind)`` returns, up to rounding.  ``y_test`` [T] holds the standardised test targets.  Where
        one launch for every point is faster (``_batch_wins``) a CTA evaluates each point in its own workspace slot
        (smnngp_test_nll_batch_f64); elsewhere, and always for N > 4096, the points run one ``test_nll`` call after
        the other."""
        dev = self.y.device
        hps = _f64(hps, dev)
        if hps.ndim != 2 or hps.shape[1] != 6:
            raise ValueError("hps must be [G, 6]")
        if kind not in KIND:
            raise ValueError(f"unknown likelihood kind '{kind}'")
        yt = _f64(y_test, dev)
        if tuple(yt.shape) != (self.t,):
            raise ValueError(f"y_test must be [{self.t}]")
        g = hps.shape[0]
        if not _batch_wins(self.n, g):
            rows = [test_nll(self.x, self.y, self.x_test, yt, y_mean, y_std, spec=self.spec, hp=hps[i], kind=kind)
                    for i in range(g)]
            return tuple(torch.stack([r[k] for r in rows]) for k in range(3)) + (torch.cat([r[3] for r in rows]),)
        nh, act, arch = self.spec.ids()
        nll = torch.empty(g, dtype=torch.float64, device=dev)
        mean = torch.empty((g, self.t), dtype=torch.float64, device=dev)
        var = torch.empty((g, self.t), dtype=torch.float64, device=dev)
        info = torch.empty(g, dtype=torch.int32, device=dev)
        # every slot a CTA the device keeps resident (test_nll_batch_kernel: two per SM), as far as half the free
        # memory holds them; more slots would only wait
        one = self.lib.smnngp_test_nll_batch_workspace_bytes(self.n, self.t, nh, arch, 1)
        with torch.cuda.device(dev):
            free = torch.cuda.mem_get_info(dev)[0]
        slots = max(1, min(g, 2 * torch.cuda.get_device_properties(dev).multi_processor_count, free // 2 // one))
        ws_bytes = slots * one
        with torch.cuda.device(dev):
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            rc = self.lib.smnngp_test_nll_batch_f64(_stream(dev), _p(self.k0dd), self.ld0, _p(self.k0td), self.ld0,
                                                    _p(self.q_d), _p(self.q_t), _p(self.y), _p(yt), self.n, self.t, g,
                                                    nh, act, arch, _p(hps), KIND[kind], float(y_mean), float(y_std),
                                                    _p(ws), ws_bytes, _p(nll), _p(mean), _p(var), C.c_void_p(0),
                                                    _p(info))
        _lib.check(rc, "test_nll_batch")
        return nll, mean, var, info


    def sweep_eps(self, eps_list, hp, group=None):
        """find.py:141 `for eps in eps_list`: every regulariser of the sweep for the scalars in ``hp`` (its eps entry is
        replaced), one epsilon per GPU when a process group is up (replica parallelism, see distributed.sweep_eps)."""
        from .distributed import sweep_eps

        def evaluate(eps):
            h = hp.clone()
            h[3] = eps
            return self.point(h)

        return sweep_eps(eps_list, evaluate, t=self.t, device=self.y.device, group=group)


def _grad_batch_wins(n, g):
    """Whether ``LossGradBatch.points`` evaluates G points of N training rows in one batched launch rather than one
    ``lml_grad`` call after the other.  Provisional: the form of ``_batch_wins`` (a CTA-point costs ~(N / 404)^1.6
    per-call evaluations), with a lower constant because one ``lml_grad`` call is ~2x a ``grid_point`` call at N = 404.
    ``profiles/grad_batch_bench.py`` times both paths at N = 404 .. 4096 and G = 1 .. 1100 to re-derive it."""
    return n <= GRID_BATCH_MAX_N and g >= 2.0 * (n / 404.0) ** 1.6


class LossGradBatch:
    """``SPR.loss`` and its six-scalar gradient at many hyper-parameter points over the same data - multi-start
    training, or gradient refinement of the best points of a grid search.  X.X^T / D and the input variances are cached
    once (smnngp_grid_base_f64 with no test rows); ``points(hps, kind)`` evaluates every row of ``hps``."""

    def __init__(self, x, y, *, spec: StackSpec):
        _require_cuda()
        self.lib = _lib.load()
        self.spec = spec
        self.x = _f64(x)
        self.y = _f64(y, self.x.device)
        self.n, d = self.x.shape
        dev = self.x.device
        self.ld0 = (self.n + 15) // 16 * 16
        self.k0dd = torch.empty((self.n, self.ld0), dtype=torch.float64, device=dev)
        self.q_d = torch.empty(self.n, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = self.lib.smnngp_grid_base_f64(_stream(dev), _p(self.x), None, self.n, 0, d, _p(self.k0dd), self.ld0,
                                               None, 0, _p(self.q_d), None)
        _lib.check(rc, "grid_base")

    def points(self, hps, kind="student_t"):
        """(out [G, 4], grad [G, 6], info [G]) for the rows of ``hps`` [G, 6] (device operand rows, see make_hp): row g
        is what ``lml_grad(x, y, hp=hps[g], kind=kind)`` returns, up to rounding.  Where one launch for every point is
        faster (``_grad_batch_wins``) a CTA evaluates each point in its own workspace slot (smnngp_lml_grad_batch_f64);
        elsewhere, and always for N > 4096, the points run one ``lml_grad`` call after the other."""
        dev = self.x.device
        hps = _f64(hps, dev)
        if hps.ndim != 2 or hps.shape[1] != 6:
            raise ValueError("hps must be [G, 6]")
        if kind not in KIND:
            raise ValueError(f"unknown likelihood kind '{kind}'")
        g = hps.shape[0]
        if not _grad_batch_wins(self.n, g):
            rows = [lml_grad(self.x, self.y, spec=self.spec, hp=hps[i], kind=kind) for i in range(g)]
            return (torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows]),
                    torch.cat([r[2] for r in rows]))
        nh, act, arch = self.spec.ids()
        out = torch.empty((g, 4), dtype=torch.float64, device=dev)
        grad = torch.empty((g, 6), dtype=torch.float64, device=dev)
        info = torch.empty(g, dtype=torch.int32, device=dev)
        # every slot a CTA the device keeps resident (lml_grad_batch_kernel: two per SM), as far as half the free
        # memory holds them (a slot is ~268 MB at N = 4096); more slots would only wait
        one = self.lib.smnngp_lml_grad_batch_workspace_bytes(self.n, nh, arch, 1)
        with torch.cuda.device(dev):
            free = torch.cuda.mem_get_info(dev)[0]
        slots = max(1, min(g, 2 * torch.cuda.get_device_properties(dev).multi_processor_count, free // 2 // one))
        ws_bytes = slots * one
        with torch.cuda.device(dev):
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            rc = self.lib.smnngp_lml_grad_batch_f64(_stream(dev), _p(self.k0dd), self.ld0, _p(self.q_d), _p(self.y),
                                                    self.n, g, nh, act, arch, _p(hps), KIND[kind], _p(ws), ws_bytes,
                                                    _p(out), _p(grad), _p(info))
        _lib.check(rc, "lml_grad_batch")
        return out, grad, info


def set_panel_width(nb: int):
    _lib.load().smnngp_set_panel_width(int(nb))


# ---------------------------------------------------------------------------------------------------------
# posterior draw stage (classification / ensemble configuration)
@_on_device_of_first_arg
def sample_f_iid(mean, var, *, hp, kind="student_t", num_samples, seed=0):
    """Prior.sample_f_iid (spax/priors.py:30-36, :60-68).  mean [T, C] (NNGPKernel.predict layout), var [T] or
    [C, T]  ->  draws [C, T, S]."""
    _require_cuda()
    lib = _lib.load()
    mean = _f64(mean)
    var = _f64(var, mean.device)
    t, c = mean.shape
    out = torch.empty((c, t, int(num_samples)), dtype=torch.float64, device=mean.device)
    rc = lib.smnngp_sample_f_iid_f64(_stream(mean.device), _p(mean), _p(var), 1 if var.ndim == 2 else 0, t, c,
                                     int(num_samples), _p(hp), KIND[kind], int(seed), _p(out))
    _lib.check(rc, "sample_f_iid")
    return out


@_on_device_of_first_arg
def draw_metrics(mean, var, label, *, hp, kind="student_t", num_samples, seed=0):
    """Fused draw -> test_log_likelihood / get_correct_count (spax/utils.py:61-74) without materialising the
    [C, T, S] draws.  Returns (nll, correct_count, ll_per_test [T], pred [T])."""
    _require_cuda()
    lib = _lib.load()
    mean = _f64(mean)
    var = _f64(var, mean.device)
    label = torch.as_tensor(label, device=mean.device).to(torch.int32).contiguous()
    t, c = mean.shape
    ll = torch.empty(t, dtype=torch.float64, device=mean.device)
    pred = torch.empty(t, dtype=torch.int32, device=mean.device)
    out = torch.empty(2, dtype=torch.float64, device=mean.device)
    rc = lib.smnngp_draw_metrics_f64(_stream(mean.device), _p(mean), _p(var), 1 if var.ndim == 2 else 0, _p(label), t,
                                     c, int(num_samples), _p(hp), KIND[kind], int(seed), _p(ll), _p(pred), _p(out))
    _lib.check(rc, "draw_metrics")
    return out[0], out[1], ll, pred
