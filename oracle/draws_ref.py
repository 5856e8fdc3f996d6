"""CPU replica of the posterior draw stage's generator (``csrc/draws.cu``), NumPy only, FP64.

TEST INFRASTRUCTURE ONLY, like ``nngp_oracle``.  The CUDA draw stage draws from a counter-based stream, so every
draw f[c, t, s] is a pure function of (seed, s, t, c) and can be recomputed here cell by cell:

* Philox4x32-10 (Salmon et al., SC'11; Random123), key (seed & 0xffffffff, seed >> 32), counter (s, t, c, n) where
  n counts the Philox calls of the cell;
* u01(hi, lo) in (0, 1] from 53 bits, two uniforms per call: (x, y) first, then (z, w);
* Box-Muller, cos branch: sqrt(-2 log u1) cospi(2 u2);
* Marsaglia & Tsang (2000) gamma(alpha): for alpha < 1 the boost u^(1/alpha) is drawn first and alpha += 1; at most
  64 trials, after which the draw is boost * d;
* Student-t with df = 2a: normal / sqrt(gamma(a) / a), the normal drawn first;
* f = e * sqrt(scale * var) + mean, scale = b / a (Student-t) or 1 (Gauss).

The rejection loop takes a different number of uniforms in every cell, so each cell keeps its own Philox counter
and two-uniform buffer, and the loop runs over the cells that are still rejecting.  The uint32 multiplies of Philox
are exact as uint64 products.  The libm of NumPy and CUDA differ by a few ulp, so the replica matches the kernel to
rounding, not bit for bit; for each cell it also returns the smallest |margin| of the decisions the gamma loop took
(v > 0 and log u < 1/2 x^2 + d - d v + d log v), so that a comparison can set aside a cell whose decision rounding
could flip.
"""
from __future__ import annotations

import numpy as np

__all__ = ["philox4x32_10", "seed_key", "u01", "cospi", "sample_f_iid"]

_M32 = np.uint64(0xFFFFFFFF)
_MUL0, _MUL1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_WEYL0, _WEYL1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(ctr, key):
    """Philox4x32-10 of the counter words ``ctr = (c0, c1, c2, c3)`` (ints or arrays) under ``key = (k0, k1)``.
    Returns the four output words as uint64 arrays holding uint32 values."""
    c0, c1, c2, c3 = (np.asarray(w, dtype=np.uint64) for w in ctr)
    a, b = (np.uint64(k) for k in key)
    for _ in range(10):
        p0 = _MUL0 * c0
        p1 = _MUL1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ a, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ b, p0 & _M32
        a = (a + _WEYL0) & _M32
        b = (b + _WEYL1) & _M32
    return c0, c1, c2, c3


def seed_key(seed):
    """Philox key of a 64-bit seed: (low word, high word)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & 0xFFFFFFFF, seed >> 32


def u01(hi, lo):
    """Uniform in (0, 1] from the 53 bits (hi << 21) ^ (lo >> 11)."""
    v = (np.asarray(hi, dtype=np.uint64) << np.uint64(21)) ^ (np.asarray(lo, dtype=np.uint64) >> np.uint64(11))
    return ((v & np.uint64((1 << 53) - 1)).astype(np.float64) + 1.0) * (1.0 / 9007199254740992.0)


def cospi(x):
    """cos(pi x) for x in [0, 2] with an exact argument reduction, so that it keeps its relative accuracy near the
    zeros at 1/2 and 3/2 the way CUDA's cospi does (np.cos(np.pi * x) is off there by ~1e-16 absolute, and the
    Student-t divides that normal by sqrt(gamma / a), which can be far below 1)."""
    x = np.asarray(x, dtype=np.float64)
    r = np.abs(x - 2.0 * np.round(0.5 * x))              # exact, in [0, 1]
    return np.where(r <= 0.25, np.cos(np.pi * r),
                    np.where(r <= 0.75, np.sin(np.pi * (0.5 - r)), -np.cos(np.pi * (1.0 - r))))


class _Cells:
    """The uniform streams of many cells at once; every method takes the indices of the cells that draw."""

    def __init__(self, seed, s, t, c):
        self.key = seed_key(seed)
        self.s, self.t, self.c = (np.asarray(x, dtype=np.uint64) for x in (s, t, c))
        self.n = np.zeros(self.s.shape, np.uint64)
        self.buf = np.zeros((4,) + self.s.shape, np.uint64)
        self.have = np.zeros(self.s.shape, np.int8)

    def uniform(self, idx):
        empty = idx[self.have[idx] == 0]
        if empty.size:
            words = philox4x32_10((self.s[empty], self.t[empty], self.c[empty], self.n[empty]), self.key)
            for k in range(4):
                self.buf[k, empty] = words[k]
            self.n[empty] += np.uint64(1)
            self.have[empty] = 2
        h = self.have[idx]
        first = h == 2
        hi = np.where(first, self.buf[0, idx], self.buf[2, idx])
        lo = np.where(first, self.buf[1, idx], self.buf[3, idx])
        self.have[idx] = h - 1
        return u01(hi, lo)

    def normal(self, idx):
        u1 = self.uniform(idx)
        u2 = self.uniform(idx)
        return np.sqrt(-2.0 * np.log(u1)) * cospi(2.0 * u2)

    def gamma(self, alpha, idx):
        """Marsaglia-Tsang gamma(alpha) of the cells idx; returns (draws, smallest |margin| of each cell)."""
        boost = np.ones(idx.size)
        if alpha < 1.0:
            boost = self.uniform(idx) ** (1.0 / alpha)
            alpha += 1.0
        d = alpha - 1.0 / 3.0
        cc = 1.0 / np.sqrt(9.0 * d)
        out = boost * d                                  # what a cell that rejects 64 times returns
        margin = np.full(idx.size, np.inf)
        rejecting = np.ones(idx.size, bool)
        for _ in range(64):
            live = np.flatnonzero(rejecting)
            if live.size == 0:
                break
            x = self.normal(idx[live])
            v = 1.0 + cc * x
            margin[live] = np.minimum(margin[live], np.abs(v))
            pos = v > 0.0
            live, x, v = live[pos], x[pos], v[pos]
            v = v * v * v
            u = self.uniform(idx[live])
            m = np.log(u) - (0.5 * x * x + d - d * v + d * np.log(v))
            margin[live] = np.minimum(margin[live], np.abs(m))
            acc = m < 0.0
            out[live[acc]] = boost[live[acc]] * d * v[acc]
            rejecting[live[acc]] = False
        return out, margin


def sample_f_iid(mean, var, *, a, b, kind, num_samples, seed):
    """The draws of ``smnngp_sample_f_iid_f64``: mean [T, C], var [T] or [C, T], kind "student_t" or "gauss".

    Returns (f, e, margin), each [C, T, S]: the draws, the standardised variates e (f = e * sigma + mean) and the
    smallest |margin| of each cell's gamma decisions (inf for Gaussian draws, which take none)."""
    mean = np.asarray(mean, dtype=np.float64)
    var = np.asarray(var, dtype=np.float64)
    T, C = mean.shape
    S = int(num_samples)
    i = np.arange(C * T * S, dtype=np.int64)
    s, t, c = i % S, (i // S) % T, i // (S * T)
    cells = _Cells(seed, s, t, c)
    idx = np.arange(i.size)
    if kind == "student_t":
        df = 2.0 * a
        z = cells.normal(idx)
        g, margin = cells.gamma(0.5 * df, idx)
        e = z / np.sqrt(g / (0.5 * df))
        scale = b / a
    elif kind == "gauss":
        e = cells.normal(idx)
        margin = np.full(i.size, np.inf)
        scale = 1.0
    else:
        raise ValueError(f"unknown kind {kind!r}")
    v = var[c, t] if var.ndim == 2 else var[t]
    f = e * np.sqrt(scale * v) + mean[t, c]
    shape = (C, T, S)
    return f.reshape(shape), e.reshape(shape), margin.reshape(shape)
