"""The posterior draw stage (csrc/draws.cu): sample_f_iid against a CPU replica of its Philox stream, draw for draw,
and draw_metrics against the oracle on the same draws.

CPU part: the replica (oracle/draws_ref.py) reproduces Random123's Philox4x32-10 known answers and its Student-t and
Gaussian variates pass KS tests, so it is a reference in its own right and not only a copy of the kernel.
GPU part: per-cell parity over class counts 1 ... 16, one to 300 test points, 1 ... 4000 draws, both variance layouts,
both kinds, shapes on both sides of the boost at a = 1 and seeds whose high word is not zero; exact closed forms at
zero variance; NaN for labels outside [0, C); argument checks of the C-ABI; a stream of a non-current device."""
import ctypes as C

import numpy as np
import pytest
import scipy.stats

from oracle import draws_ref as dr
from oracle import nngp_oracle as orc

EPS = np.finfo(np.float64).eps
SMNNGP_EINVAL = 1                                   # include/smnngp.h
KIND = {"gauss": 0, "student_t": 1}


# ---------------------------------------------------------------------------------------------------------
# CPU: the replica
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ctr,key,expect", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, expect):
    """Random123's known-answer vectors for philox4x32_10"""
    assert " ".join("%08x" % int(w) for w in dr.philox4x32_10(ctr, key)) == expect


def test_seed_key_splits_the_seed():
    assert dr.seed_key(0) == (0, 0)
    assert dr.seed_key(2**32 + 7) == (7, 1)
    assert dr.seed_key(2**64 - 1) == (0xffffffff, 0xffffffff)


def _standardised(kind, a, seed):
    T, C, S = 50, 4, 1000                                   # 2e5 variates over many (s, t, c) counters
    _, e, _ = dr.sample_f_iid(np.zeros((T, C)), np.ones(T), a=a, b=1.0, kind=kind, num_samples=S, seed=seed)
    return e.ravel()


@pytest.mark.parametrize("a", [0.3, 0.5, 0.999, 1.0, 2.5, 40.0])
def test_replica_student_t_is_t_distributed(a):
    """e = normal / sqrt(gamma(a) / a) ~ t_{2a}; a < 1 goes through the boost u^(1/a), a >= 1 does not"""
    e = _standardised("student_t", a, seed=20261021)
    assert e.size >= 200000 and np.isfinite(e).all()
    assert scipy.stats.kstest(e, scipy.stats.t(2 * a).cdf).pvalue > 1e-3


def test_replica_gauss_is_normal():
    e = _standardised("gauss", 1.0, seed=20261021)
    assert e.size >= 200000
    assert scipy.stats.kstest(e, scipy.stats.norm.cdf).pvalue > 1e-3


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


B = 1.5
# (C, T, S, var per class, kind, a, seed): every class count 1 ... 16 in use, S below, at and above one CTA of 256
# threads, var [T] and [C, T], a on both sides of 1, seeds with a zero and a non-zero high word
CASES = [
    (1, 1, 1, False, "gauss", 2.0, 0),
    (1, 37, 4000, True, "student_t", 0.3, 1234),
    (1, 300, 257, True, "student_t", 2.5, 2**64 - 1),
    (3, 300, 255, True, "student_t", 0.5, 2**32 + 7),
    (3, 1, 257, False, "student_t", 1.0, 2**64 - 1),
    (3, 37, 255, False, "student_t", 0.5, 0),
    (3, 300, 4000, True, "gauss", 2.0, 0),
    (10, 37, 4000, False, "student_t", 2.5, 1234),
    (10, 300, 1, True, "gauss", 2.0, 2**64 - 1),
    (10, 1, 255, True, "student_t", 0.3, 2**64 - 1),
    (10, 64, 1000, True, "gauss", 2.0, 1234),          # C T S > 148 * 16 * 256: the grid-stride loop wraps
    (16, 37, 257, True, "student_t", 0.3, 0),
    (16, 300, 255, False, "student_t", 2.5, 2**32 + 7),
    (16, 1, 4000, True, "gauss", 2.0, 2**32 + 7),
    (16, 37, 1, False, "student_t", 1.0, 1234),
    (16, 300, 257, True, "student_t", 1.0, 2**32 + 7),
]
_IDS = ["C%d-T%d-S%d-%s-%s%s-seed%d" % (c, t, s, "varCT" if pc else "varT", k, "" if k == "gauss" else a, sd)
        for c, t, s, pc, k, a, sd in CASES]


def _inputs(case):
    C, T, S, per_class, kind, a, seed = case
    rng = np.random.default_rng(CASES.index(case))
    mean = 2.0 * rng.standard_normal((T, C))
    var = rng.uniform(0.05, 2.0, (C, T) if per_class else T)      # differs per class, so a (c, t) swap shows
    label = rng.integers(0, C, T)
    return mean, var, label


_gpu_draws = {}


def _draws_on_gpu(sm, case):
    """sample_f_iid of a parity case, computed once for the tests that use it"""
    import torch
    if case not in _gpu_draws:
        C, T, S, per_class, kind, a, seed = case
        mean, var, _ = _inputs(case)
        f = sm.device.sample_f_iid(torch.from_numpy(mean).cuda(), torch.from_numpy(var).cuda(),
                                   hp=sm.make_hp(1.0, 0.0, 1.0, 1e-6, a, B), kind=kind, num_samples=S, seed=seed)
        _gpu_draws[case] = f.cpu().numpy()
    return _gpu_draws[case]


def _assert_matches_replica(f, mean, var, *, kind, a, seed, what=""):
    S = f.shape[2]
    f_ref, e_ref, margin = dr.sample_f_iid(mean, var, a=a, b=B, kind=kind, num_samples=S, seed=seed)
    assert f.shape == f_ref.shape and np.isfinite(f).all()
    sigma = np.sqrt((B / a if kind == "student_t" else 1.0) * (var if var.ndim == 2 else var[None, :]))[:, :, None]
    # a few ulp of fp64 libm (log, pow, cospi) between CUDA and NumPy, scaled by the draw
    tol = 1e-12 * sigma * (1.0 + np.abs(e_ref)) + 1e-14 * np.abs(mean.T)[:, :, None]
    near = margin < 1e-10                          # accept decisions within rounding of the threshold
    bad = (np.abs(f - f_ref) > tol) & ~near
    print(f"{what}: {int(near.sum())} of {near.size} cells within 1e-10 of an accept threshold")
    assert not bad.any(), (f"{int(bad.sum())} cells differ, first at {np.argwhere(bad)[0]}: "
                           f"{f[bad][0]!r} vs {f_ref[bad][0]!r}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_IDS)
def test_sample_f_iid_matches_replica(sm, case):
    C, T, S, per_class, kind, a, seed = case
    mean, var, _ = _inputs(case)
    _assert_matches_replica(_draws_on_gpu(sm, case), mean, var, kind=kind, a=a, seed=seed, what=str(case))


@pytest.mark.gpu
def test_seed_high_word_changes_the_draws(sm):
    import torch
    mean, var = np.zeros((37, 3)), np.full(37, 0.5)
    hp = sm.make_hp(1.0, 0.0, 1.0, 1e-6, 0.5, B)
    fs = []
    for seed in (7, 2**32 + 7):
        f = sm.device.sample_f_iid(torch.from_numpy(mean).cuda(), torch.from_numpy(var).cuda(), hp=hp,
                                   kind="student_t", num_samples=300, seed=seed).cpu().numpy()
        _assert_matches_replica(f, mean, var, kind="student_t", a=0.5, seed=seed, what=f"seed {seed}")
        fs.append(f)
    assert not np.any(fs[0] == fs[1])


def _class_scores(f):
    """[C, T]: logsumexp_s log_softmax_c(f) - log S.  Row label[t] holds the per-point terms whose mean is
    orc.test_log_likelihood; argmax over rows is orc.get_correct_count's prediction.  Also returns a bound on how far
    a correct evaluation may differ from these by rounding: 1e-12 relative, plus the few ulp by which a one-ulp
    difference of libm exp / log can move fmax + log(sum exp(f - fmax)) of a sample, weighted by the sample's share
    of the log-sum-exp over samples (this only matters for the heavy tails of t_{2a} at small a)."""
    S = f.shape[2]
    lsm = orc._log_softmax0(f)                                       # [C, T, S]
    lse = orc._logsumexp(lsm, 2)                                     # [C, T]
    w = np.exp(lsm - lse[:, :, None])                                # each sample's share, sums to 1 over s
    fmag = np.abs(f).max(axis=0)                                     # [T, S]
    score = lse - np.log(S)
    bound = 1e-12 * np.maximum(1.0, np.abs(score)) + 4 * EPS * (w * fmag[None]).sum(axis=2)
    return score, bound


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_IDS)
def test_draw_metrics_matches_oracle_on_the_same_draws(sm, case):
    """the fused kernel redraws what sample_f_iid wrote (the draws above are checked against the replica) and
    reduces it; it must agree per point with the oracle evaluated on those draws"""
    import torch
    C, T, S, per_class, kind, a, seed = case
    mean, var, label = _inputs(case)
    f = _draws_on_gpu(sm, case)
    nll, correct, ll, pred = sm.device.draw_metrics(torch.from_numpy(mean).cuda(), torch.from_numpy(var).cuda(),
                                                    label, hp=sm.make_hp(1.0, 0.0, 1.0, 1e-6, a, B), kind=kind,
                                                    num_samples=S, seed=seed)
    ll, pred, nll, correct = ll.cpu().numpy(), pred.cpu().numpy(), float(nll.item()), int(correct.item())
    score, bound = _class_scores(f)
    t = np.arange(T)
    ll_ref, ll_tol = score[label, t], bound[label, t]
    ref_nll = -orc.test_log_likelihood(f, label)
    assert abs(-ll_ref.mean() - ref_nll) <= 1e-14 * max(1.0, abs(ref_nll))    # the helper is the oracle's sum
    err = np.abs(ll - ll_ref)
    assert np.all(err <= ll_tol), (f"ll_per_test off at points {np.flatnonzero(err > ll_tol)}: worst "
                                   f"{err.max():.3e}")
    assert abs(nll - ref_nll) <= 1e-12 * abs(ref_nll) + ll_tol.mean(), (nll, ref_nll)
    # the prediction wherever the top two classes are further apart than rounding
    order = np.argsort(-score, axis=0, kind="stable")
    pred_ref = order[0]
    if C > 1:
        top, second = order[0], order[1]
        clear = score[top, t] - score[second, t] > 1e-12 + bound[top, t] + bound[second, t]
    else:
        clear = np.ones(T, bool)
    assert np.array_equal(pred[clear], pred_ref[clear])
    assert np.all((pred >= 0) & (pred < C))
    ref_correct = orc.get_correct_count(f, label)
    if clear.all():
        assert correct == ref_correct
    else:
        print(f"{int((~clear).sum())} points with a near tie between the top two classes")
        assert abs(correct - ref_correct) <= int((~clear).sum())
    assert correct == int(np.sum(pred == label))


# means that test the log-softmax: exp underflow (gaps > 745), logits of +-700, exact ties (first maximum wins)
_ZERO_VAR_MEANS = np.array([
    [700.0, -700.0, 0.0, 50.0, -50.0],
    [-700.0, -700.0, -700.0, -700.0, -700.0],
    [1.0, 3.0, 3.0, 2.0, 3.0],
    [0.0, 746.0, -1.0, 0.0, 746.0],
    [-700.0, 700.0, 700.0, -700.0, 0.0],
    [0.5, -0.25, 1e-3, 300.0, -300.0],
    [3.0, -3.0, 3.0, 3.0, -746.0],
    [2.0, 1.0, 0.0, -1.0, -2.0],
])
_ZERO_VAR_LABELS = np.array([1, 4, 2, 0, 3, 4, 2, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 5, 257])
@pytest.mark.parametrize("kind,per_class", [("student_t", False), ("gauss", True)])
def test_zero_variance_is_the_log_softmax_of_the_mean(sm, S, kind, per_class):
    """var = 0: every draw is fma(e, 0, mean) = mean, so ll_t = log_softmax(mean_t)[y_t] and pred_t = argmax mean_t"""
    import mpmath
    import torch
    mean, label = _ZERO_VAR_MEANS, _ZERO_VAR_LABELS
    T, C = mean.shape
    var = np.zeros((C, T) if per_class else T)
    md, vd = torch.from_numpy(mean).cuda(), torch.from_numpy(var).cuda()
    hp = sm.make_hp(1.0, 0.0, 1.0, 1e-6, 0.5, B)
    f = sm.device.sample_f_iid(md, vd, hp=hp, kind=kind, num_samples=S, seed=99).cpu().numpy()
    assert np.array_equal(f, np.broadcast_to(mean.T[:, :, None], f.shape))
    nll, correct, ll, pred = sm.device.draw_metrics(md, vd, label, hp=hp, kind=kind, num_samples=S, seed=99)
    ll, pred = ll.cpu().numpy(), pred.cpu().numpy()
    mpmath.mp.dps = 50
    refs, tols = np.empty(T), np.empty(T)
    for t in range(T):
        row = [mpmath.mpf(float(m)) for m in mean[t]]
        refs[t] = float(row[label[t]] - mpmath.log(mpmath.fsum(mpmath.exp(m) for m in row)))
        # roundings of fmax + log(se), f - lse, + log S and - log S, each half an ulp at the size of these values
        tols[t] = 1e-13 + 2 * EPS * (abs(refs[t]) + np.abs(mean[t]).max() + np.log(S))
    assert np.all(np.abs(ll - refs) <= tols), (ll, refs)
    assert np.array_equal(pred, np.argmax(mean, axis=1))
    assert abs(float(nll.item()) + refs.mean()) <= 1e-13 * abs(refs.mean()) + tols.mean()
    assert int(correct.item()) == int(np.sum(np.argmax(mean, axis=1) == label))


@pytest.mark.gpu
def test_out_of_range_label_gives_nan(sm):
    """a label outside [0, C) scores NaN instead of log p = 0, and the other points are unaffected, bit for bit"""
    import torch
    rng = np.random.default_rng(11)
    T, C, S = 37, 10, 300
    mean, var = rng.standard_normal((T, C)), rng.uniform(0.05, 2.0, T)
    label = rng.integers(0, C, T)
    bad_at = np.array([0, 5, 20, 36])
    bad = label.copy()
    bad[bad_at] = [-1, C, -1, C]
    md, vd = torch.from_numpy(mean).cuda(), torch.from_numpy(var).cuda()
    hp = sm.make_hp(1.0, 0.0, 1.0, 1e-6, 0.5, B)
    runs = []
    for lab in (label, bad):
        nll, correct, ll, pred = sm.device.draw_metrics(md, vd, lab, hp=hp, kind="student_t", num_samples=S, seed=5)
        runs.append((float(nll.item()), int(correct.item()), ll.cpu().numpy(), pred.cpu().numpy()))
    (nll0, correct0, ll0, pred0), (nll1, correct1, ll1, pred1) = runs
    assert np.isfinite(nll0) and np.isfinite(ll0).all()
    assert np.isnan(ll1[bad_at]).all() and np.isnan(nll1)
    ok = np.setdiff1d(np.arange(T), bad_at)
    assert np.array_equal(ll1[ok], ll0[ok])
    assert np.array_equal(pred1, pred0)
    assert correct1 == int(np.sum(pred0[ok] == label[ok]))
    assert correct0 == int(np.sum(pred0 == label))


def _ptr(t):
    return C.c_void_p(t.data_ptr())


@pytest.mark.gpu
def test_argument_checks_enqueue_nothing(sm):
    import torch
    lib = sm._lib.load()
    T, Cn, S = 4, 3, 8
    f64, i32 = dict(dtype=torch.float64, device="cuda"), dict(dtype=torch.int32, device="cuda")
    bufs = dict(mean=torch.zeros(T, Cn, **f64), var=torch.ones(T, **f64), label=torch.zeros(T, **i32),
                hp=sm.make_hp(1.0, 0.0, 1.0, 1e-6, 2.0, 2.0), out=torch.empty(Cn * T * S, **f64),
                ll=torch.empty(T, **f64), pred=torch.empty(T, **i32), out2=torch.empty(2, **f64))
    good = {k: _ptr(v) for k, v in bufs.items()}
    good.update(T=T, C=Cn, S=S, kind=KIND["student_t"])
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def sample(**over):
        a = dict(good, **over)
        return lib.smnngp_sample_f_iid_f64(s, a["mean"], a["var"], 0, a["T"], a["C"], a["S"], a["hp"], a["kind"], 3,
                                           a["out"])

    def metrics(**over):
        a = dict(good, **over)
        return lib.smnngp_draw_metrics_f64(s, a["mean"], a["var"], 0, a["label"], a["T"], a["C"], a["S"], a["hp"],
                                           a["kind"], 3, a["ll"], a["pred"], a["out2"])

    common = [dict(T=0), dict(C=0), dict(S=0), dict(T=-1), dict(S=-5), dict(kind=2), dict(kind=-1),
              dict(T=2**31), dict(S=2**31), dict(mean=None), dict(var=None), dict(hp=None)]
    cases = [(sample, "smnngp_sample_f_iid_f64", over) for over in
             common + [dict(C=2**31), dict(C=2**21, T=2**21, S=2**21), dict(out=None)]]
    cases += [(metrics, "smnngp_draw_metrics_f64", over) for over in
              common + [dict(C=17), dict(label=None), dict(ll=None), dict(pred=None), dict(out2=None)]]
    for call, name, over in cases:
        lib.smnngp_lml_host_f64(None, None, 0, 0, 0, 0, 0, None, 0, None, None)     # leaves another call's message
        assert name.encode() not in lib.smnngp_last_error()
        lib.smnngp_instr_reset(0)
        assert call(**over) == SMNNGP_EINVAL, (name, over)
        assert lib.smnngp_instr_launches() == 0, (name, over)
        assert name.encode() in lib.smnngp_last_error(), (name, over, lib.smnngp_last_error())
    lib.smnngp_instr_reset(0)
    assert sample() == 0 and lib.smnngp_instr_launches() == 1
    lib.smnngp_instr_reset(0)
    assert metrics() == 0 and lib.smnngp_instr_launches() == 2
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_stream_of_a_non_current_device(sm):
    """a C-ABI caller whose current device is 0 passes a stream and buffers of cuda:1: both calls launch on cuda:1,
    give the same bits as with cuda:1 current, and leave device 0 current"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    lib = sm._lib.load()
    torch.cuda.set_device(0)
    rng = np.random.default_rng(3)
    T, Cn, S = 37, 10, 500
    d1 = torch.device("cuda:1")
    md = torch.from_numpy(rng.standard_normal((T, Cn))).to(d1)
    vd = torch.from_numpy(rng.uniform(0.05, 2.0, (Cn, T))).to(d1)
    lab = torch.from_numpy(rng.integers(0, Cn, T).astype(np.int32)).to(d1)
    hp = sm.make_hp(1.0, 0.0, 1.0, 1e-6, 0.5, B, device=d1)
    stream = torch.cuda.Stream(device=d1)
    stream.wait_stream(torch.cuda.current_stream(d1))
    results = []
    for current in (0, 1, 0):
        f = torch.empty((Cn, T, S), dtype=torch.float64, device=d1)
        ll = torch.empty(T, dtype=torch.float64, device=d1)
        pred = torch.empty(T, dtype=torch.int32, device=d1)
        out = torch.empty(2, dtype=torch.float64, device=d1)
        stream.wait_stream(torch.cuda.current_stream(d1))
        with torch.cuda.device(current):
            s, kind = C.c_void_p(stream.cuda_stream), KIND["student_t"]
            assert lib.smnngp_sample_f_iid_f64(s, _ptr(md), _ptr(vd), 1, T, Cn, S, _ptr(hp), kind, 77, _ptr(f)) == 0, \
                lib.smnngp_last_error()
            assert lib.smnngp_draw_metrics_f64(s, _ptr(md), _ptr(vd), 1, _ptr(lab), T, Cn, S, _ptr(hp), kind, 77,
                                               _ptr(ll), _ptr(pred), _ptr(out)) == 0, lib.smnngp_last_error()
            assert torch.cuda.current_device() == current
        stream.synchronize()
        results.append([x.cpu().numpy() for x in (f, ll, pred, out)])
    assert torch.cuda.current_device() == 0
    for other in results[1:]:
        for x, y in zip(results[0], other):
            assert np.array_equal(x, y)
    assert np.isfinite(results[0][3]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("prior", ["student_t", "gauss"])
@pytest.mark.parametrize("layout", ["CBB", "BB", "CB", "B"])
def test_prior_sample_f_iid_reads_the_diagonal(sm, prior, layout):
    """InverseGammaPrior / GaussianPrior.sample_f_iid take a covariance or its diagonal, per class or shared"""
    import torch
    from smnngp_b200.spax import InverseGammaPrior, GaussianPrior
    rng = np.random.default_rng(17)
    Cn, Bn, S, a = 3, 7, 64, 0.5
    mean = rng.standard_normal((Cn, Bn))
    var = rng.uniform(0.1, 2.0, (Cn, Bn) if layout in ("CBB", "CB") else Bn)
    if layout in ("CBB", "BB"):
        g = rng.standard_normal(var.shape + (Bn,))
        cov = g @ np.swapaxes(g, -1, -2)
        idx = np.arange(Bn)
        cov[..., idx, idx] = var
    else:
        cov = var
    md = torch.from_numpy(mean).cuda()
    p = InverseGammaPrior(a, B) if prior == "student_t" else GaussianPrior()
    got = p.sample_f_iid(2**40 + 3, md, torch.from_numpy(cov).cuda(), S).cpu().numpy()
    want = sm.device.sample_f_iid(md.T.contiguous(), torch.from_numpy(var).cuda(), hp=p._hp(md.device), kind=prior,
                                  num_samples=S, seed=2**40 + 3).cpu().numpy()
    assert got.shape == (Cn, Bn, S)
    assert np.array_equal(got, want)
