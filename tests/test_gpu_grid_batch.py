"""Batched grid search (smnngp_grid_batch_f64 / GridSearch.points): every point of a whole (w_std, b_std, eps) grid in
one launch.  Parity with the oracle and with the per-point call, bit-exact independence of a point from the rest of its
batch, failure isolation, argument checks, a launch count that does not grow with the problem, graph capture, and the
per-point fallback above N = 4096."""
import ctypes as C

import numpy as np
import pytest

from oracle import nngp_oracle as orc
from tests.synth import regression_data, DEFAULT_HP

LML_TOL = 1e-8
POINT_TOL = 1e-9        # batched vs per-point factorisation: same matrix, different blocking and summation order

EINVAL, EWORKSPACE = 1, 3


@pytest.fixture(scope="module")
def sm():
    import torch
    import smnngp_b200 as s
    assert torch.cuda.is_available()
    s._lib.load()
    return s


def _data(n, t, d):
    import torch
    x, y, xt, *_ = regression_data(n, d, t=t)
    return (x, y, xt), tuple(torch.from_numpy(v).cuda() for v in (x, y, xt))


def _grid(sm, ws, bs, es):
    """[G, 6] device rows in (w, b, eps) order and the matching host dicts."""
    import torch
    hps, rows = [], []
    for w in ws:
        for b in bs:
            for e in es:
                hp = dict(DEFAULT_HP, w_std=w, b_std=b, eps=e)
                rows.append(hp)
                hps.append(sm.make_hp(hp["w_std"], hp["b_std"], hp["last_w_std"], hp["eps"], hp["alpha"], hp["beta"]))
    return torch.stack(hps), rows


def _random_grid(sm, g, seed=5):
    import torch
    rng = np.random.default_rng(seed)
    w = rng.uniform(0.5, 2.0, g)
    b = rng.uniform(0.01, 1.0, g)
    e = 10.0 ** rng.uniform(-4, -2, g)
    return torch.stack([sm.make_hp(w[i], b[i], 1.0, e[i]) for i in range(g)])


def _host(res):
    return tuple(r.cpu().numpy() for r in res)


def _cabi(sm, gs, hps, slots):
    """smnngp_grid_batch_f64 with a workspace of exactly `slots` slots."""
    import torch
    lib = sm._lib.load()
    nh, act, arch = gs.spec.ids()
    g, t, dev = hps.shape[0], gs.t, gs.y.device
    mean = torch.empty((g, t), dtype=torch.float64, device=dev)
    var = torch.empty((g, t), dtype=torch.float64, device=dev)
    out = torch.empty((g, 2), dtype=torch.float64, device=dev)
    info = torch.empty(g, dtype=torch.int32, device=dev)
    nbytes = lib.smnngp_grid_batch_workspace_bytes(gs.n, t, nh, arch, slots)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    rc = lib.smnngp_grid_batch_f64(C.c_void_p(torch.cuda.current_stream().cuda_stream), gs.k0dd.data_ptr(), gs.ld0,
                                   gs.k0td.data_ptr(), gs.ld0, gs.q_d.data_ptr(), gs.q_t.data_ptr(), gs.y.data_ptr(),
                                   gs.n, t, g, nh, act, arch, hps.data_ptr(), ws.data_ptr(), nbytes, mean.data_ptr(),
                                   var.data_ptr(), out.data_ptr(), info.data_ptr())
    assert rc == 0, lib.smnngp_last_error()
    return _host((mean, var, 2.0 * out[:, 0], out[:, 1], info))


def _same_bits(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def _rows(res, idx):
    return tuple(r[idx] for r in res)


# ---- parity -------------------------------------------------------------------------------------------------------
SHAPES = [(404, 52, 13, "relu", "mlp", 3), (900, 130, 8, "erf", "mlp", 2), (1500, 257, 16, "relu", "resnet", 2),
          (1, 4, 5, "relu", "mlp", 3), (17, 9, 4, "erf", "resnet", 1), (300, 1, 7, "relu", "mlp", 2),
          (250, 40, 6, "relu", "mlp", 0), (4096, 512, 8, "relu", "mlp", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,t,d,act,arch,L", SHAPES)
def test_points_match_oracle_and_point(sm, n, t, d, act, arch, L):
    """A 3 x 3 x 3 (w_std, b_std, eps) grid, eps 1e-4 .. 1e-2, against the oracle at the project's tolerances (three
    points at N = 4096, where the oracle needs seconds per point) and every point against GridSearch.point."""
    (x, y, xt), (xd, yd, xtd) = _data(n, t, d)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(L, act, arch))
    hps, rows = _grid(sm, (0.6, 1.0, 1.7), (0.05, 0.3, 0.9), (1e-4, 1e-3, 1e-2))
    mean, var, logdet, quad, info = _cabi(sm, gs, hps, 27)        # the batched kernel, whatever points() would pick
    assert mean.shape == (27, t) and var.shape == (27, t) and logdet.shape == (27,) and info.shape == (27,)
    assert np.all(info == 0)
    check = range(27) if n < 4096 else (0, 13, 26)
    for i in check:
        hp = rows[i]
        kw = dict(num_hiddens=L, act=act, w_std=hp["w_std"], b_std=hp["b_std"], last_w_std=hp["last_w_std"], arch=arch)
        m_ref, v_ref, ld_ref, q_ref = orc.find_grid_point(x, y, xt, hp["eps"], kernel_kwargs=kw)
        ktt = orc.nngp_diag(xt, **kw)
        assert np.abs(mean[i] - m_ref).max() <= LML_TOL * np.abs(m_ref).max(), f"point {i}: mean"
        assert np.all(np.abs(var[i] - v_ref) <= LML_TOL * np.abs(v_ref) + 1e-13 * ktt), f"point {i}: var"
        assert abs(logdet[i] - ld_ref) <= LML_TOL * abs(ld_ref), f"point {i}: logdet"
        assert abs(quad[i] - q_ref) <= LML_TOL * abs(q_ref), f"point {i}: quad"
    worst = 0.0
    for i in range(27):
        m1, v1, ld1, q1, i1 = _host(gs.point(hps[i]))
        assert int(i1[0]) == 0
        scale = max(np.abs(m1).max(), 1e-300)
        errs = (np.abs(mean[i] - m1).max() / scale, np.abs(var[i] - v1).max() / np.abs(v1).max(),
                abs(logdet[i] - ld1) / abs(ld1), abs(quad[i] - q1) / abs(q1))
        worst = max(worst, *errs)
    assert worst <= POINT_TOL, f"batched vs per-point: worst relative difference {worst:.3e}"
    print(f"\n[grid_batch] N={n} T={t} {act}/{arch}/L={L}: worst relative difference vs GridSearch.point {worst:.3e}")


# ---- independence and reproducibility ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_point_outputs_do_not_depend_on_the_batch(sm):
    import torch
    _, (xd, yd, xtd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    hps = _random_grid(sm, 500)
    ref = _host(gs.points(hps))
    assert np.all(ref[4] == 0)
    assert _same_bits(ref, _host(gs.points(hps))), "two calls"
    for i in (0, 1, 36, 250, 499):
        assert _same_bits(_rows(ref, slice(i, i + 1)), _cabi(sm, gs, hps[i:i + 1], 1)), f"point {i} alone"
    assert _same_bits(_rows(ref, slice(0, 37)), _host(gs.points(hps[:37]))), "batch of 37"
    perm = torch.from_numpy(np.random.default_rng(1).permutation(500)).cuda()
    got = _host(gs.points(hps[perm]))
    inv = torch.argsort(perm).cpu().numpy()
    assert _same_bits(ref, _rows(got, inv)), "permuted batch"
    for slots in (1, 7):
        assert _same_bits(_rows(ref, slice(0, 37)), _cabi(sm, gs, hps[:37].contiguous(), slots)), f"{slots} slots"
    assert _same_bits(ref, _cabi(sm, gs, hps, 500)), "one slot per point"


@pytest.mark.gpu
def test_failed_points_are_nan_and_isolated(sm):
    """eps = -2 makes both regularised matrices indefinite: info as GridSearch.point reports it, all-NaN outputs, and
    the good neighbours are the same bits as in a batch without the failed points."""
    import torch
    _, (xd, yd, xtd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    good = _random_grid(sm, 40, seed=9)
    bad_at = [0, 3, 4, 17, 41, 43]
    rows, k = [], 0
    for i in range(good.shape[0] + len(bad_at)):
        if i in bad_at:
            h = good[k % 40].clone()
            h[3] = -2.0
            rows.append(h)
        else:
            rows.append(good[k])
            k += 1
    mixed = torch.stack(rows)
    got = _host(gs.points(mixed))
    ref = _host(gs.points(good))
    ok = [i for i in range(mixed.shape[0]) if i not in bad_at]
    assert _same_bits(_rows(got, ok), ref)
    for i in bad_at:
        _, _, _, _, info1 = gs.point(mixed[i])
        assert int(got[4][i]) == int(info1.item()) != 0
        assert np.all(np.isnan(got[0][i])) and np.all(np.isnan(got[1][i]))
        assert np.isnan(got[2][i]) and np.isnan(got[3][i])


# ---- C-ABI ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_arguments_are_rejected_before_anything_is_enqueued(sm):
    import torch
    lib = sm._lib.load()
    _, (xd, yd, xtd) = _data(64, 8, 5)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(2, "relu", "mlp"))
    hps = _random_grid(sm, 4)
    out = torch.empty(4 * 8 * 2 + 8, dtype=torch.float64, device="cuda")
    info = torch.empty(4, dtype=torch.int32, device="cuda")
    nbytes = lib.smnngp_grid_batch_workspace_bytes(64, 8, 2, 0, 2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: t.data_ptr()
    good = dict(K0dd=p(gs.k0dd), ld0=gs.ld0, K0td=p(gs.k0td), ld0t=gs.ld0, q_d=p(gs.q_d), q_t=p(gs.q_t), y=p(gs.y),
                N=64, T=8, G=4, nh=2, act=0, arch=0, hp=p(hps), ws=p(ws), nbytes=nbytes, mean=p(out),
                var=p(out) + 8 * 32, out=p(out) + 8 * 64, info=p(info))

    def call(**over):
        a = dict(good, **over)
        return lib.smnngp_grid_batch_f64(s, a["K0dd"], a["ld0"], a["K0td"], a["ld0t"], a["q_d"], a["q_t"], a["y"],
                                         a["N"], a["T"], a["G"], a["nh"], a["act"], a["arch"], a["hp"], a["ws"],
                                         a["nbytes"], a["mean"], a["var"], a["out"], a["info"])

    cases = [(EWORKSPACE, dict(nbytes=nbytes // 2 - 1)), (EWORKSPACE, dict(nbytes=0)), (EWORKSPACE, dict(ws=None)),
             (EINVAL, dict(N=4097, ld0=4100, ld0t=4100)), (EINVAL, dict(T=0)), (EINVAL, dict(G=0)),
             (EINVAL, dict(ld0=63)), (EINVAL, dict(ld0t=63)), (EINVAL, dict(nh=65)), (EINVAL, dict(nh=-1)),
             (EINVAL, dict(act=2)), (EINVAL, dict(arch=2)), (EINVAL, dict(N=0))]
    cases += [(EINVAL, {k: None}) for k in ("K0dd", "K0td", "q_d", "q_t", "y", "hp", "mean", "var", "out", "info")]
    for code, over in cases:
        lib.smnngp_instr_reset(0)
        assert call(**over) == code, over
        assert lib.smnngp_instr_launches() == 0, over
    lib.smnngp_instr_reset(0)
    assert call() == 0 and lib.smnngp_instr_launches() == 1


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_problem(sm):
    import torch
    lib = sm._lib.load()
    counts = []
    for n, g in ((17, 1), (404, 37), (2000, 500)):
        _, (xd, yd, xtd) = _data(n, 12, 6)
        gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
        hps = _random_grid(sm, g)
        torch.cuda.synchronize()
        lib.smnngp_instr_reset(0)
        _, _, _, _, info = _cabi(sm, gs, hps, min(g, 296))
        counts.append(lib.smnngp_instr_launches())
        assert np.all(info == 0)
    assert counts == [1, 1, 1]


@pytest.mark.gpu
def test_graph_capture_replays_with_new_scalars(sm):
    import torch
    _, (xd, yd, xtd) = _data(404, 52, 13)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(3, "relu", "mlp"))
    hps = _random_grid(sm, 37, seed=2).clone()
    gs.points(hps)                                     # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = gs.points(hps)
    for seed in (3, 4):
        new = _random_grid(sm, 37, seed=seed)
        hps.copy_(new)
        graph.replay()
        torch.cuda.synchronize()
        assert _same_bits(_host(res), _host(gs.points(new)))


@pytest.mark.gpu
@pytest.mark.parametrize("n,g", [(4100, 3), (2048, 11)])
def test_points_fall_back_to_point(sm, n, g):
    """Above N = 4096, and where the measured crossover says the loop is faster, points() is the loop over point()."""
    assert not sm.device._batch_wins(n, g)
    _, (xd, yd, xtd) = _data(n, 8, 6)
    gs = sm.device.GridSearch(xd, yd, xtd, spec=sm.StackSpec(2, "relu", "mlp"))
    hps = _random_grid(sm, g)
    got = _host(gs.points(hps))
    for i in range(g):
        one = _host(gs.point(hps[i]))
        assert _same_bits(_rows(got, slice(i, i + 1)), (one[0][None], one[1][None], one[2][None], one[3][None], one[4]))


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,t,nh,arch", [(404, 52, 3, 0), (1, 1, 0, 0), (4096, 512, 2, 1), (17, 300, 64, 0)])
def test_grid_batch_workspace_is_affine_in_slots(n, t, nh, arch):
    import smnngp_b200 as s
    lib = s._lib.load()
    one = lib.smnngp_grid_batch_workspace_bytes(n, t, nh, arch, 1)
    assert one >= (n + t + 1) * n * 8
    for slots in (2, 7, 296):
        assert lib.smnngp_grid_batch_workspace_bytes(n, t, nh, arch, slots) == slots * one
