"""Debiased Sinkhorn divergence (``sinkhorn_divergence``, ``loss_.batch_EMD_loss``, ``psd_sinkhorn_divergence``).

The expected values come from two fp64 restatements of geomloss 0.2.x ``SamplesLoss("sinkhorn", p=2, blur, scaling,
debias=True)`` (tensorized backend, uniform weights), evaluated per cloud pair: ``ref_numpy`` (dense matrices, rows in blocks of
2048, the gradient from the extrapolation step's softmax weights) and ``ref_torch`` (geomloss's no_grad / .detach() structure, so
that autograd defines the gradient).  The CPU tests check the two against each other and against exact optimal transport; the
GPU tests check the kernel against ``ref_torch`` run in fp64 on the device, each quantity within a few times the error of an
fp32 emulation of the kernel on the same pair (test_sinkhorn_fp32.py)."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment
from scipy.special import logsumexp

from conftest import make_clouds

KINDS = ("uniform", "clustered", "lattice", "dup", "offset")


# ---------------------------------------------------------------------------------------------------------------- references
def f32(v):
    return float(np.float32(v))


def diameter(x, y):
    """sqrt(sum over axes of (max - min)^2) over both clouds, in fp64 from the fp32 extents."""
    pts = np.concatenate([x.reshape(-1, 3), y.reshape(-1, 3)]).astype(np.float64)
    return float(np.sqrt(((pts.max(0) - pts.min(0)) ** 2).sum()))


def eps_schedule(D, blur, scaling):
    """geomloss's epsilon list for p = 2, in double: [D^2] + exp(arange(2 ln D, 2 ln blur, 2 ln scaling)) + [blur^2]
    (blur and scaling as the fp32 values the kernel receives)."""
    blur, scaling = f32(blur), f32(scaling)
    return [D ** 2] + [float(np.exp(e)) for e in np.arange(2 * np.log(D), 2 * np.log(blur), 2 * np.log(scaling))] + [blur ** 2]


def log_w(k):
    return float(np.log(np.float32(1.0) / np.float32(k)))     # logf(1/k) in fp32


def _softmin_np(eps, X, Y, h, grad=False, rows=2048):
    out = np.empty(len(X))
    trans = np.empty((len(X), 3)) if grad else None
    for r0 in range(0, len(X), rows):
        xb = X[r0:r0 + rows]
        C = 0.5 * ((xb[:, None, :] - Y[None, :, :]) ** 2).sum(-1)
        z = h[None, :] - C / eps
        lse = logsumexp(z, axis=1)
        out[r0:r0 + rows] = -eps * lse
        if grad:
            P = np.exp(z - lse[:, None])
            trans[r0:r0 + rows] = xb - P @ Y            # sum_j P_ij (x_i - y_j)
    return (out, trans) if grad else out


def ref_numpy(x, y, blur=0.05, scaling=0.5):
    """One cloud pair (x [n, 3], y [m, 3] fp32) in fp64: (S, (f_ba, f_aa, g_ab, g_bb), grad_x, grad_y, rounds)."""
    X, Y = x.astype(np.float64), y.astype(np.float64)
    n, m = len(X), len(Y)
    if not (np.isfinite(X).all() and np.isfinite(Y).all()):
        nan = float("nan")
        return nan, tuple(np.full(k, nan) for k in (n, n, m, m)), np.full((n, 3), nan), np.full((m, 3), nan), 0
    D = diameter(x, y)
    if D == 0.0:
        return 0.0, tuple(np.zeros(k) for k in (n, n, m, m)), np.zeros((n, 3)), np.zeros((m, 3)), 0
    E = [f32(e) for e in eps_schedule(D, blur, scaling)]
    la, lb = log_w(n), log_w(m)
    za, zb = np.full(n, la), np.full(m, lb)
    e = E[0]
    g_ab, f_ba = _softmin_np(e, Y, X, za), _softmin_np(e, X, Y, zb)
    f_aa, g_bb = _softmin_np(e, X, X, za), _softmin_np(e, Y, Y, zb)
    for e in E:
        ft_ba, gt_ab = _softmin_np(e, X, Y, lb + g_ab / e), _softmin_np(e, Y, X, la + f_ba / e)
        ft_aa, gt_bb = _softmin_np(e, X, X, la + f_aa / e), _softmin_np(e, Y, Y, lb + g_bb / e)
        f_ba, g_ab, f_aa, g_bb = 0.5 * (f_ba + ft_ba), 0.5 * (g_ab + gt_ab), 0.5 * (f_aa + ft_aa), 0.5 * (g_bb + gt_bb)
    e = E[-1]
    (f_ba2, Pxy), (g_ab2, Pyx) = _softmin_np(e, X, Y, lb + g_ab / e, True), _softmin_np(e, Y, X, la + f_ba / e, True)
    (f_aa2, Qxx), (g_bb2, Qyy) = _softmin_np(e, X, X, la + f_aa / e, True), _softmin_np(e, Y, Y, lb + g_bb / e, True)
    S = (f_ba2 - f_aa2).mean() + (g_ab2 - g_bb2).mean()
    return float(S), (f_ba2, f_aa2, g_ab2, g_bb2), (Pxy - Qxx) / n, (Pyx - Qyy) / m, len(E)


def ref_torch(x, y, blur=0.05, scaling=0.5):
    """The same pair with torch fp64 (on x's device) and geomloss's structure: the cost matrices detach their second
    argument, the loop runs without autograd, the extrapolation step's inputs are detached; autograd gives the gradient."""
    x = x.detach().double().requires_grad_(True)
    y = y.detach().double().requires_grad_(True)
    n, m = x.shape[0], y.shape[0]
    if not (torch.isfinite(x).all() and torch.isfinite(y).all()):
        nan = float("nan")
        full = lambda *s: torch.full(s, nan, dtype=torch.float64, device=x.device)
        return nan, (full(n), full(n), full(m), full(m)), full(n, 3), full(m, 3), 0
    D = diameter(x.detach().float().cpu().numpy(), y.detach().float().cpu().numpy())
    if D == 0.0:
        z = lambda *s: torch.zeros(s, dtype=torch.float64, device=x.device)
        return 0.0, (z(n), z(n), z(m), z(m)), z(n, 3), z(m, 3), 0
    E = [f32(e) for e in eps_schedule(D, blur, scaling)]
    la, lb = log_w(n), log_w(m)
    cost = lambda u, v: 0.5 * ((u[:, None, :] - v[None, :, :]) ** 2).sum(-1)
    C_xx, C_yy, C_xy, C_yx = cost(x, x.detach()), cost(y, y.detach()), cost(x, y.detach()), cost(y, x.detach())
    sm = lambda eps, C, h: -eps * torch.logsumexp(h[None, :] - C / eps, dim=1)
    za, zb = torch.full((n,), la, dtype=torch.float64, device=x.device), torch.full((m,), lb, dtype=torch.float64, device=x.device)
    with torch.no_grad():
        e = E[0]
        g_ab, f_ba, f_aa, g_bb = sm(e, C_yx, za), sm(e, C_xy, zb), sm(e, C_xx, za), sm(e, C_yy, zb)
        for e in E:
            ft_ba, gt_ab = sm(e, C_xy, lb + g_ab / e), sm(e, C_yx, la + f_ba / e)
            ft_aa, gt_bb = sm(e, C_xx, la + f_aa / e), sm(e, C_yy, lb + g_bb / e)
            f_ba, g_ab, f_aa, g_bb = 0.5 * (f_ba + ft_ba), 0.5 * (g_ab + gt_ab), 0.5 * (f_aa + ft_aa), 0.5 * (g_bb + gt_bb)
    e = E[-1]
    f_ba, g_ab = sm(e, C_xy, (lb + g_ab / e).detach()), sm(e, C_yx, (la + f_ba / e).detach())
    f_aa, g_bb = sm(e, C_xx, (la + f_aa / e).detach()), sm(e, C_yy, (lb + g_bb / e).detach())
    S = (f_ba - f_aa).mean() + (g_ab - g_bb).mean()
    gx, gy = torch.autograd.grad(S, [x, y])
    return float(S.detach()), tuple(t.detach() for t in (f_ba, f_aa, g_ab, g_bb)), gx, gy, len(E)


# ---------------------------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("n,m,kind", [(37, 53, "uniform"), (64, 20, "clustered"), (9, 9, "lattice"), (40, 31, "offset")])
def test_numpy_and_torch_references_agree(n, m, kind):
    x, y = make_clouds(kind, 1, n, m, seed=n + m)
    S1, p1, gx1, gy1, k1 = ref_numpy(x[0], y[0])
    S2, p2, gx2, gy2, k2 = ref_torch(torch.from_numpy(x[0]), torch.from_numpy(y[0]))
    assert k1 == k2 >= 2
    assert math.isclose(S1, S2, rel_tol=1e-9, abs_tol=1e-12)
    for a, b in zip(p1, p2):
        np.testing.assert_allclose(a, b.numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(gx1, gx2.numpy(), rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(gy1, gy2.numpy(), rtol=1e-8, atol=1e-12)


def test_schedule_length_follows_numpy_arange():
    def expected(D, blur, scaling):
        v = math.ceil((2 * math.log(f32(blur)) - 2 * math.log(D)) / (2 * math.log(f32(scaling))))
        return 2 + max(0, v)
    for D, blur, scaling in ((math.sqrt(3), 0.05, 0.5), (1.0, 0.01, 0.9), (0.03, 0.05, 0.5), (f32(0.05), 0.05, 0.5),
                             (1e-7, 0.05, 0.5), (250.0, 0.05, 0.5), (1.0, 0.002, 0.98)):
        E = eps_schedule(D, blur, scaling)
        assert len(E) == expected(D, blur, scaling)
        assert E[0] == D ** 2 and E[-1] == f32(blur) ** 2
    assert len(eps_schedule(math.sqrt(3), 0.05, 0.5)) == 8
    assert len(eps_schedule(0.03, 0.05, 0.5)) == 2           # 0 < D <= blur: [D^2, blur^2]


def test_reference_is_zero_on_identical_clouds():
    x, _ = make_clouds("uniform", 1, 200, 1, seed=11)
    S, pots, gx, gy, _ = ref_numpy(x[0], x[0])
    assert abs(S) < 1e-12
    assert np.abs(gx).max() < 1e-12 and np.abs(gy).max() < 1e-12


def test_small_blur_approaches_exact_optimal_transport():
    """At blur 0.002 / scaling 0.98 the debiased divergence is within 1 % of the exact OT cost mean 1/2 |x_i - y_s(i)|^2."""
    x, y = make_clouds("uniform", 1, 256, 256, seed=21)
    X, Y = x[0].astype(np.float64), y[0].astype(np.float64)
    C = 0.5 * ((X[:, None, :] - Y[None, :, :]) ** 2).sum(-1)
    r, c = linear_sum_assignment(C)
    W = C[r, c].mean()
    S = ref_numpy(x[0], y[0], blur=0.002, scaling=0.98)[0]
    assert abs(S - W) <= 0.01 * W, (S, W)
    S_default = ref_numpy(x[0], y[0])[0]
    assert S_default < 0.9 * W          # the default blur is far from the EMD


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
vp = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())


def run(lib, x, y, blur=0.05, scaling=0.5, cluster=0, grads=True, stream=None):
    """psd_sinkhorn_divergence(_cluster) on device tensors: (loss, grad_x, grad_y, potentials, rounds)."""
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    dev = x.device
    loss = torch.full((b,), -1.0, device=dev)
    gx = torch.full((b, n, 3), -1.0, device=dev) if grads else None
    gy = torch.full((b, m, 3), -1.0, device=dev) if grads else None
    pot = torch.full((b, 2 * n + 2 * m), -1.0, device=dev)
    rounds = torch.full((b,), -7, dtype=torch.int32, device=dev)
    st = ctypes.c_void_p(stream.cuda_stream) if stream is not None else None
    if cluster:
        rc = lib.psd_sinkhorn_divergence_cluster(vp(x), vp(y), b, n, m, blur, scaling, vp(loss), vp(gx), vp(gy), vp(pot),
                                                 vp(rounds), cluster, st)
    else:
        rc = lib.psd_sinkhorn_divergence(vp(x), vp(y), b, n, m, blur, scaling, vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds), st)
    assert rc == 1
    return loss, gx, gy, pot, rounds


def bits_equal(a, b):
    if a is None or b is None:
        return a is None and b is None
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def assert_runs_equal(r1, r2):
    for a, b in zip(r1, r2):
        assert bits_equal(a, b)


WORST = {"pot": 0.0, "loss": 0.0, "grad": 0.0}     # worst observed error / tolerance


@pytest.fixture(scope="module", autouse=True)
def report_worst_error():
    yield
    if any(WORST.values()):
        print("\nsinkhorn worst error / tolerance:", {k: round(v, 4) for k, v in WORST.items()})


def record_worst(ratios):
    """Fold one pair's error / tolerance per quantity (test_sinkhorn_fp32.error_ratios) into WORST."""
    WORST["pot"] = max(WORST["pot"], *(ratios[q] for q in ("f_ba", "f_aa", "g_ab", "g_bb")))
    WORST["loss"] = max(WORST["loss"], ratios["S"])
    WORST["grad"] = max(WORST["grad"], ratios["grad_x"], ratios["grad_y"])


def check_against_reference(lib, x, y, blur=0.05, scaling=0.5, cluster=0):
    """Every pair of the batch against ref_torch, within the tolerance that test_sinkhorn_fp32 calibrates from the fp32
    emulation of the kernel on that pair."""
    from test_sinkhorn_fp32 import emulate_pairs, error_ratios, tolerance      # that module imports this one
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    loss, gx, gy, pot, rounds = run(lib, x, y, blur, scaling, cluster)
    torch.cuda.synchronize()
    xc, yc = x.cpu().numpy(), y.cpu().numpy()
    refs = [ref_torch(x[i], y[i], blur, scaling) for i in range(b)]
    emus = emulate_pairs([(xc[i], yc[i]) for i in range(b) if refs[i][4] != 0], blur, scaling)
    for i in range(b):
        K = refs[i][4]
        assert int(rounds[i]) == K
        if K == 0:
            continue
        emu = emus.pop(0)
        assert emu[4] == K
        tol = tolerance(refs[i], emu, diameter(xc[i], yc[i]), n, m, blur, scaling)
        got = (float(loss[i]), (pot[i, :n], pot[i, n:2 * n], pot[i, 2 * n:2 * n + m], pot[i, 2 * n + m:]), gx[i], gy[i])
        ratios = error_ratios(got, refs[i], tol)
        record_worst(ratios)
        assert all(r <= 1.0 for r in ratios.values()), (i, ratios)       # False for NaN
    return loss, gx, gy, pot, rounds


# ---------------------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,b", [(1, 32), (2, 32), (7, 32), (128, 32), (256, 16), (1000, 4), (1024, 4), (2048, 2), (4099, 1)])
def test_matches_reference_equal_sizes(pkg, cuda, kind, n, b):
    x, y = make_clouds(kind, b, n, n, seed=n * 7 + len(kind))
    check_against_reference(pkg._lib.lib, torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda))


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,b", [(128, 1024, 8), (1024, 2048, 2), (1, 300, 16), (300, 1, 16), (1000, 2049, 2)])
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_matches_reference_different_sizes(pkg, cuda, n, m, b, kind):
    x, y = make_clouds(kind, b, n, m, seed=n + 3 * m)
    check_against_reference(pkg._lib.lib, torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda))


@pytest.mark.gpu
@pytest.mark.parametrize("blur,scaling", [(0.01, 0.9), (0.002, 0.95), (0.3, 0.5)])
def test_matches_reference_other_settings(pkg, cuda, blur, scaling):
    x, y = make_clouds("uniform", 4, 256, 200, seed=5)
    check_against_reference(pkg._lib.lib, torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda), blur, scaling)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,b", [(300, 700, 5), (1024, 2048, 3), (5, 3, 9)])
def test_bit_identical_across_cluster_sizes_streams_graphs_and_gradient_requests(pkg, cuda, n, m, b):
    lib = pkg._lib.lib
    x, y = (torch.from_numpy(a).to(cuda) for a in make_clouds("clustered", b, n, m, seed=n * m))
    base = run(lib, x, y)
    for cl in (1, 2, 4, 8):
        assert_runs_equal(run(lib, x, y, cluster=cl), base)
    # without gradients: the same loss, potentials and rounds
    nog = run(lib, x, y, grads=False)
    assert bits_equal(nog[0], base[0]) and bits_equal(nog[3], base[3]) and bits_equal(nog[4], base[4])
    # after unrelated kernels that leave garbage in freed memory (the workspace comes from the stream-ordered pool)
    junk = torch.full((64 << 20,), float("nan"), device=cuda)
    _ = torch.cdist(torch.rand(2048, 64, device=cuda), torch.rand(2048, 64, device=cuda))
    del junk, _
    assert_runs_equal(run(lib, x, y), base)
    # on a side stream
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = run(lib, x, y, stream=s)
    s.synchronize()
    assert_runs_equal(side, base)
    # inside a captured CUDA graph, replayed twice
    bn, nn, mm = b, n, m
    loss = torch.empty(bn, device=cuda)
    gx, gy = torch.empty(bn, nn, 3, device=cuda), torch.empty(bn, mm, 3, device=cuda)
    pot = torch.empty(bn, 2 * nn + 2 * mm, device=cuda)
    rounds = torch.empty(bn, dtype=torch.int32, device=cuda)
    g = torch.cuda.CUDAGraph()
    cs = torch.cuda.Stream()
    cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cs):
        with torch.cuda.graph(g, stream=cs):
            rc = lib.psd_sinkhorn_divergence(vp(x), vp(y), bn, nn, mm, 0.05, 0.5, vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds),
                                             ctypes.c_void_p(cs.cuda_stream))
    assert rc == 1
    for _ in range(2):
        loss.fill_(-1.0); gx.fill_(-1.0); gy.fill_(-1.0); pot.fill_(-1.0); rounds.fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        assert_runs_equal((loss, gx, gy, pot, rounds), base)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(1, 1), (7, 130), (1024, 1024), (1000, 2048)])
def test_identity_and_symmetry_bit_for_bit(pkg, cuda, n, m):
    lib = pkg._lib.lib
    x, y = (torch.from_numpy(a).to(cuda) for a in make_clouds("uniform", 3, n, m, seed=n + m + 1))
    same = run(lib, x, x)
    assert bool((same[0] == 0).all()), same[0]
    assert bool((same[1] == 0).all()) and bool((same[2] == 0).all())
    xy, yx = run(lib, x, y), run(lib, y, x)
    assert bits_equal(xy[0], yx[0])
    assert bits_equal(xy[1], yx[2]) and bits_equal(xy[2], yx[1])
    f_ba, f_aa, g_ab, g_bb = xy[3][:, :n], xy[3][:, n:2 * n], xy[3][:, 2 * n:2 * n + m], xy[3][:, 2 * n + m:]
    r = yx[3]
    assert bits_equal(r[:, :m], g_ab) and bits_equal(r[:, m:2 * m], g_bb)
    assert bits_equal(r[:, 2 * m:2 * m + n], f_ba) and bits_equal(r[:, 2 * m + n:], f_aa)
    assert bits_equal(xy[4], yx[4])


@pytest.mark.gpu
def test_autograd_through_batch_emd_loss(pkg, cuda):
    x0, y0 = (torch.from_numpy(a).to(cuda) for a in make_clouds("uniform", 4, 300, 500, seed=31))
    B = x0.shape[0]
    ref = [ref_torch(x0[i], y0[i]) for i in range(B)]
    rgx = torch.stack([r[2] for r in ref]) / B
    rgy = torch.stack([r[3] for r in ref]) / B
    S_ref = sum(r[0] for r in ref) / B
    from test_sinkhorn_fp32 import emulate_pairs, tolerance
    xc, yc = x0.cpu().numpy(), y0.cpu().numpy()
    tol = [tolerance(r, e, diameter(xc[i], yc[i]), 300, 500, 0.05, 0.5)
           for i, (r, e) in enumerate(zip(ref, emulate_pairs(list(zip(xc, yc)))))]
    # both clouds require grad
    x, y = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
    loss = pkg.loss_.batch_EMD_loss(x, y)
    # the fp32 mean of B losses adds at most a few units of 2^-24
    assert abs(float(loss.detach()) - S_ref) <= sum(t["S"] for t in tol) / B + 2.0 ** -21 * abs(S_ref)
    loss.backward()
    for i in range(B):      # the upstream 1 / B = 1 / 4 scales exactly
        assert float((x.grad[i].double() - rgx[i]).abs().max()) <= tol[i]["grad_x"] / B
        assert float((y.grad[i].double() - rgy[i]).abs().max()) <= tol[i]["grad_y"] / B
    gx_both, gy_both = x.grad.clone(), y.grad.clone()
    # only one
    x = x0.clone().requires_grad_(True)
    pkg.loss_.batch_EMD_loss(x, y0).backward()
    assert bits_equal(x.grad, gx_both)
    y = y0.clone().requires_grad_(True)
    pkg.loss_.batch_EMD_loss(x0, y).backward()
    assert bits_equal(y.grad, gy_both)
    # a transposed view ([B, 3, N] storage)
    xt = x0.transpose(1, 2).contiguous().requires_grad_(True)
    pkg.loss_.batch_EMD_loss(xt.transpose(1, 2), y0).backward()
    assert bits_equal(xt.grad.transpose(1, 2), gx_both)
    # per-cloud upstream weights
    x = x0.clone().requires_grad_(True)
    w = torch.arange(1, B + 1, device=cuda, dtype=torch.float32)
    (pkg.sinkhorn_divergence(x, y0) * w).sum().backward()
    assert torch.allclose(x.grad, gx_both * B * w[:, None, None], rtol=1e-6, atol=0)
    # no input requires grad: plain forward
    assert pkg.sinkhorn_divergence(x0, y0).requires_grad is False


@pytest.mark.gpu
def test_edge_cases(pkg, cuda):
    lib = pkg._lib.lib
    x, y = (torch.from_numpy(a).to(cuda) for a in make_clouds("uniform", 4, 100, 60, seed=41))
    # D = 0: every point of both clouds coincident
    p = torch.full((1, 5, 3), 0.25, device=cuda)
    loss, gx, gy, pot, rounds = run(lib, p, torch.full((1, 9, 3), 0.25, device=cuda))
    assert float(loss[0]) == 0.0 and int(rounds[0]) == 0
    assert bool((gx == 0).all()) and bool((gy == 0).all()) and bool((pot == 0).all())
    # 0 < D <= blur: the two-entry schedule
    xs, ys = x * 0.02, y * 0.02
    res = check_against_reference(lib, xs, ys)
    assert bool((res[4] == 2).all())
    # NaN and inf coordinates in one cloud of the batch: that pair is NaN, the others are as in a run of their own
    for bad in (float("nan"), float("inf"), -float("inf")):
        xb = x.clone()
        xb[2, 17, 1] = bad
        loss, gx, gy, pot, rounds = run(lib, xb, y)
        assert math.isnan(float(loss[2])) and int(rounds[2]) == 0
        assert bool(torch.isnan(gx[2]).all()) and bool(torch.isnan(gy[2]).all()) and bool(torch.isnan(pot[2]).all())
        for i in (0, 1, 3):
            alone = run(lib, x[i:i + 1].contiguous(), y[i:i + 1].contiguous())
            got = (loss[i:i + 1], gx[i:i + 1], gy[i:i + 1], pot[i:i + 1], rounds[i:i + 1])
            assert_runs_equal(got, alone)


@pytest.mark.gpu
def test_argument_errors_and_empty_batch(pkg, cuda):
    lib = pkg._lib.lib
    x = torch.rand(2, 8, 3, device=cuda)
    loss = torch.full((2,), 5.0, device=cuda)
    call = lambda b=2, n=8, m=8, blur=0.05, scaling=0.5, out=loss: lib.psd_sinkhorn_divergence(
        vp(x), vp(x), b, n, m, blur, scaling, vp(out), None, None, None, None, None)
    for kw in (dict(b=-1), dict(b=65536), dict(n=0), dict(m=0), dict(n=(1 << 20) + 1), dict(m=(1 << 20) + 1),
               dict(blur=0.0), dict(blur=-0.1), dict(blur=float("nan")), dict(blur=float("inf")),
               dict(scaling=0.0), dict(scaling=1.0), dict(scaling=1.5), dict(scaling=float("nan")), dict(out=None)):
        assert call(**kw) == -1, kw
        assert "psd_sinkhorn_divergence" in pkg._lib.last_error()
    for cl in (0, 3, 16, -2):
        assert lib.psd_sinkhorn_divergence_cluster(vp(x), vp(x), 2, 8, 8, 0.05, 0.5, vp(loss), None, None, None, None, cl, None) == -1
    assert call(b=0) == 1
    torch.cuda.synchronize()
    assert bool((loss == 5.0).all())
    with pytest.raises(ValueError):
        pkg.sinkhorn_divergence(x, x, blur=0.0)
    with pytest.raises(ValueError):
        pkg.sinkhorn_divergence(x, x, scaling=1.0)
    with pytest.raises(AssertionError):
        pkg.sinkhorn_divergence(x, torch.rand(3, 8, 3, device=cuda))
    with pytest.raises(AssertionError):
        pkg.sinkhorn_divergence(x[:, :, :2], x[:, :, :2])


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [0, 1, 2, 8])
def test_stays_in_bounds(pkg, cuda, cluster):
    from test_gpu_guards import Arena
    lib = pkg._lib.lib
    b, n, m = 3, 333, 1025
    x, y = make_clouds("clustered", b, n, m, seed=51)
    A = Arena(cuda)
    tx, ty = A.tensor(x), A.tensor(y)
    loss, gx, gy = A.empty((b,)), A.empty((b, n, 3)), A.empty((b, m, 3))
    pot, rounds = A.empty((b, 2 * n + 2 * m)), A.empty((b,), torch.int32)
    if cluster:
        rc = lib.psd_sinkhorn_divergence_cluster(vp(tx), vp(ty), b, n, m, 0.05, 0.5, vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds),
                                                 cluster, None)
    else:
        rc = lib.psd_sinkhorn_divergence(vp(tx), vp(ty), b, n, m, 0.05, 0.5, vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds), None)
    assert rc == 1
    A.check(f"sinkhorn, cluster {cluster}")
    assert bool(torch.isfinite(loss).all() & torch.isfinite(gx).all() & torch.isfinite(gy).all() & torch.isfinite(pot).all())
    assert lib.psd_sinkhorn_divergence(vp(tx), vp(ty), b, n, m, 0.05, 0.5, vp(loss), None, None, None, None, None) == 1
    A.check("sinkhorn, loss only")
    assert np.array_equal(tx.cpu().numpy(), x) and np.array_equal(ty.cpu().numpy(), y)


@pytest.mark.gpu
def test_large_clouds_properties(pkg, cuda):
    """n = m = 16384: no dense fp64 reference; symmetry, S(x, x) = 0, cluster-size bit-equality, finite."""
    lib = pkg._lib.lib
    x, y = (torch.from_numpy(a).to(cuda) for a in make_clouds("uniform", 2, 16384, 16384, seed=61))
    xy = run(lib, x, y)
    assert all(bool(torch.isfinite(t).all()) for t in xy[:4]) and bool((xy[0] > 0).all())
    for cl in (1, 8):
        assert_runs_equal(run(lib, x, y, cluster=cl), xy)
    yx = run(lib, y, x)
    assert bits_equal(xy[0], yx[0]) and bits_equal(xy[1], yx[2]) and bits_equal(xy[2], yx[1])
    same = run(lib, x, x)
    assert bool((same[0] == 0).all()) and bool((same[1] == 0).all()) and bool((same[2] == 0).all())
