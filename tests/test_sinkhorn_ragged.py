"""Sinkhorn divergence for ragged and weighted batches (``psd_sinkhorn_divergence_weighted``, ``sinkhorn_divergence(...,
x_lengths, y_lengths, x_weights, y_weights)``, ``pack_clouds``).

The references generalise those of test_sinkhorn.py to point weights: ``ref_numpy_w`` / ``ref_torch_w`` put log a_i per point
into the softmins (a weight of 0 gives h = -inf), weight S as sum_i a_i (f_ba - f_aa) + sum_j b_j (g_ab - g_bb) and scale
gradient row i by a_i.  Log-weights are taken in fp64, so that a point of weight 2/n is the same measure as that point twice.
``emulate_w`` restates the weighted kernel in fp32 from the pieces of test_sinkhorn_fp32.py: h = (logf(w_j) + pot_j / ε) · log₂e
per target, a_i in the gradient, S in fp64, and the kernel's skip of a group of 8 targets whose weights are all 0 (such a group
is left out of the target list, which keeps the other groups' boundaries).  The tolerance is that of test_sinkhorn_fp32.py:
A · err_emu + F per quantity, with the log-weight term of F from max |ln w_j| and a gradient floor 2 a_i ρ D per row.  The
gradient's A · err_emu term is taken per unit of weight (the error of row i over a_i, at most over the rows, times a_i), so
that light rows are not measured against the error of heavy ones."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import make_clouds
from test_sinkhorn import KINDS, _softmin_np, bits_equal, diameter, eps_schedule, f32, log_w, ref_numpy, ref_torch, run, vp
from test_sinkhorn_fp32 import (A, EX2_REL, F32, HALF_LOG2E, LN2, LOG2E, LOG_ULPS, QUANTITIES, _as_dict, _lse, _log2, _ulp,
                                emulate, kernel_eps, max_err, rounding_bound)

POTS = ("f_ba", "f_aa", "g_ab", "g_bb")


# ---------------------------------------------------------------------------------------------------------------- references
def _log(w):
    with np.errstate(divide="ignore"):
        return np.log(np.asarray(w, np.float64))


def _valid(x, y, a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return (np.isfinite(x).all() and np.isfinite(y).all() and np.isfinite(a).all() and np.isfinite(b).all() and
            (a >= 0).all() and (b >= 0).all() and (a > 0).any() and (b > 0).any())


def ref_numpy_w(x, y, a, b, blur=0.05, scaling=0.5):
    """ref_numpy with point weights a [n], b [m]: (S, (f_ba, f_aa, g_ab, g_bb), grad_x, grad_y, rounds)."""
    X, Y = x.astype(np.float64), y.astype(np.float64)
    n, m = len(X), len(Y)
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if not _valid(x, y, a, b):
        nan = float("nan")
        return nan, tuple(np.full(k, nan) for k in (n, n, m, m)), np.full((n, 3), nan), np.full((m, 3), nan), 0
    D = diameter(x, y)
    if D == 0.0:
        return 0.0, tuple(np.zeros(k) for k in (n, n, m, m)), np.zeros((n, 3)), np.zeros((m, 3)), 0
    E = [f32(e) for e in eps_schedule(D, blur, scaling)]
    la, lb = _log(a), _log(b)
    e = E[0]
    g_ab, f_ba = _softmin_np(e, Y, X, la), _softmin_np(e, X, Y, lb)
    f_aa, g_bb = _softmin_np(e, X, X, la), _softmin_np(e, Y, Y, lb)
    for e in E:
        ft_ba, gt_ab = _softmin_np(e, X, Y, lb + g_ab / e), _softmin_np(e, Y, X, la + f_ba / e)
        ft_aa, gt_bb = _softmin_np(e, X, X, la + f_aa / e), _softmin_np(e, Y, Y, lb + g_bb / e)
        f_ba, g_ab, f_aa, g_bb = 0.5 * (f_ba + ft_ba), 0.5 * (g_ab + gt_ab), 0.5 * (f_aa + ft_aa), 0.5 * (g_bb + gt_bb)
    e = E[-1]
    (f_ba2, Pxy), (g_ab2, Pyx) = _softmin_np(e, X, Y, lb + g_ab / e, True), _softmin_np(e, Y, X, la + f_ba / e, True)
    (f_aa2, Qxx), (g_bb2, Qyy) = _softmin_np(e, X, X, la + f_aa / e, True), _softmin_np(e, Y, Y, lb + g_bb / e, True)
    S = (a * (f_ba2 - f_aa2)).sum() + (b * (g_ab2 - g_bb2)).sum()
    return float(S), (f_ba2, f_aa2, g_ab2, g_bb2), a[:, None] * (Pxy - Qxx), b[:, None] * (Pyx - Qyy), len(E)


def ref_torch_w(x, y, a, b, blur=0.05, scaling=0.5):
    """ref_torch with point weights a [n], b [m] (tensors on x's device); autograd gives the gradient."""
    x = x.detach().double().requires_grad_(True)
    y = y.detach().double().requires_grad_(True)
    a, b = a.detach().double().to(x.device), b.detach().double().to(x.device)
    n, m = x.shape[0], y.shape[0]
    if not _valid(x.detach().cpu().numpy(), y.detach().cpu().numpy(), a.cpu().numpy(), b.cpu().numpy()):
        nan = float("nan")
        full = lambda *s: torch.full(s, nan, dtype=torch.float64, device=x.device)
        return nan, (full(n), full(n), full(m), full(m)), full(n, 3), full(m, 3), 0
    D = diameter(x.detach().float().cpu().numpy(), y.detach().float().cpu().numpy())
    if D == 0.0:
        z = lambda *s: torch.zeros(s, dtype=torch.float64, device=x.device)
        return 0.0, (z(n), z(n), z(m), z(m)), z(n, 3), z(m, 3), 0
    E = [f32(e) for e in eps_schedule(D, blur, scaling)]
    la, lb = torch.log(a), torch.log(b)
    cost = lambda u, v: 0.5 * ((u[:, None, :] - v[None, :, :]) ** 2).sum(-1)
    C_xx, C_yy, C_xy, C_yx = cost(x, x.detach()), cost(y, y.detach()), cost(x, y.detach()), cost(y, x.detach())
    sm = lambda eps, C, h: -eps * torch.logsumexp(h[None, :] - C / eps, dim=1)
    with torch.no_grad():
        e = E[0]
        g_ab, f_ba, f_aa, g_bb = sm(e, C_yx, la), sm(e, C_xy, lb), sm(e, C_xx, la), sm(e, C_yy, lb)
        for e in E:
            ft_ba, gt_ab = sm(e, C_xy, lb + g_ab / e), sm(e, C_yx, la + f_ba / e)
            ft_aa, gt_bb = sm(e, C_xx, la + f_aa / e), sm(e, C_yy, lb + g_bb / e)
            f_ba, g_ab, f_aa, g_bb = 0.5 * (f_ba + ft_ba), 0.5 * (g_ab + gt_ab), 0.5 * (f_aa + ft_aa), 0.5 * (g_bb + gt_bb)
    e = E[-1]
    f_ba, g_ab = sm(e, C_xy, (lb + g_ab / e).detach()), sm(e, C_yx, (la + f_ba / e).detach())
    f_aa, g_bb = sm(e, C_xx, (la + f_aa / e).detach()), sm(e, C_yy, (lb + g_bb / e).detach())
    S = (a * (f_ba - f_aa)).sum() + (b * (g_ab - g_bb)).sum()
    gx, gy = torch.autograd.grad(S, [x, y])
    return float(S.detach()), tuple(t.detach() for t in (f_ba, f_aa, g_ab, g_bb)), gx, gy, len(E)


# ---------------------------------------------------------------------------------------------------------------- emulation
def _kept(w):
    """Indices of the targets left after the kernel skips each 8-aligned group whose weights are all 0 (a tile of 512 holds
    whole groups, and only the last group of the cloud is partial)."""
    nt = len(w)
    pos = np.zeros(-(-nt // 8) * 8, bool)
    pos[:nt] = np.asarray(w) > 0
    idx = np.arange(len(pos)).reshape(-1, 8)[pos.reshape(-1, 8).any(1)].reshape(-1)
    return idx[idx < nt]


DEFECTS = ("grad_unweighted", "S_unweighted", "weights_swapped", "padding_included")


def emulate_w(x, y, a, b, blur=0.05, scaling=0.5, defect=None):
    """One valid weighted pair (x [n, 3], y [m, 3], a [n], b [m] fp32) as the weighted sinkhorn_kernel computes it:
    (S, (f_ba, f_aa, g_ab, g_bb), grad_x, grad_y, rounds).  ``defect`` (one of DEFECTS but padding_included, which the caller
    makes by passing the padded cloud) changes one step."""
    x, y, a, b = (np.asarray(v, F32) for v in (x, y, a, b))
    if defect == "weights_swapped":
        a, b = b, a
    n, m = len(x), len(y)
    D = diameter(x, y)
    assert D > 0 and np.isfinite(D)
    E = kernel_eps(D, blur, scaling)
    rounds = [E[0]] + E + [E[-1]]
    K = len(rounds) - 2
    la, lb = _log(a).astype(F32), _log(b).astype(F32)
    kx, ky = _kept(a), _kept(b)
    Q = np.concatenate([x, y])
    sel = np.repeat(np.array([0, 1]), [n, m])
    pot = [np.zeros(n, F32), np.zeros(n, F32), np.zeros(m, F32), np.zeros(m, F32)]    # f_ba, f_aa, g_ab, g_bb
    grad_sums = None
    for t, eps in enumerate(rounds):
        eps = F32(eps)
        init, extrap = t == 0, t == K + 1
        kk = HALF_LOG2E / eps
        nel = -eps * LN2
        f_ba, f_aa, g_ab, g_bb = pot
        h = lambda lw, p: (lw + p / eps) * LOG2E
        MY, sY, WY = _lse(Q, y[ky], np.stack([h(lb, g_ab), h(lb, g_bb)])[:, ky], sel, kk, extrap)
        MX, sX, WX = _lse(Q, x[kx], np.stack([h(la, f_aa), h(la, f_ba)])[:, kx], sel, kk, extrap)
        cross = (np.concatenate([MY[:n], MX[n:]]), np.concatenate([sY[:n], sX[n:]]), np.concatenate([WY[:n], WX[n:]]))
        self_ = (np.concatenate([MX[:n], MY[n:]]), np.concatenate([sX[:n], sY[n:]]), np.concatenate([WX[:n], WY[n:]]))
        fc = nel * (cross[0] + _log2(cross[1]))
        fs = nel * (self_[0] + _log2(self_[1]))
        if not init and not extrap:
            fc = F32(0.5) * (np.concatenate([pot[0], pot[2]]) + fc)
            fs = F32(0.5) * (np.concatenate([pot[1], pot[3]]) + fs)
        pot = [fc[:n], fs[:n], fc[n:], fs[n:]]
        if extrap:
            grad_sums = cross, self_
    (_, sc, Wc), (_, ss, Ws) = grad_sums
    g = Wc / sc[:, None] - Ws / ss[:, None]
    if defect == "grad_unweighted":
        gx, gy = F32(1) / F32(n) * g[:n], F32(1) / F32(m) * g[n:]
    else:
        gx, gy = a[:, None] * g[:n], b[:, None] * g[n:]
    d64 = lambda u, v: u.astype(np.float64) - v
    if defect == "S_unweighted":
        S = d64(pot[0], pot[1]).mean() + d64(pot[2], pot[3]).mean()
    else:
        S = (a.astype(np.float64) * d64(pot[0], pot[1])).sum() + (b.astype(np.float64) * d64(pot[2], pot[3])).sum()
    return float(F32(S)), tuple(pot), gx, gy, len(E)


def _emulate_job(args):
    return emulate_w(*args)


_pool = None


def emulate_w_pairs(jobs):
    """emulate_w(*job) of each job, in parallel processes when there are several."""
    global _pool
    import os
    if len(jobs) <= 1 or (os.cpu_count() or 1) == 1:
        return [emulate_w(*j) for j in jobs]
    if _pool is None:
        import atexit
        import concurrent.futures
        import multiprocessing
        _pool = concurrent.futures.ProcessPoolExecutor(min(32, os.cpu_count()), multiprocessing.get_context("spawn"))
        atexit.register(_pool.shutdown)
    return list(_pool.map(_emulate_job, jobs))


# ---------------------------------------------------------------------------------------------------------------- tolerance
def floors_w(D, a, b, blur, scaling):
    """test_sinkhorn_fp32.floors with point weights: logf(w_j) shifts h_j by at most LOG_ULPS ulp of max |ln w_j| (over the
    positive weights), and the gradient floor of row i is 2 a_i ρ D."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    N = max(len(a), len(b))
    lnw = float(np.abs(np.log(np.concatenate([a[a > 0], b[b > 0]]))).max())
    E = kernel_eps(D, blur, scaling)
    c = 2 * EX2_REL + LOG_ULPS * math.log(2) * _ulp(math.log2(N)) + LOG_ULPS * _ulp(lnw)
    f_pot = c * (E[0] + sum(E) + E[-1])
    rho = 2 * EX2_REL + 2 * c
    return {"S": 4 * f_pot, "f_ba": f_pot, "f_aa": f_pot, "g_ab": f_pot, "g_bb": f_pot,
            "grad_x": 2 * a[:, None] * rho * D, "grad_y": 2 * b[:, None] * rho * D}


def tolerance_w(ref, emu, D, a, b, blur, scaling):
    """A · err_emu + F per quantity; the gradients per row (arrays [n, 1] / [m, 1])."""
    ref, e, F = _as_dict(ref), _as_dict(emu), floors_w(D, a, b, blur, scaling)
    tol = {q: A * max_err(e[q], ref[q]) + F[q] for q in ("S",) + POTS}
    bound = rounding_bound(D, emu[4], blur)
    for q in POTS:
        tol[q] = min(tol[q], bound)
    tol["S"] = min(tol["S"], 2 * bound)
    for q, w in (("grad_x", a), ("grad_y", b)):
        w = np.asarray(w, np.float64)[:, None]
        err = np.abs(e[q] - ref[q])
        per_weight = (err / np.where(w > 0, w, 1.0))[(w > 0)[:, 0]].max()
        tol[q] = A * per_weight * w + F[q]
    return tol


def error_ratios_w(got, ref, tol):
    """max |got − ref| / tolerance per quantity (rows of weight 0 must match exactly; NaN fails)."""
    got, ref = _as_dict(got), _as_dict(ref)
    out = {}
    for q in QUANTITIES:
        err = np.abs(got[q] - ref[q])
        with np.errstate(divide="ignore", invalid="ignore"):
            out[q] = float(np.max(np.where(err == 0, 0.0, err / tol[q])))
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU tests
def _dirichlet(rng, k):
    return rng.dirichlet(np.ones(k)).astype(F32)


def _weights(pattern, rng, k):
    """fp32 weights of one cloud: Dirichlet(1); 90 % zeros and Dirichlet on the rest; one point with 0.99 of the mass."""
    if pattern == "dirichlet":
        return _dirichlet(rng, k)
    w = np.zeros(k, F32)
    if pattern == "sparse":
        keep = rng.permutation(k)[:max(1, k // 10)]
        w[keep] = _dirichlet(rng, len(keep))
    elif pattern == "heavy":
        w[:] = 0.01 / max(k - 1, 1)
        w[rng.integers(k)] = 0.99 if k > 1 else 1.0
    return w


def _defect_case(name):
    """(x, y, a, b) padded with zero rows and positive garbage weights, and the lengths (n_c = m_c, so that x and y weights can
    be swapped)."""
    rng = np.random.default_rng(len(name))
    if name == "dirichlet 300":
        x, y = make_clouds("uniform", 1, 320, 310, seed=1)
        k, a, b = 300, _dirichlet(rng, 300), _dirichlet(rng, 300)
    elif name == "sparse 256":
        x, y = make_clouds("clustered", 1, 270, 256, seed=2)
        k, a, b = 256, _weights("sparse", rng, 256), _dirichlet(rng, 256)
    elif name == "heavy 200":
        x, y = make_clouds("uniform", 1, 208, 240, seed=3)
        k, a, b = 200, _dirichlet(rng, 200), _weights("heavy", rng, 200)
    elif name == "ragged 240":
        x, y = make_clouds("offset", 1, 300, 256, seed=4)
        k, a, b = 240, _dirichlet(rng, 240), _dirichlet(rng, 240)
    x, y = x[0].copy(), y[0].copy()
    x[k:], y[k:] = 0, 0
    pad = lambda w, N: np.concatenate([w, np.resize(w, N - k) + F32(0.01)]).astype(F32)
    return x, y, pad(a, len(x)), pad(b, len(y)), k


DEFECT_CASES = ("dirichlet 300", "sparse 256", "heavy 200", "ragged 240")
_cache = {}


def _case_reference(name):
    if name not in _cache:
        x, y, a, b, k = _defect_case(name)
        ref, emu = ref_numpy_w(x[:k], y[:k], a[:k], b[:k]), emulate_w(x[:k], y[:k], a[:k], b[:k])
        _cache[name] = x, y, a, b, k, ref, emu, tolerance_w(ref, emu, diameter(x[:k], y[:k]), a[:k], b[:k], 0.05, 0.5)
    return _cache[name]


@pytest.mark.parametrize("n,m,kind", [(37, 53, "uniform"), (64, 20, "clustered"), (9, 9, "lattice"), (40, 31, "offset")])
def test_weighted_references_agree_and_reduce_to_the_uniform_ones(n, m, kind):
    x, y = make_clouds(kind, 1, n, m, seed=n + m)
    x, y = x[0], y[0]
    rng = np.random.default_rng(n)
    a, b = _dirichlet(rng, n), _weights("sparse", rng, m)
    r1 = ref_numpy_w(x, y, a, b)
    r2 = ref_torch_w(torch.from_numpy(x), torch.from_numpy(y), torch.from_numpy(a), torch.from_numpy(b))
    assert r1[4] == r2[4] >= 2
    assert math.isclose(r1[0], r2[0], rel_tol=1e-9, abs_tol=1e-12)
    for u, v in zip(r1[1] + r1[2:4], r2[1] + r2[2:4]):
        np.testing.assert_allclose(u, v.numpy(), rtol=1e-8, atol=1e-12)
    # uniform weights: the references of test_sinkhorn.py, which take log(1/n) rounded to fp32
    ua, ub = np.full(n, math.exp(log_w(n))), np.full(m, math.exp(log_w(m)))
    for got, want in ((ref_numpy_w(x, y, ua, ub), ref_numpy(x, y)),
                      (ref_torch_w(*(torch.from_numpy(v) for v in (x, y, ua, ub))), ref_torch(torch.from_numpy(x), torch.from_numpy(y)))):
        g, w = _as_dict(got), _as_dict(want)
        assert got[4] == want[4]
        for q in QUANTITIES:
            np.testing.assert_allclose(g[q], w[q], rtol=1e-6, atol=1e-12, err_msg=q)


def test_a_double_weight_is_a_duplicated_point():
    x, y = make_clouds("uniform", 1, 40, 30, seed=9)
    x, y = x[0], y[0]
    n, m = len(x), len(y)
    a = np.full(n, 1.0 / (n + 1))
    a[7] = 2.0 / (n + 1)
    dup = np.concatenate([x, x[7:8]])
    r1 = ref_numpy_w(x, y, a, np.full(m, 1.0 / m))
    r2 = ref_numpy_w(dup, y, np.full(n + 1, 1.0 / (n + 1)), np.full(m, 1.0 / m))
    assert r1[4] == r2[4]
    assert abs(r1[0] - r2[0]) <= 1e-12
    np.testing.assert_allclose(r1[1][0], r2[1][0][:n], rtol=0, atol=1e-12)       # f_ba
    np.testing.assert_allclose(r1[1][1], r2[1][1][:n], rtol=0, atol=1e-12)       # f_aa
    np.testing.assert_allclose(r1[1][2], r2[1][2], rtol=0, atol=1e-12)           # g_ab
    np.testing.assert_allclose(r1[1][3], r2[1][3], rtol=0, atol=1e-12)           # g_bb
    np.testing.assert_allclose(r1[3], r2[3], rtol=0, atol=1e-12)
    gd = r2[2][:n].copy()
    gd[7] += r2[2][n]                                                            # both copies move with x_7
    np.testing.assert_allclose(r1[2], gd, rtol=0, atol=1e-12)


@pytest.mark.parametrize("n,m", [(37, 53), (300, 200), (9, 1)])
def test_emulation_with_uniform_weights_gives_the_bits_of_the_uniform_emulation(n, m):
    x, y = make_clouds("clustered", 1, n, m, seed=n * m)
    a, b = np.full(n, F32(1) / F32(n), F32), np.full(m, F32(1) / F32(m), F32)
    got, want = emulate_w(x[0], y[0], a, b), emulate(x[0], y[0])
    assert got[4] == want[4]
    for u, v in zip(got[1] + got[2:4], want[1] + want[2:4]):
        assert np.array_equal(u.view(np.int32), v.view(np.int32))
    assert abs(got[0] - want[0]) <= 2 * _ulp(want[0])


@pytest.mark.parametrize("name", DEFECT_CASES)
def test_weighted_emulation_is_close_to_the_fp64_reference(name):
    x, y, a, b, k, ref, emu, tol = _case_reference(name)
    assert emu[4] == ref[4]
    r, e = _as_dict(ref), _as_dict(emu)
    for q in ("grad_x", "grad_y"):
        assert max_err(e[q], r[q]) <= 1e-3 * np.abs(r[q]).max(), q
    assert max(error_ratios_w(emu, ref, tol).values()) <= 1 / A


def test_zero_weight_groups_are_skipped_not_nan():
    """90 % zero weights leave whole groups of 8 without mass, some of them before the first positive weight."""
    x, y, a, b, k, ref, emu, tol = _case_reference("sparse 256")
    assert len(_kept(a[:k])) < k
    assert all(np.isfinite(v).all() for v in _as_dict(emu).values())


@pytest.mark.parametrize("defect", DEFECTS)
@pytest.mark.parametrize("name", DEFECT_CASES)
def test_weighted_defects_fail_the_check_tenfold(name, defect):
    x, y, a, b, k, ref, emu, tol = _case_reference(name)
    if defect == "padding_included":
        bad = emulate_w(x, y, a, b)
        bad = (bad[0], tuple(p[:k] for p in bad[1]), bad[2][:k], bad[3][:k], bad[4])
    else:
        bad = emulate_w(x[:k], y[:k], a[:k], b[:k], defect=defect)
    ratios = error_ratios_w(bad, ref, tol)
    assert max(ratios.values()) >= 10, (defect, ratios)


def test_python_validates_host_lengths_and_weights(pkg):
    x, y = torch.rand(2, 5, 3), torch.rand(2, 4, 3)
    for kw in (dict(x_lengths=[0, 3]), dict(x_lengths=[1, 6]), dict(y_lengths=[5, 1]), dict(x_lengths=[1, 2, 3]),
               dict(x_lengths=[1.0, 2.0]), dict(y_lengths=torch.tensor([-1, 2])),
               dict(x_weights=torch.rand(2, 4)), dict(y_weights=torch.rand(2, 4, 1))):
        with pytest.raises(ValueError):
            pkg.sinkhorn_divergence(x, y, **kw)
    with pytest.raises(ValueError, match="not differentiable"):
        pkg.sinkhorn_divergence(x, y, x_weights=torch.rand(2, 5, requires_grad=True))


def test_pack_clouds_round_trip(pkg):
    clouds = [torch.rand(k, 3) for k in (5, 1, 9, 3)]
    xp, lengths = pkg.pack_clouds(clouds)
    assert xp.shape == (4, 9, 3) and lengths.dtype == torch.int32 and lengths.tolist() == [5, 1, 9, 3]
    for i, c in enumerate(clouds):
        assert torch.equal(xp[i, :len(c)], c) and bool((xp[i, len(c):] == 0).all())
    for bad in ([], [torch.rand(0, 3)], [torch.rand(4, 2)]):
        with pytest.raises(ValueError):
            pkg.pack_clouds(bad)


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
def run_w(lib, x, y, xl=None, yl=None, xw=None, yw=None, blur=0.05, scaling=0.5, cluster=0, grads=True, stream=None):
    """psd_sinkhorn_divergence_weighted(_cluster) on device tensors: (loss, grad_x, grad_y, potentials, rounds)."""
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    dev = x.device
    loss = torch.full((b,), -1.0, device=dev)
    gx = torch.full((b, n, 3), -1.0, device=dev) if grads else None
    gy = torch.full((b, m, 3), -1.0, device=dev) if grads else None
    pot = torch.full((b, 2 * n + 2 * m), -1.0, device=dev)
    rounds = torch.full((b,), -7, dtype=torch.int32, device=dev)
    st = ctypes.c_void_p(stream.cuda_stream) if stream is not None else None
    if cluster:
        rc = lib.psd_sinkhorn_divergence_weighted_cluster(vp(x), vp(y), b, n, m, vp(xl), vp(yl), vp(xw), vp(yw), blur, scaling,
                                                          vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds), cluster, st)
    else:
        rc = lib.psd_sinkhorn_divergence_weighted(vp(x), vp(y), b, n, m, vp(xl), vp(yl), vp(xw), vp(yw), blur, scaling, vp(loss),
                                                  vp(gx), vp(gy), vp(pot), vp(rounds), st)
    assert rc == 1
    return loss, gx, gy, pot, rounds


def pair(res, c, nc, mc):
    """Pair c of a run with padded sizes, cut to its lengths: (loss, grad_x, grad_y, f_ba, f_aa, g_ab, g_bb, rounds)."""
    loss, gx, gy, pot, rounds = res
    n, m = gx.shape[1], gy.shape[1]
    P = pot[c]
    return (loss[c:c + 1], gx[c, :nc], gy[c, :mc], P[:nc], P[n:n + nc], P[2 * n:2 * n + mc], P[2 * n + m:2 * n + m + mc],
            rounds[c:c + 1])


def assert_pairs_equal(p1, p2, what=""):
    for i, (u, v) in enumerate(zip(p1, p2)):
        assert bits_equal(u, v), (what, i)


def assert_padding_zero(res, c, nc, mc):
    loss, gx, gy, pot, rounds = res
    n, m = gx.shape[1], gy.shape[1]
    P = pot[c]
    for t in (gx[c, nc:], gy[c, mc:], P[nc:n], P[n + nc:2 * n], P[2 * n + mc:2 * n + m], P[2 * n + m + mc:]):
        assert bits_equal(t, torch.zeros_like(t))


def _dev(a, cuda, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda) if dtype is None else torch.as_tensor(a, dtype=dtype).to(cuda)


WORST = {"pot": 0.0, "loss": 0.0, "grad": 0.0}     # worst observed error / tolerance over the weighted cases


@pytest.fixture(scope="module", autouse=True)
def report_worst_weighted_error():
    yield
    if any(WORST.values()):
        print("\nweighted sinkhorn worst error / tolerance:", {k: round(v, 4) for k, v in WORST.items()})


def check_weighted(lib, x, y, xl, yl, xw, yw, blur=0.05, scaling=0.5, cluster=0):
    """Every pair of one ragged / weighted launch against ref_torch_w on its participating points, within the tolerance
    calibrated by emulate_w on that pair."""
    b = x.shape[0]
    res = run_w(lib, x, y, xl, yl, xw, yw, blur, scaling, cluster)
    torch.cuda.synchronize()
    lx, ly = xl.tolist(), yl.tolist()
    parts = [(x[c, :lx[c]], y[c, :ly[c]], xw[c, :lx[c]], yw[c, :ly[c]]) for c in range(b)]
    refs = [ref_torch_w(*p, blur, scaling) for p in parts]
    emus = emulate_w_pairs([tuple(t.cpu().numpy() for t in p) + (blur, scaling) for p in parts])
    for c in range(b):
        K = refs[c][4]
        assert K > 0 and emus[c][4] == K and int(res[4][c]) == K
        xa, ya, wa, wb = (t.cpu().numpy() for t in parts[c])
        tol = tolerance_w(refs[c], emus[c], diameter(xa, ya), wa, wb, blur, scaling)
        _, gx, gy, f_ba, f_aa, g_ab, g_bb, _ = pair(res, c, lx[c], ly[c])
        ratios = error_ratios_w((float(res[0][c]), (f_ba, f_aa, g_ab, g_bb), gx, gy), refs[c], tol)
        WORST["pot"] = max(WORST["pot"], *(ratios[q] for q in POTS))
        WORST["loss"] = max(WORST["loss"], ratios["S"])
        WORST["grad"] = max(WORST["grad"], ratios["grad_x"], ratios["grad_y"])
        assert all(r <= 1.0 for r in ratios.values()), (c, ratios)
        assert_padding_zero(res, c, lx[c], ly[c])
    return res


# ---------------------------------------------------------------------------------------------------------------- GPU tests
LENGTHS = {
    "ones": lambda n, m: ([1] * 6, [1] * 6),
    "full": lambda n, m: ([n] * 6, [m] * 6),
    "mixed": lambda n, m: ([1, n, 300, 7, n - 1, 1000], [m, 1, 17, 1024, 513, 2]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [0, 1, 2, 4, 8])
@pytest.mark.parametrize("lengths", list(LENGTHS))
def test_ragged_pairs_equal_standalone_runs(pkg, cuda, lengths, cluster):
    """Each pair of one ragged launch has the bits of psd_sinkhorn_divergence on x[c, :n_c], y[c, :m_c] alone; rows past the
    lengths are 0, and NaN in the padding is never read.  n = m = 4099 padded, so "mixed" has 1 point against 4099."""
    lib = pkg._lib.lib
    n = m = 4099
    x, y = make_clouds("clustered", 6, n, m, seed=17)
    lx, ly = LENGTHS[lengths](n, m)
    for c in range(6):
        x[c, lx[c]:], y[c, ly[c]:] = np.nan, np.nan
    tx, ty = _dev(x, cuda), _dev(y, cuda)
    xl, yl = _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32)
    res = run_w(lib, tx, ty, xl, yl, cluster=cluster)
    torch.cuda.synchronize()
    for c in range(6):
        alone = run(lib, tx[c:c + 1, :lx[c]].contiguous(), ty[c:c + 1, :ly[c]].contiguous(), cluster=cluster)
        assert_pairs_equal(pair(res, c, lx[c], ly[c]), pair(alone, 0, lx[c], ly[c]), (lengths, c))
        assert_padding_zero(res, c, lx[c], ly[c])
        assert int(res[4][c]) >= 2
    if lengths == "full":
        assert_pairs_equal(run_w(lib, tx, ty, cluster=cluster), res)     # NULL lengths: n and m


@pytest.mark.gpu
def test_ragged_batch_of_65535_tiny_pairs(pkg, cuda):
    """b = 65535 pairs of 1 to 4 points padded to 4: each equals the plain kernel on a batch of the pairs with its lengths."""
    lib = pkg._lib.lib
    b = 65535
    rng = np.random.default_rng(5)
    x, y = rng.random((b, 4, 3), dtype=np.float32), rng.random((b, 4, 3), dtype=np.float32)
    lx, ly = rng.integers(1, 5, b), rng.integers(1, 5, b)
    for c in range(b):
        x[c, lx[c]:], y[c, ly[c]:] = np.nan, np.nan
    tx, ty = _dev(x, cuda), _dev(y, cuda)
    res = run_w(lib, tx, ty, _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32))
    torch.cuda.synchronize()
    loss, gx, gy, pot, rounds = res
    for nc in range(1, 5):
        for mc in range(1, 5):
            idx = torch.from_numpy(np.nonzero((lx == nc) & (ly == mc))[0]).to(cuda)
            ref = run(lib, tx[idx, :nc].contiguous(), ty[idx, :mc].contiguous())
            assert bits_equal(loss[idx], ref[0]) and bits_equal(rounds[idx], ref[4])
            assert bits_equal(gx[idx, :nc], ref[1]) and bits_equal(gy[idx, :mc], ref[2])
            P, R = pot[idx], ref[3]
            for (o, k, ro) in ((0, nc, 0), (4, nc, nc), (8, mc, 2 * nc), (8 + 4, mc, 2 * nc + mc)):
                assert bits_equal(P[:, o:o + k], R[:, ro:ro + k]), (nc, mc, o)
            assert bool((gx[idx, nc:] == 0).all()) and bool((gy[idx, mc:] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("nc,mc", [(500, 333), (7, 1030)])
def test_zero_weight_padding_keeps_the_bits(pkg, cuda, nc, mc):
    """Padding a cloud's tail with zero-weight copies of its first point leaves D as it is, and gives the bits of the unpadded
    cloud with the same weights (groups of zero weight are skipped)."""
    lib = pkg._lib.lib
    b, n, m = 3, nc + 45, mc + 530
    x, y = make_clouds("uniform", b, nc, mc, seed=nc + mc)
    rng = np.random.default_rng(nc)
    a = np.stack([_dirichlet(rng, nc) for _ in range(b)])
    w = np.stack([_weights("sparse", rng, mc) for _ in range(b)])
    xp = np.concatenate([x, np.repeat(x[:, :1], n - nc, 1)], 1)
    yp = np.concatenate([y, np.repeat(y[:, :1], m - mc, 1)], 1)
    ap = np.concatenate([a, np.zeros((b, n - nc), F32)], 1)
    wp = np.concatenate([w, np.zeros((b, m - mc), F32)], 1)
    small = run_w(lib, _dev(x, cuda), _dev(y, cuda), xw=_dev(a, cuda), yw=_dev(w, cuda))
    padded = run_w(lib, _dev(xp, cuda), _dev(yp, cuda), xw=_dev(ap, cuda), yw=_dev(wp, cuda))
    torch.cuda.synchronize()
    for c in range(b):
        assert_pairs_equal(pair(padded, c, nc, mc), pair(small, c, nc, mc), c)
        assert bool((padded[1][c, nc:] == 0).all()) and bool((padded[2][c, mc:] == 0).all())   # weight 0: no gradient


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [0, 2])
def test_explicit_uniform_weights_equal_null_weights(pkg, cuda, cluster):
    lib = pkg._lib.lib
    b, n, m = 4, 700, 513
    x, y = make_clouds("clustered", b, n, m, seed=3)
    lx, ly = [700, 1, 333, 64], [513, 200, 1, 100]
    a = np.full((b, n), 7.0, F32)           # past the lengths: never read
    w = np.full((b, m), np.nan, F32)
    for c in range(b):
        a[c, :lx[c]] = F32(1) / F32(lx[c])
        w[c, :ly[c]] = F32(1) / F32(ly[c])
    tx, ty = _dev(x, cuda), _dev(y, cuda)
    xl, yl = _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32)
    null = run_w(lib, tx, ty, xl, yl, cluster=cluster)
    expl = run_w(lib, tx, ty, xl, yl, _dev(a, cuda), _dev(w, cuda), cluster=cluster)
    torch.cuda.synchronize()
    for c in range(b):
        p0, p1 = pair(null, c, lx[c], ly[c]), pair(expl, c, lx[c], ly[c])
        assert_pairs_equal(p0[1:], p1[1:], c)
        S0, S1 = float(p0[0]), float(p1[0])
        assert abs(S0 - S1) <= 2 * _ulp(S0), (c, S0, S1)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["dirichlet", "sparse", "heavy"])
@pytest.mark.parametrize("kind", KINDS)
def test_weighted_matches_reference(pkg, cuda, kind, pattern):
    """Ragged (n ≠ m) weighted pairs against the weighted fp64 torch reference, within 4 · err_emu + F."""
    b, n, m = 3, 230, 170
    x, y = make_clouds(kind, b, n, m, seed=len(kind) * 13 + len(pattern))
    lx, ly = [200, 230, 57], [150, 170, 170]
    rng = np.random.default_rng(len(pattern))
    a, w = np.zeros((b, n), F32), np.zeros((b, m), F32)
    for c in range(b):
        a[c, :lx[c]] = _weights(pattern, rng, lx[c])
        w[c, :ly[c]] = _weights("dirichlet" if pattern == "sparse" else pattern, rng, ly[c])
    check_weighted(pkg._lib.lib, _dev(x, cuda), _dev(y, cuda), _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32),
                   _dev(a, cuda), _dev(w, cuda))


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [1, 8])
def test_weighted_matches_reference_other_settings(pkg, cuda, cluster):
    """blur 0.01 / scaling 0.9 and forced cluster sizes, with 1 point against 400."""
    b, n, m = 3, 400, 128
    x, y = make_clouds("uniform", b, n, m, seed=77)
    lx, ly = [1, 400, 250], [128, 100, 1]
    rng = np.random.default_rng(1)
    a, w = np.zeros((b, n), F32), np.zeros((b, m), F32)
    for c in range(b):
        a[c, :lx[c]] = _dirichlet(rng, lx[c])
        w[c, :ly[c]] = _weights("heavy", rng, ly[c])
    check_weighted(pkg._lib.lib, _dev(x, cuda), _dev(y, cuda), _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32),
                   _dev(a, cuda), _dev(w, cuda), 0.01, 0.9, cluster)


def _sym_inputs(cuda, b=4, n=300, m=700):
    x, y = make_clouds("clustered", b, n, m, seed=n * m)
    rng = np.random.default_rng(2)
    lx, ly = [300, 5, 211, 1], [700, 650, 3, 399]
    a, w = np.zeros((b, n), F32), np.zeros((b, m), F32)
    for c in range(b):
        a[c, :lx[c]] = _weights("sparse", rng, lx[c])
        w[c, :ly[c]] = _dirichlet(rng, ly[c])
    return (_dev(x, cuda), _dev(y, cuda), _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32), _dev(a, cuda),
            _dev(w, cuda))


@pytest.mark.gpu
def test_weighted_symmetry_bit_for_bit(pkg, cuda):
    lib = pkg._lib.lib
    x, y, xl, yl, xw, yw = _sym_inputs(cuda)
    n, m = x.shape[1], y.shape[1]
    xy, yx = run_w(lib, x, y, xl, yl, xw, yw), run_w(lib, y, x, yl, xl, yw, xw)
    assert bits_equal(xy[0], yx[0]) and bits_equal(xy[4], yx[4])
    assert bits_equal(xy[1], yx[2]) and bits_equal(xy[2], yx[1])
    p, r = xy[3], yx[3]
    assert bits_equal(r[:, :m], p[:, 2 * n:2 * n + m]) and bits_equal(r[:, m:2 * m], p[:, 2 * n + m:])
    assert bits_equal(r[:, 2 * m:2 * m + n], p[:, :n]) and bits_equal(r[:, 2 * m + n:], p[:, n:2 * n])
    same = run_w(lib, x, x, xl, xl, xw, xw)
    assert bool((same[0] == 0).all()) and bool((same[1] == 0).all()) and bool((same[2] == 0).all())


@pytest.mark.gpu
def test_weighted_bit_identical_across_cluster_sizes_streams_graphs_and_gradient_requests(pkg, cuda):
    lib = pkg._lib.lib
    x, y, xl, yl, xw, yw = _sym_inputs(cuda)
    args = (x, y, xl, yl, xw, yw)
    base = run_w(lib, *args)
    for cl in (1, 2, 4, 8):
        assert_pairs_equal(run_w(lib, *args, cluster=cl), base, cl)
    nog = run_w(lib, *args, grads=False)
    assert bits_equal(nog[0], base[0]) and bits_equal(nog[3], base[3]) and bits_equal(nog[4], base[4])
    junk = torch.full((64 << 20,), float("nan"), device=cuda)
    del junk
    assert_pairs_equal(run_w(lib, *args), base, "after junk")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = run_w(lib, *args, stream=s)
    s.synchronize()
    assert_pairs_equal(side, base, "side stream")
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    loss, gx, gy = torch.empty(b, device=cuda), torch.empty(b, n, 3, device=cuda), torch.empty(b, m, 3, device=cuda)
    pot, rounds = torch.empty(b, 2 * n + 2 * m, device=cuda), torch.empty(b, dtype=torch.int32, device=cuda)
    g = torch.cuda.CUDAGraph()
    cs = torch.cuda.Stream()
    cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cs):
        with torch.cuda.graph(g, stream=cs):
            rc = lib.psd_sinkhorn_divergence_weighted(vp(x), vp(y), b, n, m, vp(xl), vp(yl), vp(xw), vp(yw), 0.05, 0.5,
                                                      vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds),
                                                      ctypes.c_void_p(cs.cuda_stream))
    assert rc == 1
    for _ in range(2):
        loss.fill_(-1.0); gx.fill_(-1.0); gy.fill_(-1.0); pot.fill_(-1.0); rounds.fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        assert_pairs_equal((loss, gx, gy, pot, rounds), base, "graph")


@pytest.mark.gpu
def test_invalid_lengths_and_weights_make_only_their_pair_nan(pkg, cuda):
    lib = pkg._lib.lib
    b, n, m = 10, 60, 50
    x, y = make_clouds("uniform", b, n, m, seed=8)
    rng = np.random.default_rng(3)
    lx, ly = [60, 0, 40, -3, 60, 60, 60, 60, 30, 20], [50, 50, 51, 50, 50, 50, 50, 50, 50, 10]
    a, w = np.zeros((b, n), F32), np.zeros((b, m), F32)
    for c in range(b):
        a[c, :max(lx[c], 1)] = _dirichlet(rng, min(max(lx[c], 1), n))
        w[c, :ly[c] if ly[c] <= m else m] = _dirichlet(rng, min(ly[c], m))
    a[0, 10] = 0.0                      # a zero weight is valid
    a[8, 30:] = np.nan                  # past the length: never read
    a[4, 5] = -1e-30                    # negative
    w[5, 7] = np.nan
    a[6, 0] = np.inf
    a[7, :] = 0.0                       # all zero on x
    w[9, :10] = 0.0                     # all participating y weights zero (the rest, past the length, is not)
    w[9, 10:] = 0.5
    bad = {1, 2, 3, 4, 5, 6, 7, 9}
    tx, ty = _dev(x, cuda), _dev(y, cuda)
    xl, yl, xw, yw = _dev(lx, cuda, torch.int32), _dev(ly, cuda, torch.int32), _dev(a, cuda), _dev(w, cuda)
    loss, gx, gy, pot, rounds = run_w(lib, tx, ty, xl, yl, xw, yw)
    torch.cuda.synchronize()
    for c in range(b):
        if c in bad:
            assert math.isnan(float(loss[c])) and int(rounds[c]) == 0, c
            assert bool(torch.isnan(gx[c]).all()) and bool(torch.isnan(gy[c]).all()) and bool(torch.isnan(pot[c]).all()), c
        else:
            alone = run_w(lib, tx[c:c + 1], ty[c:c + 1], xl[c:c + 1], yl[c:c + 1], xw[c:c + 1], yw[c:c + 1])
            got = (loss[c:c + 1], gx[c:c + 1], gy[c:c + 1], pot[c:c + 1], rounds[c:c + 1])
            assert_pairs_equal(got, alone, c)
            assert bool(torch.isfinite(loss[c])), c
    # a NaN coordinate inside the length, and one past it
    x2 = x.copy()
    x2[0, 59, 1] = np.nan
    x2[8, 45, 0] = np.nan
    res = run_w(lib, _dev(x2, cuda), ty, xl, yl, xw, yw)
    assert math.isnan(float(res[0][0])) and bool(torch.isnan(res[1][0]).all())
    assert bits_equal(res[0][8:9], loss[8:9]) and bits_equal(res[1][8], gx[8])


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [0, 1, 8])
def test_weighted_stays_in_bounds(pkg, cuda, cluster):
    from test_gpu_guards import Arena
    lib = pkg._lib.lib
    b, n, m = 3, 333, 1025
    x, y = make_clouds("clustered", b, n, m, seed=51)
    lx, ly = np.array([333, 100, 1], np.int32), np.array([1025, 1, 700], np.int32)
    rng = np.random.default_rng(4)
    a = np.stack([_weights("sparse", rng, n) for _ in range(b)])
    w = np.stack([_dirichlet(rng, m) for _ in range(b)])
    for c in range(b):
        a[c, :lx[c]][0] = 0.5           # at least one positive participating weight per side
        w[c, :ly[c]][0] = 0.5
    Ar = Arena(cuda)
    tx, ty, txl, tyl, txw, tyw = (Ar.tensor(v) for v in (x, y, lx, ly, a, w))
    loss, gx, gy = Ar.empty((b,)), Ar.empty((b, n, 3)), Ar.empty((b, m, 3))
    pot, rounds = Ar.empty((b, 2 * n + 2 * m)), Ar.empty((b,), torch.int32)
    if cluster:
        rc = lib.psd_sinkhorn_divergence_weighted_cluster(vp(tx), vp(ty), b, n, m, vp(txl), vp(tyl), vp(txw), vp(tyw), 0.05, 0.5,
                                                          vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds), cluster, None)
    else:
        rc = lib.psd_sinkhorn_divergence_weighted(vp(tx), vp(ty), b, n, m, vp(txl), vp(tyl), vp(txw), vp(tyw), 0.05, 0.5,
                                                  vp(loss), vp(gx), vp(gy), vp(pot), vp(rounds), None)
    assert rc == 1
    Ar.check(f"weighted sinkhorn, cluster {cluster}")
    assert bool(torch.isfinite(loss).all() & torch.isfinite(gx).all() & torch.isfinite(gy).all() & torch.isfinite(pot).all())
    assert lib.psd_sinkhorn_divergence_weighted(vp(tx), vp(ty), b, n, m, vp(txl), None, None, vp(tyw), 0.05, 0.5, vp(loss),
                                                None, None, None, None, None) == 1
    Ar.check("weighted sinkhorn, loss only")
    for t, v in ((tx, x), (ty, y), (txl, lx), (tyl, ly), (txw, a), (tyw, w)):
        assert np.array_equal(t.cpu().numpy(), v, equal_nan=True)


@pytest.mark.gpu
def test_weighted_argument_errors(pkg, cuda):
    lib = pkg._lib.lib
    x = torch.rand(2, 8, 3, device=cuda)
    loss = torch.full((2,), 5.0, device=cuda)
    call = lambda b=2, n=8, m=8, blur=0.05, scaling=0.5, out=loss: lib.psd_sinkhorn_divergence_weighted(
        vp(x), vp(x), b, n, m, None, None, None, None, blur, scaling, vp(out), None, None, None, None, None)
    for kw in (dict(b=-1), dict(b=65536), dict(n=0), dict(m=0), dict(n=(1 << 20) + 1), dict(blur=0.0),
               dict(blur=float("nan")), dict(scaling=1.0), dict(scaling=0.0), dict(out=None)):
        assert call(**kw) == -1, kw
        assert "psd_sinkhorn_divergence_weighted" in pkg._lib.last_error()
    for cl in (0, 3, 16):
        assert lib.psd_sinkhorn_divergence_weighted_cluster(vp(x), vp(x), 2, 8, 8, None, None, None, None, 0.05, 0.5, vp(loss),
                                                            None, None, None, None, cl, None) == -1
    assert call(b=0) == 1
    torch.cuda.synchronize()
    assert bool((loss == 5.0).all())


@pytest.mark.gpu
def test_python_ragged_weighted_autograd(pkg, cuda):
    b, n, m = 3, 120, 90
    x0, y0 = (_dev(v, cuda) for v in make_clouds("uniform", b, n, m, seed=12))
    lx, ly = [120, 64, 5], [90, 90, 33]
    rng = np.random.default_rng(6)
    a, w = np.zeros((b, n), F32), np.zeros((b, m), F32)
    for c in range(b):
        a[c, :lx[c]] = _dirichlet(rng, lx[c])
        w[c, :ly[c]] = _weights("sparse", rng, ly[c])
    xw, yw = _dev(a, cuda), _dev(w, cuda)
    x, y = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
    up = torch.tensor([1.0, -2.0, 0.5], device=cuda)
    S = pkg.sinkhorn_divergence(x, y, x_lengths=lx, y_lengths=torch.tensor(ly), x_weights=xw, y_weights=yw)
    (S * up).sum().backward()
    for c in range(b):
        parts = (x0[c, :lx[c]], y0[c, :ly[c]], xw[c, :lx[c]], yw[c, :ly[c]])
        ref = ref_torch_w(*parts)
        emu = emulate_w(*(t.cpu().numpy() for t in parts))
        tol = tolerance_w(ref, emu, diameter(*(t.cpu().numpy() for t in parts[:2])), a[c, :lx[c]], w[c, :ly[c]], 0.05, 0.5)
        assert abs(float(S[c]) - ref[0]) <= tol["S"]
        u = float(up[c])        # a power of 2: scales exactly
        assert bool(((x.grad[c, :lx[c]].double() - u * ref[2]).abs() <= abs(u) * torch.from_numpy(tol["grad_x"]).to(cuda)).all())
        assert bool(((y.grad[c, :ly[c]].double() - u * ref[3]).abs() <= abs(u) * torch.from_numpy(tol["grad_y"]).to(cuda)).all())
        assert bool((x.grad[c, lx[c]:] == 0).all()) and bool((y.grad[c, ly[c]:] == 0).all())
    # the same lengths as a CUDA tensor, and pack_clouds
    xp, lp = pkg.pack_clouds([x0[c, :lx[c]] for c in range(b)])
    assert lp.is_cuda
    S2 = pkg.sinkhorn_divergence(xp, y0, x_lengths=lp, y_lengths=torch.tensor(ly, device=cuda), x_weights=xw, y_weights=yw)
    assert bits_equal(S2, S.detach())
    # weights that require grad
    with pytest.raises(ValueError):
        pkg.sinkhorn_divergence(x, y, x_weights=xw.clone().requires_grad_(True))
    with torch.no_grad():
        S3 = pkg.sinkhorn_divergence(x0, y0, x_lengths=lx, y_lengths=ly, x_weights=xw.clone().requires_grad_(True), y_weights=yw)
    assert bits_equal(S3, S.detach())
    # a length out of range in a CUDA tensor is not checked on the host: that pair is NaN
    S4 = pkg.sinkhorn_divergence(x0, y0, x_lengths=torch.tensor([0, 64, 5], device=cuda, dtype=torch.int32))
    assert math.isnan(float(S4[0])) and bool(torch.isfinite(S4[1:]).all())
