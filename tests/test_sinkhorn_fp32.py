"""``sinkhorn_kernel`` against an fp32 emulation of its own arithmetic.

``emulate`` restates csrc/sinkhorn.cu operation for operation in numpy: the ε of each round as ``eps_of_round`` rounds it, log a
and log b as logf(1/n), the staged h = (log w + potential / ε) · log₂e, kk = ½ log₂e / ε, z = fma(−|q − t|², kk, h) with the
squared distance of ``sqdist_exact``, the running base-2 maximum updated once per group of 8 targets in index order (with the
rescale of s and of the three gradient accumulators), the averaging of rounds 1 to K, the extrapolation round with its fused
gradient a · (W_c / s_c − W_s / s_s), and S summed in fp64.  Every fp32 operation is rounded to fp32; an fma is evaluated in
fp64 and rounded once.  Where the kernel uses an approximation, the emulation rounds the exact value instead: ``ex2.approx.ftz``
becomes exp2 rounded to fp32 with subnormal results flushed to zero, and logf / log2f become the rounded fp64 logarithms.

Against the fp64 references of test_sinkhorn.py, the emulation's error err_emu = max |emu − ref| of each quantity measures what
fp32 arithmetic in this operation order costs on that cloud pair.  The kernel must then satisfy, per quantity,
max |kernel − ref| ≤ A · err_emu + F (``tolerance``).  F covers what the emulation cannot reproduce, the approximate ex2 / logf
/ log2f, from the error bounds that the PTX ISA and the CUDA math documentation state (``floors``).  The potentials and S are
also held to the older rounding bound (``rounding_bound``) where that is tighter.

The CPU tests run the emulation with deliberate defects (``DEFECTS``) and require each to fail the same check by a factor of
10 or more, so that the check is known to see a wrong gradient, a missing round or a stale buffer.  The GPU tests run the
kernel at coordinate scales from 1e-21 to 1e17, at extreme size ratios and at forced cluster sizes."""
import atexit
import math
import os

import numpy as np
import pytest
import torch

from conftest import make_clouds
from test_sinkhorn import check_against_reference, diameter, eps_schedule, ref_numpy, report_worst_error  # noqa: F401

F32 = np.float32
LOG2E, HALF_LOG2E, LN2 = F32(1.4426950408889634), F32(0.7213475204444817), F32(0.6931471805599453)
MIN_EPS = 2.0 ** -128       # csrc/sinkhorn.cu kSkMinEps: the least ε for which ½ log₂e / ε is finite in fp32

A = 4.0                     # kernel error / emulation error allowed per quantity
EX2_REL = 2.0 ** -22        # ex2.approx.f32: at most 2 ulp from 2^x (PTX ISA), a relative error of at most 2^-22
LOG_ULPS = 1.5              # logf / log2f: at most 1 ulp (CUDA math documentation), against the emulation's 0.5 ulp rounding

QUANTITIES = ("S", "f_ba", "f_aa", "g_ab", "g_bb", "grad_x", "grad_y")

DEFECTS = ("grad_scaled", "grad_no_debias", "grad_x_over_m", "grad_no_rescale", "grad_from_loop", "drop_round",
           "extra_round", "self_not_averaged", "stale_h")


# ---------------------------------------------------------------------------------------------------------------- emulation
def _fma(a, b, c):
    """fmaf: the product of two fp32 values is exact in fp64; the fp64 sum is rounded to fp32 (a double rounding, which can
    differ from a true fma by one ulp in rare ties)."""
    return (np.asarray(a, np.float64) * b + c).astype(F32)


def _ex2(v):
    """ex2.approx.ftz.f32 as 2^v rounded to fp32, with subnormal results flushed to zero."""
    r = np.exp2(np.asarray(v, np.float64)).astype(F32)
    r[r < np.finfo(F32).tiny] = 0
    return r


def _log2(v):
    return np.log2(np.asarray(v, np.float64)).astype(F32)


def _lse(Q, T, h, sel, kk, grad, rescale_grad=True):
    """lse_tile over all targets T [nt, 3] for the queries Q [nq, 3]: query i reads the staged h of row sel[i] of h [2, nt].
    Returns the running maximum M, the sum s and the gradient accumulators W [nq, 3]."""
    nq, nt = len(Q), len(T)
    pad = -nt % 8                          # the tile's tail: zero coordinates, h = -inf
    T = np.concatenate([T, np.zeros((pad, 3), F32)])
    h = np.concatenate([h, np.full((2, pad), -np.inf, F32)], axis=1)
    M = np.full(nq, -np.inf, F32)
    s = np.zeros(nq, F32)
    W = np.zeros((nq, 3), F32)
    buf = np.empty((nq, 9), F32)
    chunk = 512
    for c0 in range(0, nt + pad, chunk):
        d = Q[:, None, :] - T[None, c0:c0 + chunk, :]
        sq = _fma(d[..., 2], d[..., 2], _fma(d[..., 0], d[..., 0], d[..., 1] * d[..., 1]))
        z = _fma(-sq, kk, h[sel, c0:c0 + chunk]).reshape(nq, -1, 8)
        # the running maximum after each group; where it moves the kernel multiplies s (and W) by 2^(M_old - M_new), 0 while
        # M is -inf; where it stays, the factor here is 2^0 = 1 and the product is exact, as if skipped
        Mg = np.maximum.accumulate(np.concatenate([M[:, None], z.max(2)], axis=1), axis=1)
        fac = _ex2(Mg[:, :-1] - Mg[:, 1:])
        e = _ex2(z - Mg[:, 1:, None])
        for g in range(z.shape[1]):
            buf[:, 0] = s * fac[:, g]
            buf[:, 1:] = e[:, g]
            s = np.add.accumulate(buf, axis=1)[:, -1]      # the 8 fp32 additions in order
            if grad:
                if rescale_grad:
                    W = W * fac[:, g, None]
                for u in range(8):
                    W = _fma(e[:, g, u, None], d[:, 8 * g + u], W)
        M = Mg[:, -1]
    return M, s, W


def kernel_eps(D, blur, scaling):
    """The ε of each loop round as eps_of_round computes it: the schedule in double, rounded to fp32, at least MIN_EPS."""
    return [max(float(F32(e)), MIN_EPS) for e in eps_schedule(D, blur, scaling)]


def emulate(x, y, blur=0.05, scaling=0.5, defect=None):
    """One finite cloud pair with D > 0 (x [n, 3], y [m, 3] fp32), as sinkhorn_kernel computes it:
    (S, (f_ba, f_aa, g_ab, g_bb), grad_x, grad_y, rounds).  ``defect`` (one of DEFECTS, None) changes one step."""
    x, y = np.asarray(x, F32), np.asarray(y, F32)
    n, m = len(x), len(y)
    D = diameter(x, y)
    assert D > 0 and np.isfinite(D)
    E = kernel_eps(D, blur, scaling)
    loop = E[:-1] if defect == "drop_round" else E + [E[-1]] if defect == "extra_round" else E
    rounds = [E[0]] + loop + [E[-1]]                  # init, the loop, the extrapolation
    K = len(rounds) - 2
    logw = lambda k: F32(np.log(np.float64(F32(1) / F32(k))))
    la, lb = logw(n), logw(m)
    Q = np.concatenate([x, y])
    sel = np.repeat(np.array([0, 1]), [n, m])         # row 0 of h for the x-queries, row 1 for the y-queries
    pot = [np.zeros(n, F32), np.zeros(n, F32), np.zeros(m, F32), np.zeros(m, F32)]    # f_ba, f_aa, g_ab, g_bb
    older = pot
    grad_sums = None
    for t, eps in enumerate(rounds):
        eps = F32(eps)
        init, extrap = t == 0, t == K + 1
        grad = t == (K if defect == "grad_from_loop" else K + 1)
        kk = HALF_LOG2E / eps
        nel = -eps * LN2
        f_ba, f_aa, g_ab, g_bb = older if defect == "stale_h" else pot
        h = lambda lw, p: (lw + p / eps) * LOG2E
        # targets Y: the x-queries' cross softmin (h of g_ab), the y-queries' self softmin (h of g_bb); targets X: the
        # x-queries' self softmin (f_aa), the y-queries' cross softmin (f_ba)
        rescale = defect != "grad_no_rescale"
        MY, sY, WY = _lse(Q, y, np.stack([h(lb, g_ab), h(lb, g_bb)]), sel, kk, grad, rescale)
        MX, sX, WX = _lse(Q, x, np.stack([h(la, f_aa), h(la, f_ba)]), sel, kk, grad, rescale)
        cross = (np.concatenate([MY[:n], MX[n:]]), np.concatenate([sY[:n], sX[n:]]), np.concatenate([WY[:n], WX[n:]]))
        self_ = (np.concatenate([MX[:n], MY[n:]]), np.concatenate([sX[:n], sY[n:]]), np.concatenate([WX[:n], WY[n:]]))
        fc = nel * (cross[0] + _log2(cross[1]))
        fs = nel * (self_[0] + _log2(self_[1]))
        if not init and not extrap:
            fc = F32(0.5) * (np.concatenate([pot[0], pot[2]]) + fc)
            if defect != "self_not_averaged":
                fs = F32(0.5) * (np.concatenate([pot[1], pot[3]]) + fs)
        older, pot = pot, [fc[:n], fs[:n], fc[n:], fs[n:]]
        if grad:
            grad_sums = cross, self_
    (_, sc, Wc), (_, ss, Ws) = grad_sums
    if defect == "grad_no_debias":
        Ws = np.zeros_like(Ws)
    g = Wc / sc[:, None] - Ws / ss[:, None]
    ax, ay = F32(1) / F32(m if defect == "grad_x_over_m" else n), F32(1) / F32(m)
    gx, gy = ax * g[:n], ay * g[n:]
    if defect == "grad_scaled":
        k = F32(0.95 if blur < 0.01 else 0.99)
        gx, gy = gx * k, gy * k
    S = float(F32((pot[0].astype(np.float64) - pot[1]).mean() + (pot[2].astype(np.float64) - pot[3]).mean()))
    return S, tuple(pot), gx, gy, len(loop)


def _emulate_pair(args):
    return emulate(*args)


_pool = None


def emulate_pairs(pairs, blur=0.05, scaling=0.5):
    """emulate() of each (x, y) in pairs, in parallel processes when there are several (seconds per pair at n + m ~ 2000)."""
    global _pool
    jobs = [(x, y, blur, scaling) for x, y in pairs]
    if len(jobs) <= 1 or (os.cpu_count() or 1) == 1:
        return [emulate(*j) for j in jobs]
    if _pool is None:
        import concurrent.futures
        import multiprocessing
        _pool = concurrent.futures.ProcessPoolExecutor(min(32, os.cpu_count()), multiprocessing.get_context("spawn"))
        atexit.register(_pool.shutdown)
    return list(_pool.map(_emulate_pair, jobs))


# ---------------------------------------------------------------------------------------------------------------- tolerance
def _ulp(v):
    return float(np.spacing(F32(abs(v))))


def floors(D, n, m, blur, scaling):
    """F per quantity: the difference between the kernel's ex2.approx / logf / log2f and the emulation's rounded exact values.
    One softmin at ε: each term 2^(z − M) and each rescale factor is off by at most EX2_REL relative, so log₂ s by
    2 EX2_REL / ln 2 and the potential by 2 ε EX2_REL; log₂ s ∈ [0, log₂ N] carries LOG_ULPS ulp of log₂ N (times ε ln 2), and
    logf(1/N) shifts every h by LOG_ULPS ulp of ln N (times ε): c ε in all.  ex2.approx's error need not average out like a
    rounding error, and a bias common to all terms moves every potential of every round; the softmin is 1-Lipschitz in the
    potentials it reads and the averaging is a convex combination, so the potentials carry at most F_pot = c Σ_t ε_t over the
    K + 2 rounds.  S is two means of potential differences: 4 F_pot.  A bias common to the weights cancels in the gradient
    a Σ_j P_j (q − t_j), minus the same over the own cloud; what does not is each weight's own error, 2 EX2_REL from its ex2
    terms and the potential errors of the last two rounds (at blur²) in its h, ρ = 2 EX2_REL + 2 c relative, which moves each
    weighted mean by at most ρ D: F = 2 a ρ D."""
    N = max(n, m)
    E = kernel_eps(D, blur, scaling)
    c = 2 * EX2_REL + LOG_ULPS * math.log(2) * _ulp(math.log2(N)) + LOG_ULPS * _ulp(math.log(N))
    f_pot = c * (E[0] + sum(E) + E[-1])
    rho = 2 * EX2_REL + 2 * c
    fg = lambda k: 2.0 / k * rho * D
    return {"S": 4 * f_pot, "f_ba": f_pot, "f_aa": f_pot, "g_ab": f_pot, "g_bb": f_pot, "grad_x": fg(n), "grad_y": fg(m)}


def _as_dict(res):
    S, (f_ba, f_aa, g_ab, g_bb), gx, gy = res[:4]
    a = lambda v: np.asarray(v.cpu() if torch.is_tensor(v) else v, np.float64)
    return {"S": np.float64(S), "f_ba": a(f_ba), "f_aa": a(f_aa), "g_ab": a(g_ab), "g_bb": a(g_bb), "grad_x": a(gx),
            "grad_y": a(gy)}


def max_err(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max())


def rounding_bound(D, rounds, blur):
    """A bound on a potential's error from fp32 rounding alone, kept where it is tighter than A · err_emu + F: an exponent
    h_j − C_ij / ε carries a few units of 2^-24 of its size (about max(D², ε) / ε), so each round adds about
    max(D², blur²) 2^-24 to a potential, 16 (K + 2) such units in all.  S: twice that."""
    return 16.0 * (rounds + 2) * max(D * D, float(F32(blur)) ** 2) * 2.0 ** -24


def tolerance(ref, emu, D, n, m, blur, scaling):
    """A · err_emu + F per quantity, the potentials and S at most rounding_bound; ref and emu as returned by ref_numpy /
    ref_torch and emulate."""
    ref, emu, F = _as_dict(ref), _as_dict(emu), floors(D, n, m, blur, scaling)
    tol = {q: A * max_err(emu[q], ref[q]) + F[q] for q in QUANTITIES}
    bound = rounding_bound(D, emu[4] if isinstance(emu, tuple) else len(kernel_eps(D, blur, scaling)), blur)
    for q in ("f_ba", "f_aa", "g_ab", "g_bb"):
        tol[q] = min(tol[q], bound)
    tol["S"] = min(tol["S"], 2 * bound)
    return tol


def error_ratios(got, ref, tol):
    """max |got − ref| / tolerance per quantity."""
    got, ref = _as_dict(got), _as_dict(ref)
    return {q: max_err(got[q], ref[q]) / tol[q] for q in QUANTITIES}


# ---------------------------------------------------------------------------------------------------------------- CPU tests
def _case(name):
    """The cloud pairs the defect tests use: (x, y, blur, scaling)."""
    if name == "clustered 1024":
        x, y = make_clouds("clustered", 1, 1024, 1024, seed=7)
    elif name == "uniform 1000/2049":
        x, y = make_clouds("uniform", 1, 1000, 2049, seed=8)
    elif name == "blur 0.002":
        x, y = make_clouds("uniform", 1, 256, 200, seed=5)
        return x[0], y[0], 0.002, 0.95
    elif name == "D <= blur":
        x, y = make_clouds("uniform", 1, 100, 60, seed=41)
        x, y = x * F32(0.028), y * F32(0.028)             # D = 0.047
    return x[0], y[0], 0.05, 0.5


CASES = ("clustered 1024", "uniform 1000/2049", "blur 0.002", "D <= blur")
_cache = {}


def _reference_and_emulation(name):
    if name not in _cache:
        x, y, blur, scaling = _case(name)
        ref, emu = ref_numpy(x, y, blur, scaling), emulate(x, y, blur, scaling)
        _cache[name] = x, y, blur, scaling, ref, emu, tolerance(ref, emu, diameter(x, y), len(x), len(y), blur, scaling)
    return _cache[name]


@pytest.mark.parametrize("name", CASES)
def test_emulation_is_close_to_the_fp64_reference(name):
    """The emulation follows the reference's schedule; its error is fp32 rounding, far inside a 1 % gradient budget."""
    x, y, blur, scaling, ref, emu, tol = _reference_and_emulation(name)
    assert emu[4] == ref[4]
    r, e = _as_dict(ref), _as_dict(emu)
    assert abs(e["S"] - r["S"]) <= 1e-6 * max(np.abs(r[q]).max() for q in ("f_ba", "f_aa", "g_ab", "g_bb"))
    for q in ("grad_x", "grad_y"):
        assert max_err(e[q], r[q]) <= 1e-3 * np.abs(r[q]).max(), q
        assert tol[q] <= 0.01 * np.abs(r[q]).max(), q
    assert max(error_ratios(emu, ref, tol).values()) <= 1 / A


# Defects that do not change the fp64 result on a case beyond what the kernel's documented ex2 error allows, and why
UNDETECTABLE = {
    ("clustered 1024", "grad_x_over_m"): "n = m: 1/m is 1/n",
    ("blur 0.002", "grad_no_debias"): "at ε = blur² = 4e-6 each point's self-transport plan is itself, so the debias term is 0",
    ("D <= blur", "grad_from_loop"): "at ε = blur² > D² the loop's last round has converged: its weights are the extrapolation's",
    ("D <= blur", "extra_round"): "at ε = blur² > D² the loop's last round has converged: one more changes nothing",
}


@pytest.mark.parametrize("defect", DEFECTS)
@pytest.mark.parametrize("name", CASES)
def test_defects_fail_the_check_tenfold(name, defect):
    x, y, blur, scaling, ref, emu, tol = _reference_and_emulation(name)
    if (name, defect) in UNDETECTABLE:
        pytest.skip(UNDETECTABLE[name, defect])
    bad = emulate(x, y, blur, scaling, defect)
    worst = max(error_ratios(bad, ref, tol).values())
    assert worst >= 10, (defect, error_ratios(bad, ref, tol))


def test_emulation_at_tiny_diameter_matches_the_reference():
    """At D ~ 1e-21 the first rounds' ε = D² is raised to MIN_EPS (2^-128); the rounds at blur² do not see the difference."""
    x, y = make_clouds("uniform", 1, 64, 48, seed=5)
    for s in (1e-21, 1e-19):
        xs, ys = x[0] * F32(s), y[0] * F32(s)
        ref, emu = ref_numpy(xs, ys), emulate(xs, ys)
        assert all(np.isfinite(v).all() for v in _as_dict(emu).values())
        tol = tolerance(ref, emu, diameter(xs, ys), 64, 48, 0.05, 0.5)
        assert max(error_ratios(emu, ref, tol).values()) <= 1 / A
        r = _as_dict(ref)
        assert max_err(_as_dict(emu)["grad_x"], r["grad_x"]) <= 1e-5 * np.abs(r["grad_x"]).max()


# ---------------------------------------------------------------------------------------------------------------- GPU tests
def _pair(x, y, cuda):
    return torch.from_numpy(np.ascontiguousarray(x, F32)).to(cuda), torch.from_numpy(np.ascontiguousarray(y, F32)).to(cuda)


@pytest.mark.gpu
@pytest.mark.parametrize("shift,scale", [(0.0, 1e-21), (0.0, 1e-19), (0.0, 1e-12), (0.0, 1e-3), (0.0, 1e4), (0.0, 1e12),
                                         (0.0, 1e17), (1e4, 1.0), (-1e4, 1.0)])
def test_coordinate_scales(pkg, cuda, shift, scale):
    """One cloud pair scaled from D ~ 1e-21 (where the first rounds' ε = D² is raised to 2^-128) to D ~ 1e17, and moved to
    ±1e4 (coordinates with an ulp of 1e-3): finite, and within the calibrated tolerance of the fp64 reference."""
    x, y = make_clouds("uniform", 2, 64, 48, seed=5)
    x, y = (x * F32(scale) + F32(shift)).astype(F32), (y * F32(scale) + F32(shift)).astype(F32)
    loss, gx, gy, pot, rounds = check_against_reference(pkg._lib.lib, *_pair(x, y, cuda))
    assert all(bool(torch.isfinite(t).all()) for t in (loss, gx, gy, pot)) and bool((rounds >= 2).all())


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(1, 4099), (4099, 1)])
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_extreme_size_ratios(pkg, cuda, n, m, kind):
    x, y = make_clouds(kind, 1, n, m, seed=n + 2 * m)
    check_against_reference(pkg._lib.lib, *_pair(x, y, cuda))


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [1, 8])
@pytest.mark.parametrize("name", CASES)
def test_tolerance_holds_for_every_cluster_size(pkg, cuda, name, cluster):
    x, y, blur, scaling = _case(name)
    check_against_reference(pkg._lib.lib, *_pair(x[None], y[None], cuda), blur, scaling, cluster)
