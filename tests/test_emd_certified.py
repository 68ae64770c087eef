"""Certified EMD: epsilon-scaling phases of the auction and the weak-duality certificate (psd_emd_certified,
psd_emd_dual_bound, emd_module.emd_certified, metrics.certified_emd_distance).

The references live here: `eps_scaling` runs the phases over the CPU oracle's auction (bit-faithful to the GPU kernel)
with the prices carried from phase to phase, `dual_bound` is the certificate in numpy fp64, and the exact optimum comes
from scipy's linear_sum_assignment on the Euclidean cost.  The CPU tests check the method itself; the GPU tests check the
library against these references."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from conftest import make_clouds


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def phase_eps(eps_end=1e-4, eps_start=0.05, scale=4.0):
    """psd_emd_certified's schedule: eps_start / scale^i in double (from the float arguments), rounded to float, down to
    exactly eps_end."""
    e, end, s = float(np.float32(eps_start)), float(np.float32(eps_end)), float(np.float32(scale))
    out = []
    while e > end:
        out.append(np.float32(e))
        e /= s
    out.append(np.float32(end))
    return out


def eps_scaling(O, x, y, eps_end=1e-4, eps_start=0.05, scale=4.0, max_iters_per_phase=20000, nthreads=8):
    """The phases over the oracle's C auction: each from assignment = -1 (assignment_inv = -1, other scratch 0: the
    reference's initial state) and the previous phase's prices.  Returns dist, assignment, price, bidder scans per phase."""
    x, y = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(y, np.float32)
    b, n, _ = x.shape
    f, i = O._f, O._i
    price = np.zeros((b, n), np.float32)
    dist = np.zeros((b, n), np.float32)
    scans = []
    for eps in phase_eps(eps_end, eps_start, scale):
        ass = np.full((b, n), -1, np.int32)
        inv = np.full((b, n), -1, np.int32)
        bid, binc, minc = np.zeros((b, n), np.int32), np.zeros((b, n), np.float32), np.zeros((b, n), np.float32)
        uidx, midx = np.zeros(b * n, np.int32), np.zeros(b * n, np.int32)
        stats = np.zeros(3, np.int64)
        rc = O._c().oracle_emd_forward(b, n, n, f(x), f(y), f(dist), i(ass), f(price), i(inv), i(bid), f(binc), f(minc), i(uidx),
                                       i(midx), ctypes.c_float(eps), int(max_iters_per_phase),
                                       stats.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), None, int(nthreads))
        assert rc == 1
        scans.append(int(stats[0]))
    return dist, ass, price, scans


def dual_bound(x, y, assignment, price=None):
    """The certificate in numpy fp64, round to nearest: bounds[B, 2] = (L / n, U / n), status[B]."""
    x1, x2 = np.asarray(x, np.float32).astype(np.float64), np.asarray(y, np.float32).astype(np.float64)
    b, n, _ = x1.shape
    p = np.zeros((b, n)) if price is None else np.asarray(price, np.float32).astype(np.float64)
    bounds, status = np.zeros((b, 2)), np.zeros(b, np.int32)
    for c in range(b):
        mins = np.empty(n)
        for j0 in range(0, n, 512):
            d = np.sqrt(((x1[c, j0:j0 + 512, None, :] - x2[c, None, :, :]) ** 2).sum(-1))
            mins[j0:j0 + 512] = (d + p[c][None, :]).min(1)
        bounds[c, 0] = (mins.sum() - p[c].sum()) / n
        a = np.asarray(assignment[c])
        perm = bool(((a >= 0) & (a < n)).all()) and np.unique(a).size == n
        status[c] = int(perm)
        bounds[c, 1] = np.sqrt(((x1[c] - x2[c][a]) ** 2).sum(-1)).sum() / n if perm else np.nan
    return bounds, status


def exact_emd(x, y):
    """Optimal matching cost per point of every cloud (Euclidean, fp64)."""
    x1, x2 = np.asarray(x, np.float64), np.asarray(y, np.float64)
    out = []
    for c in range(x1.shape[0]):
        cost = np.sqrt(((x1[c][:, None, :] - x2[c][None, :, :]) ** 2).sum(-1))
        r, k = linear_sum_assignment(cost)
        out.append(cost[r, k].sum() / x1.shape[1])
    return np.array(out)


_CACHE = {}


def case(O, kind, b, n, eps_end, seed=None, max_iters_per_phase=20000):
    key = (kind, b, n, eps_end, seed, max_iters_per_phase)
    if key not in _CACHE:
        x, y = make_clouds(kind, b, n, n, seed=seed if seed is not None else 500 + n)
        dist, ass, price, scans = eps_scaling(O, x, y, eps_end, max_iters_per_phase=max_iters_per_phase)
        _CACHE[key] = dict(x=x, y=y, dist=dist, ass=ass, price=price, scans=scans)
    return _CACHE[key]


def exact_of(c):
    if "exact" not in c:
        c["exact"] = exact_emd(c["x"], c["y"])
    return c["exact"]


def assert_brackets(bounds, exact, rel=1e-12):
    lo, hi = bounds[:, 0], bounds[:, 1]
    assert (lo <= exact * (1 + rel)).all(), (lo, exact)
    assert (exact <= hi * (1 + rel)).all(), (exact, hi)


def is_perm(a):
    n = a.shape[-1]
    return all(np.array_equal(np.sort(r), np.arange(n)) for r in np.asarray(a))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the method
# ---------------------------------------------------------------------------------------------------------------------
def test_phase_schedule():
    s = phase_eps(1e-5, 0.05, 4.0)
    assert len(s) == 8 and s[0] == np.float32(0.05) and s[1] == np.float32(0.0125) and s[-1] == np.float32(1e-5)
    assert phase_eps(1e-4, 1e-4, 4.0) == [np.float32(1e-4)]


@pytest.mark.parametrize("n,eps_end", [(1024, 1e-5), (2048, 1e-4)])
@pytest.mark.parametrize("kind", ["uniform", "clustered", "lattice", "dup"])
def test_eps_scaling_reaches_certified_matching(oracle, kind, n, eps_end):
    c = case(oracle, kind, 2, n, eps_end)
    assert is_perm(c["ass"])
    bounds, status = dual_bound(c["x"], c["y"], c["ass"], c["price"])
    assert (status == 1).all()
    assert_brackets(bounds, exact_of(c))
    assert (bounds[:, 1] - bounds[:, 0] <= eps_end).all(), bounds[:, 1] - bounds[:, 0]
    # the matching's own cost (what dist reports, in fp32) is the upper bound up to fp32 rounding
    assert np.allclose(np.sqrt(c["dist"].astype(np.float64)).mean(1), bounds[:, 1], rtol=1e-6, atol=0)


def test_dual_bound_is_a_lower_bound_for_any_prices(oracle):
    x, y = make_clouds("clustered", 2, 1024, 1024, seed=11)
    exact = exact_emd(x, y)
    rng = np.random.default_rng(12)
    ident = np.tile(np.arange(1024, dtype=np.int32), (2, 1))
    _, _, state = oracle.emd_forward(x, y, 0.05, 3000, nthreads=8, full_state=True)
    for price in (None, np.zeros((2, 1024), np.float32), rng.random((2, 1024), dtype=np.float32) * 2 - 1, state["price"]):
        bounds, status = dual_bound(x, y, ident, price)
        assert (status == 1).all()
        assert (bounds[:, 0] <= exact * (1 + 1e-12)).all()
        assert (exact <= bounds[:, 1]).all()   # any permutation is an upper bound


def test_evaluation_setting_is_not_a_matching(oracle):
    """Metrics._get_emd_distance's setting (eps 0.005, 50 iterations) ends with forced assignments: the certificate says so
    and keeps only the lower bound, which the returned value undercuts."""
    x, y = make_clouds("uniform", 2, 1024, 1024, seed=13)
    dist, ass = oracle.emd_forward(x, y, 0.005, 50, nthreads=2)
    bounds, status = dual_bound(x, y, ass)
    assert (status == 0).all() and np.isnan(bounds[:, 1]).all()
    exact = exact_emd(x, y)
    assert (bounds[:, 0] <= exact).all()
    assert (np.sqrt(dist.astype(np.float64)).mean(1) < exact).all()


def test_python_limits_fire_before_device_work(pkg):
    import torch
    with pytest.raises(AssertionError):
        pkg.emd_certified(torch.rand(2, 1000, 3), torch.rand(2, 1000, 3))
    with pytest.raises(AssertionError):
        pkg.emd_certified(torch.rand(2, 1024, 3), torch.rand(2, 2048, 3))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the library against the references
# ---------------------------------------------------------------------------------------------------------------------
def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def run_certified(pkg, dev, x, y, eps_end, eps_start=0.05, scale=4.0, max_iters=20000, cluster=None, stream=None):
    import torch
    b, n, _ = x.shape
    tx, ty = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    dist = torch.full((b, n), float("nan"), device=dev)
    ass = torch.full((b, n), 7, device=dev, dtype=torch.int32)
    price = torch.full((b, n), float("nan"), device=dev)
    bounds = torch.full((b, 2), -1.0, device=dev, dtype=torch.float64)
    status = torch.full((b,), 7, device=dev, dtype=torch.int32)
    lib = pkg._lib.lib
    args = (vp(tx), vp(ty), b, n, eps_start, eps_end, scale, max_iters, vp(dist), vp(ass), vp(price), vp(bounds), vp(status))
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())   # the inputs were copied on the current stream
    s = pkg._lib.stream_of(tx) if stream is None else ctypes.c_void_p(stream.cuda_stream)
    rc = lib.psd_emd_certified(*args, s) if cluster is None else lib.psd_emd_certified_cluster(*args, cluster, s)
    assert rc == 1, pkg._lib.last_error()
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in (dist, ass, price, bounds, status)]


def assert_close_bounds(got, want, rel=1e-12):
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert (np.abs(got[ok] - want[ok]) <= rel * np.abs(want[ok])).all(), (got, want)


GPU_CASES = [("uniform", 2, 1024, 1e-4), ("clustered", 2, 2048, 1e-5), ("lattice", 2, 1024, 1e-4), ("dup", 2, 1024, 1e-5)]


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [None, 1, 2, 4, 8, -2])
@pytest.mark.parametrize("cfg", GPU_CASES)
def test_gpu_certified_matches_reference(pkg, oracle, cuda, cluster, cfg):
    """dist, assignment and final prices bit-equal to the reference phases for every decomposition of the auction kernel
    (None = automatic, negative = the global-workspace form); bounds within 1e-12 of the numpy certificate and around the
    exact optimum."""
    kind, b, n, eps_end = cfg
    c = case(oracle, kind, b, n, eps_end)
    dist, ass, price, bounds, status = run_certified(pkg, cuda, c["x"], c["y"], eps_end, cluster=cluster)
    assert np.array_equal(ass, c["ass"]), f"assignment differs in {(ass != c['ass']).sum()} places"
    assert np.array_equal(dist.view(np.uint32), c["dist"].view(np.uint32))
    assert np.array_equal(price.view(np.uint32), c["price"].view(np.uint32))
    want, wstatus = dual_bound(c["x"], c["y"], c["ass"], c["price"])
    assert np.array_equal(status, wstatus) and (status == 1).all()
    assert_close_bounds(bounds, want)
    assert_brackets(bounds, exact_of(c), rel=0.0)   # the GPU bounds are directed-rounded: no slack needed
    assert (bounds[:, 1] - bounds[:, 0] <= eps_end).all()


@pytest.mark.gpu
def test_gpu_budget_exhausted_reports_no_matching(pkg, oracle, cuda):
    """A phase that runs out of iterations ends with the auction's forced assignment, where several winners of one object
    add to its price in the same iteration (a race in the reference too): the prices the next phase starts from, and so
    the result, are not reproducible bit for bit.  What must hold is that the certificate of whatever came out is right."""
    c = case(oracle, "uniform", 2, 1024, 1e-4, max_iters_per_phase=3)
    assert not is_perm(c["ass"])
    dist, ass, price, bounds, status = run_certified(pkg, cuda, c["x"], c["y"], 1e-4, max_iters=3)
    assert (status == 0).all() and np.isnan(bounds[:, 1]).all()
    want, wstatus = dual_bound(c["x"], c["y"], ass, price)
    assert (wstatus == 0).all()
    assert_close_bounds(bounds, want)
    assert (bounds[:, 0] <= exact_of(c)).all()


@pytest.mark.gpu
def test_gpu_limits_return_minus_one(pkg, cuda):
    import torch
    lib = pkg._lib.lib
    b, n = 2, 1024
    t = torch.zeros(b * n * 4, device=cuda, dtype=torch.float64)   # large enough for every buffer; never written on -1
    p = vp(t)
    bad = [dict(b=513), dict(n=1000), dict(n=0), dict(eps_end=1e-6), dict(eps_end=float("nan")), dict(eps_end=0.1),
           dict(scale=1.0), dict(scale=0.5), dict(scale=1.0001), dict(max_iters=0)]
    for kw in bad:
        a = dict(b=b, n=n, eps_start=0.05, eps_end=1e-4, scale=4.0, max_iters=100)
        a.update(kw)
        for fn, extra in ((lib.psd_emd_certified, ()), (lib.psd_emd_certified_cluster, (2,))):
            rc = fn(p, p, a["b"], a["n"], a["eps_start"], a["eps_end"], a["scale"], a["max_iters"], p, p, p, p, p, *extra, None)
            assert rc == -1, kw
            assert pkg._lib.last_error(), kw
    assert lib.psd_emd_dual_bound(p, p, -1, n, p, p, p, p, None) == -1
    assert lib.psd_emd_dual_bound(p, p, b, 0, p, p, p, p, None) == -1
    assert lib.psd_emd_dual_bound(p, p, b, (1 << 20) + 1, p, p, p, p, None) == -1
    torch.cuda.synchronize()
    assert float(t.abs().sum()) == 0.0
    x = torch.rand(2, 1024, 3, device=cuda)
    with pytest.raises(ValueError, match="eps_end"):
        pkg.emd_certified(x, x, eps_end=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 4099])
def test_gpu_dual_bound_any_assignment(pkg, cuda, n):
    """Standalone certificate at ragged sizes (rows past the last CTA's 64, several 2048-object tiles): permutations with
    random, zero and NULL prices; a non-permutation keeps its lower bound."""
    import torch
    b = 3
    x, y = make_clouds("uniform", b, n, n, seed=21)
    rng = np.random.default_rng(22)
    perm = np.stack([rng.permutation(n) for _ in range(b)]).astype(np.int32)
    notperm = perm.copy()
    notperm[1, 5] = notperm[1, 6]
    notperm[2, 0] = n          # out of range
    lib = pkg._lib.lib
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    for a, price in ((perm, rng.random((b, n), dtype=np.float32)), (perm, None), (notperm, np.zeros((b, n), np.float32))):
        ta = torch.from_numpy(a).to(cuda)
        tp = None if price is None else torch.from_numpy(price).to(cuda)
        bounds = torch.zeros(b, 2, device=cuda, dtype=torch.float64)
        status = torch.full((b,), 7, device=cuda, dtype=torch.int32)
        assert lib.psd_emd_dual_bound(vp(tx), vp(ty), b, n, vp(ta), vp(tp), vp(bounds), vp(status), None) == 1, pkg._lib.last_error()
        want, wstatus = dual_bound(x, y, a, price)
        assert np.array_equal(status.cpu().numpy(), wstatus)
        assert_close_bounds(bounds.cpu().numpy(), want)
    assert wstatus.tolist() == [1, 0, 0]


@pytest.mark.gpu
def test_gpu_dual_bound_certifies_the_reference_interface(pkg, oracle, cuda):
    """psd_emd_dual_bound on the (assignment, price) that the 14-tensor psd_emd_forward leaves at the training setting."""
    import torch
    b, n = 2, 1024
    x, y = make_clouds("uniform", b, n, n, seed=23)
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    z = lambda dt=torch.float32: torch.zeros(b, n, device=cuda, dtype=dt)
    dist, ass, price, inv = z(), z(torch.int32) - 1, z(), z(torch.int32) - 1
    lib = pkg._lib.lib
    assert lib.psd_emd_forward(vp(tx), vp(ty), b, n, n, vp(dist), vp(ass), vp(price), vp(inv), vp(z(torch.int32)), vp(z()), vp(z()),
                               None, None, None, None, None, 0.05, 3000, None) == 1
    bounds = torch.zeros(b, 2, device=cuda, dtype=torch.float64)
    status = torch.zeros(b, device=cuda, dtype=torch.int32)
    assert lib.psd_emd_dual_bound(vp(tx), vp(ty), b, n, vp(ass), vp(price), vp(bounds), vp(status), None) == 1
    want, wstatus = dual_bound(x, y, ass.cpu().numpy(), price.cpu().numpy())
    assert np.array_equal(status.cpu().numpy(), wstatus)
    assert_close_bounds(bounds.cpu().numpy(), want)
    exact = exact_emd(x, y)
    assert_brackets(bounds.cpu().numpy(), exact, rel=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [None, 2, -2])
def test_gpu_certified_stays_in_bounds(pkg, cuda, cluster):
    import torch
    from test_gpu_guards import Arena
    b, n = 3, 1024
    x, y = make_clouds("clustered", b, n, n, seed=24)
    A = Arena(cuda)
    tx, ty = A.tensor(x), A.tensor(y)
    dist, ass, price = A.empty((b, n), fill=0.0), A.empty((b, n), torch.int32, fill=0), A.empty((b, n), fill=0.0)
    bounds, status = A.empty((b, 4)).view(torch.float64), A.empty((b,), torch.int32)
    lib = pkg._lib.lib
    args = (vp(tx), vp(ty), b, n, 0.05, 1e-4, 4.0, 20000, vp(dist), vp(ass), vp(price), vp(bounds), vp(status))
    rc = lib.psd_emd_certified(*args, None) if cluster is None else lib.psd_emd_certified_cluster(*args, cluster, None)
    assert rc == 1, pkg._lib.last_error()
    A.check(f"certified, cluster {cluster}")
    assert (status == 1).all()
    for nn in (1000, 4099):
        xs, ys = make_clouds("uniform", 2, nn, nn, seed=25)
        B = Arena(cuda)
        sx, sy = B.tensor(xs), B.tensor(ys)
        sa = B.tensor(np.tile(np.arange(nn, dtype=np.int32), (2, 1)))
        sp, sb, ss = B.tensor(np.ones((2, nn), np.float32)), B.empty((2, 4)).view(torch.float64), B.empty((2,), torch.int32)
        assert lib.psd_emd_dual_bound(vp(sx), vp(sy), 2, nn, vp(sa), vp(sp), vp(sb), vp(ss), None) == 1
        B.check(f"dual bound n={nn}")
    assert np.array_equal(tx.cpu().numpy(), x) and np.array_equal(ty.cpu().numpy(), y)


@pytest.mark.gpu
def test_gpu_gradients(pkg, oracle, cuda):
    """xyz1: the reference's gradient kernel through the assignment; xyz2: the mirrored term."""
    import torch
    c = case(oracle, "uniform", 2, 1024, 1e-4)
    x, y = c["x"], c["y"]
    tx = torch.from_numpy(x).to(cuda).requires_grad_(True)
    ty = torch.from_numpy(y).to(cuda).requires_grad_(True)
    dist, ass, bounds, status = pkg.emd_certified(tx, ty, eps_end=1e-4)
    w = np.random.default_rng(26).random((2, 1024), dtype=np.float32)
    (dist * torch.from_numpy(w).to(cuda)).sum().backward()
    a = ass.cpu().numpy()
    assert np.array_equal(a, c["ass"]) and (status.cpu().numpy() == 1).all()
    g1 = oracle.emd_backward(x, y, w, a)
    assert np.array_equal(tx.grad.cpu().numpy(), g1)
    g2 = np.zeros_like(y)
    for k in range(2):
        g2[k][a[k]] = -g1[k]
    assert np.array_equal(ty.grad.cpu().numpy(), g2)
    # the metric: the value of the matching and a gap that brackets the exact batch mean
    value, gap = pkg.certified_emd_distance(tx.detach(), ty.detach(), eps_end=1e-4)
    exact = exact_of(c).mean() * 100
    assert 0 <= gap <= 1e-4 * 100 and abs(value - exact) <= gap + 1e-5 * exact


@pytest.mark.gpu
def test_gpu_stream_and_graph_capture(pkg, oracle, cuda):
    import torch
    c = case(oracle, "uniform", 2, 1024, 1e-4)
    side = torch.cuda.Stream()
    ref = run_certified(pkg, cuda, c["x"], c["y"], 1e-4, stream=side)
    assert np.array_equal(ref[1], c["ass"])
    b, n = 2, 1024
    tx, ty = torch.from_numpy(c["x"]).to(cuda), torch.from_numpy(c["y"]).to(cuda)
    dist, ass, price = torch.empty(b, n, device=cuda), torch.empty(b, n, device=cuda, dtype=torch.int32), torch.empty(b, n, device=cuda)
    bounds, status = torch.empty(b, 2, device=cuda, dtype=torch.float64), torch.empty(b, device=cuda, dtype=torch.int32)
    lib = pkg._lib.lib
    call = lambda: lib.psd_emd_certified(vp(tx), vp(ty), b, n, 0.05, 1e-4, 4.0, 20000, vp(dist), vp(ass), vp(price), vp(bounds),
                                         vp(status), pkg._lib.stream_of(tx))
    assert call() == 1
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        assert call() == 1, pkg._lib.last_error()
    for t in (dist, price, bounds):
        t.fill_(float("nan"))
    ass.fill_(7)
    status.fill_(7)
    g.replay()
    torch.cuda.synchronize()
    got = [t.cpu().numpy() for t in (dist, ass, price, bounds, status)]
    for a, r in zip(got, ref):
        assert np.array_equal(a, r, equal_nan=a.dtype.kind == "f")
