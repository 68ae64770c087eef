"""Chamfer distance and F-score on ragged batches: psd_chamfer_forward_ragged / psd_chamfer_backward_ragged and the Python
``chamfer_ragged`` / ``chamfer_fscore_fused(..., x_lengths, y_lengths)``.

The reference for pair c is the library's own uniform launch on the pair's participating points alone, which the rest of the
suite pins to the CPU oracle bit for bit.  Pairs with the same lengths are run together in one uniform launch (every pair of a
uniform launch is computed on its own), and a few cases go to single-pair calls and to the oracle directly."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import make_clouds

vp = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
NAN_BITS = 0x7FC00000
KINDS = ["uniform", "clustered", "lattice", "dup", "offset"]


def test_host_lengths_are_checked_before_any_device_work(pkg):
    x, y = torch.rand(2, 5, 3), torch.rand(2, 7, 3)
    for xl, yl in (([0, 5], None), ([1, 6], None), (None, [7, 8]), (torch.tensor([1, 2, 3]), None), ([1.0, 2.0], None)):
        with pytest.raises(ValueError):
            pkg.chamfer_ragged(x, y, xl, yl)
        with pytest.raises(ValueError):
            pkg.chamfer_fscore_fused(x, y, x_lengths=xl, y_lengths=yl)
    with pytest.raises(RuntimeError, match="CUDA"):   # valid lengths: the CPU clouds are refused as by chamfer_3DDist
        pkg.chamfer_ragged(x, y, [5, 1], torch.tensor([7, 2]))


# ------------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------------------------------
def stream_ptr(cuda):
    return ctypes.c_void_p(torch.cuda.current_stream(cuda).cuda_stream)


def as_layout(a, bit, layout, cuda):
    """device tensor of the padded cloud a [b, k, 3] in the given layout (the raw [b, 3, k] tensor when transposed)"""
    t = torch.from_numpy(np.ascontiguousarray(a.transpose(0, 2, 1) if layout & bit else a)).to(cuda)
    return t


def ragged(lib, cuda, x, y, l1, l2, layout=0, thr=1e-3, zero=None):
    """one psd_chamfer_forward_ragged launch on numpy clouds; lengths None = NULL.  Returns numpy d1, d2, i1, i2, sums, cnt."""
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    tx, ty = as_layout(x, 1, layout, cuda), as_layout(y, 2, layout, cuda)
    tl1 = None if l1 is None else torch.as_tensor(np.asarray(l1, np.int32)).to(cuda)
    tl2 = None if l2 is None else torch.as_tensor(np.asarray(l2, np.int32)).to(cuda)
    d1, d2 = torch.full((b, n), 7.0, device=cuda), torch.full((b, m), 7.0, device=cuda)
    i1, i2 = torch.full((b, n), 7, device=cuda, dtype=torch.int32), torch.full((b, m), 7, device=cuda, dtype=torch.int32)
    sums, cnt = torch.zeros(b, 2, device=cuda), torch.zeros(b, 2, device=cuda, dtype=torch.int32)
    rc = lib.psd_chamfer_forward_ragged(vp(tx), vp(ty), b, n, m, layout, vp(tl1), vp(tl2), vp(d1), vp(d2), vp(i1), vp(i2),
                                        vp(sums), thr, vp(cnt), vp(zero), 0 if zero is None else zero.numel(), stream_ptr(cuda))
    assert rc == 1
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in (d1, d2, i1, i2, sums, cnt))


def uniform(lib, cuda, x, y):
    """psd_chamfer_forward_ex on contiguous numpy clouds [b, n, 3] / [b, m, 3]"""
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    tx, ty = torch.from_numpy(np.ascontiguousarray(x)).to(cuda), torch.from_numpy(np.ascontiguousarray(y)).to(cuda)
    d1, d2 = torch.empty(b, n, device=cuda), torch.empty(b, m, device=cuda)
    i1, i2 = torch.empty(b, n, device=cuda, dtype=torch.int32), torch.empty(b, m, device=cuda, dtype=torch.int32)
    assert lib.psd_chamfer_forward_ex(vp(tx), vp(ty), b, n, m, 0, vp(d1), vp(d2), vp(i1), vp(i2), None, 0.0, None, 0, -1,
                                      stream_ptr(cuda)) == 1
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in (d1, d2, i1, i2))


def per_pair_reference(lib, cuda, x, y, l1, l2):
    """{c: (d1, d2, i1, i2)} of uniform launches on each pair's participating points, pairs with equal lengths together"""
    groups = {}
    for c, (a, b) in enumerate(zip(l1, l2)):
        groups.setdefault((int(a), int(b)), []).append(c)
    out = {}
    for (a, b), cs in groups.items():
        r = uniform(lib, cuda, x[cs, :a], y[cs, :b])
        for k, c in enumerate(cs):
            out[c] = tuple(v[k] for v in r)
    return out


def assert_matches_pairs(got, ref, l1, l2, what=""):
    d1, d2, i1, i2 = got[:4]
    for c, (a, b) in enumerate(zip(l1, l2)):
        r1, r2, j1, j2 = ref[c]
        assert np.array_equal(d1[c, :a].view(np.int32), r1.view(np.int32)), f"{what} pair {c}: dist1 bits"
        assert np.array_equal(d2[c, :b].view(np.int32), r2.view(np.int32)), f"{what} pair {c}: dist2 bits"
        assert np.array_equal(i1[c, :a], j1) and np.array_equal(i2[c, :b], j2), f"{what} pair {c}: idx"
        assert (d1[c, a:] == 0).all() and (i1[c, a:] == -1).all(), f"{what} pair {c}: padding rows of dist1 / idx1"
        assert (d2[c, b:] == 0).all() and (i2[c, b:] == -1).all(), f"{what} pair {c}: padding rows of dist2 / idx2"


class variant:
    def __init__(self, lib, v):
        self.lib, self.v = lib, v

    def __enter__(self):
        self.old = self.lib.psd_chamfer_nn_variant(self.v)

    def __exit__(self, *a):
        self.lib.psd_chamfer_nn_variant(self.old)


def fallbacks(lib):
    out = np.zeros(2, np.int64)
    assert lib.psd_chamfer_stats(out.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), 1) == 1
    return int(out[1])


def lengths_for(pattern, b, n, m, rng):
    if pattern == "full":
        return np.full(b, n), np.full(b, m)
    if pattern == "ones":
        return np.ones(b, int), np.ones(b, int)
    if pattern == "one_vs_max":
        return np.where(np.arange(b) % 2 == 0, 1, n), np.where(np.arange(b) % 2 == 0, m, 1)
    l1, l2 = rng.integers(1, n + 1, b), rng.integers(1, m + 1, b)
    if pattern == "multitile":   # padded M > 2048, most pairs <= 2048 targets
        l2 = np.minimum(l2, 2048)
        l2[0] = m
    return l1, l2


PATTERNS = {   # pattern -> (b, n, m)
    "full": (5, 700, 1100),
    "ones": (6, 300, 260),
    "random": (9, 700, 1100),
    "one_vs_max": (4, 300, 4099),
    "multitile": (7, 900, 4099),
    "small": (8, 100, 128),
}


# ------------------------------------------------------------------------------------------------------------------------
# bits
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("var", [0, 1, 3])
@pytest.mark.parametrize("pattern", list(PATTERNS))
def test_pairs_equal_standalone_launches(pkg, cuda, var, pattern):
    lib = pkg._lib.lib
    b, n, m = PATTERNS[pattern]
    x, y = make_clouds("uniform", b, n, m, seed=11)
    l1, l2 = lengths_for("random" if pattern == "small" else pattern, b, n, m, np.random.default_rng(5))
    with variant(lib, var):
        got = ragged(lib, cuda, x, y, l1, l2)
        assert_matches_pairs(got, per_pair_reference(lib, cuda, x, y, l1, l2), l1, l2, pattern)
        if pattern == "multitile":   # single-pair calls of the pairs that run single-tile alone
            for c in range(b):
                r = uniform(lib, cuda, x[c:c + 1, :l1[c]], y[c:c + 1, :l2[c]])
                assert_matches_pairs(tuple(v[c:c + 1] for v in got[:4]), {0: tuple(v[0] for v in r)}, l1[c:c + 1], l2[c:c + 1])


@pytest.mark.gpu
@pytest.mark.parametrize("var", [0, 1, 3])
@pytest.mark.parametrize("layout", [0, 1, 2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_every_layout_and_cloud_kind(pkg, cuda, var, layout, kind):
    lib = pkg._lib.lib
    b, n, m = 6, 640, 2300
    x, y = make_clouds(kind, b, n, m, seed=3)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(layout))
    with variant(lib, var):
        got = ragged(lib, cuda, x, y, l1, l2, layout=layout)
        assert_matches_pairs(got, per_pair_reference(lib, cuda, x, y, l1, l2), l1, l2, f"{kind} layout {layout}")


@pytest.mark.gpu
@pytest.mark.parametrize("var", [1, 3])
def test_non_finite_participating_points_follow_the_512_tile_rule(pkg, cuda, var):
    lib = pkg._lib.lib
    b, n, m = 6, 700, 2600
    x, y = make_clouds("uniform", b, n, m, seed=4)
    l1, l2 = np.array([700, 513, 650, 1, 100, 600]), np.array([2600, 1500, 513, 1024, 2049, 900])
    y[0, 0, 1] = np.nan        # target 0: poisons every query of pair 0
    y[1, 600, 0] = np.inf      # inside the second 512-target tile
    y[2, 512, 2] = np.nan      # first target of the second tile
    x[3, 0, 0] = np.nan        # a NaN query
    y[4, 2048, 0] = -np.inf    # a second target tile in multi-tile mode
    x[5, 10] = np.inf
    with variant(lib, var):
        got = ragged(lib, cuda, x, y, l1, l2)
        assert_matches_pairs(got, per_pair_reference(lib, cuda, x, y, l1, l2), l1, l2, "non-finite")


@pytest.mark.gpu
def test_a_few_pairs_against_the_oracle(pkg, oracle, cuda):
    lib = pkg._lib.lib
    b, n, m = 4, 600, 2500
    x, y = make_clouds("lattice", b, n, m, seed=8)
    l1, l2 = np.array([600, 1, 333, 517]), np.array([2500, 77, 2048, 1])
    for var in (1, 3):
        with variant(lib, var):
            got = ragged(lib, cuda, x, y, l1, l2)
        for c in range(b):
            want = oracle.chamfer_forward(x[c:c + 1, :l1[c]], y[c:c + 1, :l2[c]], nthreads=4)
            for g, w, k in zip(got[:4], want, (l1[c], l2[c], l1[c], l2[c])):
                assert np.array_equal(g[c, :k], w[0]), f"variant {var} pair {c}"


@pytest.mark.gpu
def test_65535_tiny_pairs(pkg, cuda):
    lib = pkg._lib.lib
    b = 65535
    rng = np.random.default_rng(1)
    x, y = rng.random((b, 4, 3), dtype=np.float32), rng.random((b, 4, 3), dtype=np.float32)
    l1, l2 = rng.integers(1, 5, b), rng.integers(1, 5, b)
    for var in (0, 1, 3):
        with variant(lib, var):
            got = ragged(lib, cuda, x, y, l1, l2)
            ref = per_pair_reference(lib, cuda, x, y, l1, l2)
        assert_matches_pairs(got, ref, l1, l2, f"variant {var}")


# ------------------------------------------------------------------------------------------------------------------------
# padding, sums and counts
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("var", [1, 3])
@pytest.mark.parametrize("shape", [(6, 700, 1100), (5, 900, 4099)])
def test_padding_is_never_read(pkg, cuda, var, shape):
    lib = pkg._lib.lib
    b, n, m = shape
    x, y = make_clouds("clustered", b, n, m, seed=2)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(9))
    results = []
    for fill in (0.0, np.nan, np.inf, -np.inf, 1e30):
        xp, yp = x.copy(), y.copy()
        for c in range(b):
            xp[c, l1[c]:] = fill
            yp[c, l2[c]:] = fill
        with variant(lib, var):
            fallbacks(lib)
            r = ragged(lib, cuda, xp, yp, l1, l2, thr=5e-4)
            results.append((fill, r, fallbacks(lib)))
    (_, r0, fb0) = results[0]
    for fill, r, fb in results[1:]:
        for a, g in zip(r0[:4], r[:4]):
            assert np.array_equal(a.view(np.int32), g.view(np.int32)), f"padding {fill} changed an output"
        assert np.array_equal(r0[5], r[5]), f"padding {fill} changed fs_count"
        assert fb == fb0, f"padding {fill}: {fb} exact fallbacks against {fb0} with zero padding"
    for c in range(b):
        assert (r0[0][c, l1[c]:] == 0).all() and (r0[2][c, l1[c]:] == -1).all()
        assert (r0[1][c, l2[c]:] == 0).all() and (r0[3][c, l2[c]:] == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("var", [0, 1, 3])
@pytest.mark.parametrize("shape", [(8, 1000, 1024), (5, 900, 4099)])
def test_sums_counts_and_fscore(pkg, cuda, var, shape):
    lib = pkg._lib.lib
    b, n, m = shape
    x, y = make_clouds("uniform", b, n, m, seed=6)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(3))
    thr = 4e-4
    with variant(lib, var):
        d1, d2, i1, i2, sums, cnt = ragged(lib, cuda, x, y, l1, l2, thr=thr)
        ref = per_pair_reference(lib, cuda, x, y, l1, l2)
        for c in range(b):
            assert cnt[c, 0] == int((ref[c][0] < np.float32(thr)).sum()) and cnt[c, 1] == int((ref[c][1] < np.float32(thr)).sum())
            np.testing.assert_allclose(sums[c], [ref[c][0].astype(np.float64).sum(), ref[c][1].astype(np.float64).sum()], rtol=1e-5)
        tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
        for lens in ((l1.tolist(), l2.tolist()), (torch.tensor(l1).to(cuda), torch.tensor(l2, dtype=torch.int64).to(cuda))):
            r = pkg.chamfer_fscore_fused(tx, ty, thr, x_lengths=lens[0], y_lengths=lens[1])
            torch.cuda.synchronize()
            assert np.array_equal(r["counts"].cpu().numpy(), cnt)
            p1 = torch.from_numpy(cnt[:, 0]).float() / torch.from_numpy(l1).float()
            p2 = torch.from_numpy(cnt[:, 1]).float() / torch.from_numpy(l2).float()
            assert torch.equal(r["precision_1"].cpu(), p1) and torch.equal(r["precision_2"].cpu(), p2)
            want = sums[:, 0].astype(np.float64) / l1 + sums[:, 1].astype(np.float64) / l2
            np.testing.assert_allclose(r["chamfer"].cpu().numpy(), want, rtol=1e-5)
            np.testing.assert_array_equal(r["dist1"].cpu().numpy().view(np.int32), d1.view(np.int32))


# ------------------------------------------------------------------------------------------------------------------------
# gradients
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("transposed", [False, True])
@pytest.mark.parametrize("shape", [(6, 700, 1100), (4, 900, 4099), (8, 100, 128)])
def test_autograd_against_per_pair_chamfer_3DDist(pkg, cuda, transposed, shape):
    b, n, m = shape
    x, y = make_clouds("clustered", b, n, m, seed=12)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(b))
    rng = np.random.default_rng(7)
    g1 = torch.from_numpy(rng.random((b, n), dtype=np.float32)).to(cuda)   # nonzero on the padding rows too
    g2 = torch.from_numpy(rng.random((b, m), dtype=np.float32)).to(cuda)
    if transposed:
        xr = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).to(cuda).requires_grad_(True)
        xv = xr.transpose(2, 1)
    else:
        xr = torch.from_numpy(x).to(cuda).requires_grad_(True)
        xv = xr
    ty = torch.from_numpy(y).to(cuda).requires_grad_(True)
    d1, d2, i1, i2 = pkg.chamfer_ragged(xv, ty, torch.tensor(l1).to(cuda), l2.tolist())
    ((d1 * g1).sum() + (d2 * g2).sum()).backward()
    torch.cuda.synchronize()
    gx = xr.grad.transpose(2, 1) if transposed else xr.grad
    assert xr.grad.shape == xr.shape and ty.grad.shape == ty.shape
    for c in range(b):
        a, k = int(l1[c]), int(l2[c])
        px = torch.from_numpy(x[c:c + 1, :a]).to(cuda).requires_grad_(True)
        py = torch.from_numpy(y[c:c + 1, :k]).to(cuda).requires_grad_(True)
        e1, e2, j1, j2 = pkg.chamfer_3DDist()(px, py)
        ((e1 * g1[c:c + 1, :a]).sum() + (e2 * g2[c:c + 1, :k]).sum()).backward()
        assert torch.equal(d1[c, :a].view(torch.int32), e1[0].view(torch.int32)) and torch.equal(i2[c, :k], j2[0])
        torch.testing.assert_close(gx[c, :a], px.grad[0], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(ty.grad[c, :k], py.grad[0], rtol=1e-5, atol=1e-6)
        assert bool((gx[c, a:] == 0).all()) and bool((ty.grad[c, k:] == 0).all()), f"pair {c}: gradient past the lengths"


@pytest.mark.gpu
def test_both_lengths_none_is_chamfer_3DDist(pkg, cuda):
    x, y = make_clouds("uniform", 3, 300, 500, seed=1)
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    a, b = pkg.chamfer_ragged(tx, ty), pkg.chamfer_3DDist()(tx, ty)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    c = pkg.chamfer_ragged(tx, ty, [300, 300, 300], None)   # explicit full lengths: the same bits
    for u, v in zip(c, b):
        assert torch.equal(u, v)


# ------------------------------------------------------------------------------------------------------------------------
# invalid lengths, streams and graphs, guard zones
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("var", [1, 3])
@pytest.mark.parametrize("shape", [(5, 700, 1100), (5, 700, 4099)])
def test_invalid_device_lengths_make_only_their_pair_nan(pkg, cuda, var, shape):
    lib = pkg._lib.lib
    b, n, m = shape
    x, y = make_clouds("uniform", b, n, m, seed=21)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(4))
    with variant(lib, var):
        good = ragged(lib, cuda, x, y, l1, l2)
        for side, c, bad in ((0, 1, 0), (0, 3, n + 1), (1, 2, 0), (1, 4, m + 1), (0, 0, -5)):
            b1, b2 = l1.copy(), l2.copy()
            (b1 if side == 0 else b2)[c] = bad
            got = ragged(lib, cuda, x, y, b1, b2)
            for k in range(b):
                for i in (0, 1, 2, 3, 5):   # (sums are float atomics: their order is not fixed)
                    if k != c:
                        assert np.array_equal(got[i][k].view(np.int32), good[i][k].view(np.int32)), f"pair {k} changed by pair {c}"
            assert (got[0][c].view(np.int32) == NAN_BITS).all() and (got[1][c].view(np.int32) == NAN_BITS).all()
            assert (got[2][c] == -1).all() and (got[3][c] == -1).all()
            assert np.isnan(got[4][c]).all() and (got[5][c] == 0).all()
    # the gradient of an invalid pair is NaN, the others are finite and match the valid launch
    tx, ty = torch.from_numpy(x).to(cuda).requires_grad_(True), torch.from_numpy(y).to(cuda).requires_grad_(True)
    bl = torch.tensor(l1).to(cuda)
    bl[2] = n + 1
    d1, d2, _, _ = pkg.chamfer_ragged(tx, ty, bl, torch.tensor(l2).to(cuda))
    (d1.nan_to_num().sum() + d2.nan_to_num().sum()).backward()
    assert bool(torch.isnan(tx.grad[2]).all()) and bool(torch.isnan(ty.grad[2]).all())
    keep = [k for k in range(b) if k != 2]
    assert bool(torch.isfinite(tx.grad[keep]).all()) and bool(torch.isfinite(ty.grad[keep]).all())


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6, 700, 1100), (5, 900, 4099)])
def test_side_stream_and_graph_capture_give_the_same_bits(pkg, cuda, shape):
    lib = pkg._lib.lib
    b, n, m = shape
    x, y = make_clouds("uniform", b, n, m, seed=30)
    l1, l2 = lengths_for("random", b, n, m, np.random.default_rng(30))
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    tl1, tl2 = torch.tensor(l1, dtype=torch.int32).to(cuda), torch.tensor(l2, dtype=torch.int32).to(cuda)
    gd1 = torch.from_numpy(np.random.default_rng(1).random((b, n), dtype=np.float32)).to(cuda)
    gd2 = torch.from_numpy(np.random.default_rng(2).random((b, m), dtype=np.float32)).to(cuda)
    outs = [(torch.empty(b, n, device=cuda), torch.empty(b, m, device=cuda), torch.empty(b, n, device=cuda, dtype=torch.int32),
             torch.empty(b, m, device=cuda, dtype=torch.int32), torch.empty(3 * b * (n + m), device=cuda)) for _ in range(3)]

    def step(o):
        d1, d2, i1, i2, g = o
        sp = ctypes.c_void_p(torch.cuda.current_stream(cuda).cuda_stream)
        assert lib.psd_chamfer_forward_ragged(vp(tx), vp(ty), b, n, m, 0, vp(tl1), vp(tl2), vp(d1), vp(d2), vp(i1), vp(i2),
                                              None, 0.0, None, vp(g), g.numel(), sp) == 1
        assert lib.psd_chamfer_backward_ragged(vp(tx), vp(ty), vp(g[:3 * b * n]), vp(g[3 * b * n:]), vp(gd1), vp(gd2), vp(i1),
                                               vp(i2), vp(tl1), vp(tl2), b, n, m, 0, sp) == 1

    step(outs[0])
    side = torch.cuda.Stream(cuda)
    side.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(side):
        step(outs[1])
    torch.cuda.current_stream(cuda).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    cap = torch.cuda.Stream(cuda)
    cap.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(cap):
        with torch.cuda.graph(graph, stream=cap):
            step(outs[2])
    torch.cuda.current_stream(cuda).wait_stream(cap)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    for o in outs[1:]:
        for a, g in zip(outs[0][:4], o[:4]):
            assert torch.equal(a.view(torch.int32), g.view(torch.int32))
        torch.testing.assert_close(o[4], outs[0][4], rtol=1e-5, atol=1e-6)   # float atomics: order may differ
        ga = o[4][:3 * b * n].view(b, n, 3)
        for c in range(b):
            assert bool((ga[c, l1[c]:] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("variant_", [1, 3])
@pytest.mark.parametrize("shape", [(3, 257, 130), (2, 1, 700), (2, 2049, 4099)])
@pytest.mark.parametrize("layout", [0, 1, 2, 3])
def test_entry_points_stay_in_bounds(pkg, cuda, variant_, shape, layout):
    from test_gpu_guards import Arena
    lib = pkg._lib.lib
    b, n, m = shape
    x, y = make_clouds("uniform", b, n, m, seed=3)
    rng = np.random.default_rng(layout)
    l1, l2 = rng.integers(1, n + 1, b).astype(np.int32), rng.integers(1, m + 1, b).astype(np.int32)
    l2[-1] = m
    A = Arena(cuda)
    tx = A.tensor(np.ascontiguousarray(x.transpose(0, 2, 1)) if layout & 1 else x)
    ty = A.tensor(np.ascontiguousarray(y.transpose(0, 2, 1)) if layout & 2 else y)
    tl1, tl2 = A.tensor(l1), A.tensor(l2)
    d1, d2 = A.empty((b, n)), A.empty((b, m))
    i1, i2 = A.empty((b, n), torch.int32), A.empty((b, m), torch.int32)
    sums, cnt = A.empty((b, 2), fill=0.0), A.empty((b, 2), torch.int32, fill=0)
    grads = A.empty((3 * b * (n + m),), fill=float("nan"))
    gd1 = A.tensor(np.random.default_rng(1).random((b, n), dtype=np.float32))
    gd2 = A.tensor(np.random.default_rng(2).random((b, m), dtype=np.float32))
    before = [t.clone() for t in (tx, ty, tl1, tl2, gd1, gd2)]
    with variant(lib, variant_):
        assert lib.psd_chamfer_forward_ragged(vp(tx), vp(ty), b, n, m, layout, vp(tl1), vp(tl2), vp(d1), vp(d2), vp(i1), vp(i2),
                                              vp(sums), 1e-3, vp(cnt), vp(grads), grads.numel(), None) == 1
        A.check("forward_ragged")
        assert float(grads.abs().sum()) == 0.0
        assert lib.psd_chamfer_backward_ragged(vp(tx), vp(ty), vp(grads[:3 * b * n]), vp(grads[3 * b * n:]), vp(gd1), vp(gd2),
                                               vp(i1), vp(i2), vp(tl1), vp(tl2), b, n, m, layout, None) == 1
        A.check("backward_ragged")
    for t, o in zip((tx, ty, tl1, tl2, gd1, gd2), before):
        assert torch.equal(t.view(torch.int32), o.view(torch.int32)), "an input was modified"
    assert lib.psd_chamfer_forward_ragged(vp(tx), vp(ty), b, n, m, 4, None, None, vp(d1), vp(d2), vp(i1), vp(i2), None, 0.0,
                                          None, None, 0, None) == -1
    assert lib.psd_chamfer_backward_ragged(vp(tx), vp(ty), vp(grads), vp(grads), vp(gd1), vp(gd2), vp(i1), vp(i2), None, None,
                                           b, n, m, -1, None) == -1
