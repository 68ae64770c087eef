"""Batched ICP on ragged batches: psd_icp_batch_ragged and the Python ``icp_ragged``.

A sample whose source and destination lengths are equal must give the bits of ``icp_batch`` on its participating points
alone (which tests/test_icp.py pins to the reference).  Samples of unequal sizes are compared with ``icp_unequal`` below,
the reference's icp() without its shape assert, built from the oracle's own NN and best_fit_transform; it equals
``oracle.icp`` bit for bit at equal sizes and is checked against an independent restatement (scipy's KD-tree and numpy's
SVD) at unequal ones.  Tolerances of tests/test_icp.py: iterations exact, distances 1e-12, transforms 1e-9."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import make_clouds

T_TOL, D_TOL = 1e-9, 1e-12
KINDS = ["uniform", "clustered", "lattice", "dup", "offset"]


def rot(axis, th):
    axis = np.asarray(axis, dtype=np.float64)
    axis /= np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def moved_copies(rng, B, k, dtype):
    """rotated, shifted, slightly noisy and permuted copies of the first k points of B [batch, *, 3]"""
    A = np.empty((B.shape[0], k, 3), dtype)
    for s in range(B.shape[0]):
        R = rot(rng.standard_normal(3), 0.05 + 0.1 * rng.random())
        P = B[s, :k].astype(np.float64)
        A[s] = ((P - P.mean(0)) @ R.T + P.mean(0) + 0.02 * rng.standard_normal(3) + 0.003 * rng.standard_normal((k, 3)))[rng.permutation(k)]
    return A


def icp_unequal(oracle, A, B, init_pose=None, max_iterations=20, tolerance=0.001):
    """utils/icp.py:68-118 (oracle.icp) without its shape assert: a source A [N, 3] and a destination B [M, 3] of any sizes.
    The algorithm needs none: the NN query takes any destination, best_fit_transform(src, dst[indices]) gets matched shapes,
    and the final best_fit_transform(A, src) compares A with its own moved copy."""
    A = np.asarray(A)
    B = np.asarray(B)
    assert A.ndim == 2 and A.shape[1] == 3 and B.ndim == 2 and B.shape[1] == 3
    m = A.shape[1]
    src = np.ones((m + 1, A.shape[0]))
    dst = np.ones((m + 1, B.shape[0]))
    src[:m, :] = np.copy(A.T)
    dst[:m, :] = np.copy(B.T)
    if init_pose is not None:
        src = np.dot(init_pose, src)
    prev_error = 0
    for i in range(max_iterations):
        distances, indices = oracle.icp_nearest_neighbor(src[:m, :].T, dst[:m, :].T)
        T, _, _ = oracle.icp_best_fit_transform(src[:m, :].T, dst[:m, indices].T)
        src = np.dot(T, src)
        mean_error = np.mean(distances)
        if np.abs(prev_error - mean_error) < tolerance:
            break
        prev_error = mean_error
    T, _, _ = oracle.icp_best_fit_transform(A, src[:m, :].T)
    return T, distances, i


POSE = np.array([[0.99500417, -0.09983342, 0.0, 0.05], [0.09983342, 0.99500417, 0.0, -0.02], [0.0, 0.0, 1.0, 0.01],
                 [0.0, 0.0, 0.0, 1.0]])


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the oracle and the host-side checks
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("pose", [None, POSE])
def test_icp_unequal_is_the_oracle_at_equal_sizes(oracle, dtype, pose):
    rng = np.random.default_rng(1)
    B = rng.random((1, 300, 3)).astype(dtype)
    A = moved_copies(rng, B, 300, dtype)[0]
    want = oracle.icp(A, B[0], init_pose=pose, max_iterations=60, tolerance=1e-10)
    got = icp_unequal(oracle, A, B[0], init_pose=pose, max_iterations=60, tolerance=1e-10)
    assert got[2] == want[2] and np.array_equal(got[1], want[1]) and np.array_equal(got[0], want[0])
    with pytest.raises(AssertionError):
        oracle.icp(A, B[0, :299])
    with pytest.raises(AssertionError):
        icp_unequal(oracle, A[:, :2], B[0])


def independent_icp(A, B, max_iterations, tolerance):
    """utils/icp.py:68-118 restated with scipy's KD-tree for the NN and numpy's SVD with the reflection rule (:32-35)"""
    from scipy.spatial import cKDTree
    tree = cKDTree(np.asarray(B, np.float64))

    def fit(P, Q):
        cP, cQ = P.mean(axis=0), Q.mean(axis=0)
        U, _, Vt = np.linalg.svd((P - cP).T @ (Q - cQ))
        R = Vt.T @ U.T
        if np.linalg.det(R) < 0:
            Vt[2, :] *= -1
            R = Vt.T @ U.T
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = R, cQ - R @ cP
        return T

    src = np.asarray(A, np.float64).copy()
    prev = 0.0
    for i in range(max_iterations):
        d, idx = tree.query(src)
        T = fit(src, np.asarray(B, np.float64)[idx])
        src = src @ T[:3, :3].T + T[:3, 3]
        if abs(prev - d.mean()) < tolerance:
            break
        prev = d.mean()
    return fit(np.asarray(A), src), d, i


@pytest.mark.parametrize("na,nb", [(256, 1500), (1200, 64), (700, 701)])
def test_icp_unequal_matches_an_independent_restatement(oracle, na, nb):
    rng = np.random.default_rng(na + nb)
    B = rng.random((1, max(na, nb), 3))
    src = B if na <= nb else rng.random((1, na, 3))
    A = moved_copies(rng, src, na, np.float64)[0]
    T, d, i = icp_unequal(oracle, A, B[0, :nb], max_iterations=80, tolerance=1e-10)
    wT, wd, wi = independent_icp(A, B[0, :nb], 80, 1e-10)
    assert i == wi and 3 < i < 79
    assert np.abs(d - wd).max() <= 1e-12
    assert np.abs(T - wT).max() <= 1e-12


def test_host_errors_raise_before_any_device_work(pkg):
    A, B = np.zeros((2, 5, 3), np.float32), np.zeros((2, 7, 3), np.float32)
    f = pkg.icp_ragged
    for la, lb in (([0, 5], None), ([1, 6], None), (None, [7, 8]), (None, [0, 1]), (torch.tensor([1, 2, 3]), None),
                   ([1.0, 2.0], None), (torch.tensor([5, 6]), None)):
        with pytest.raises(ValueError):
            f(A, B, la, lb)
    with pytest.raises(ValueError):
        f(A, B, max_iterations=0)
    with pytest.raises(ValueError):
        f(np.zeros((1, 4097, 3)), np.zeros((1, 10, 3)))              # n > 4096
    with pytest.raises(ValueError):
        f(np.zeros((1, 4000, 3)), np.zeros((1, 4193, 3)))            # n + m > 8192
    with pytest.raises(ValueError):
        f(np.zeros((2, 5, 3)), np.zeros((3, 5, 3)))                  # batch sizes differ
    with pytest.raises(ValueError):
        f(np.zeros((2, 5, 2)), np.zeros((2, 5, 2)))                  # not 3-D
    with pytest.raises(ValueError):
        f(np.zeros((2, 0, 3)), np.zeros((2, 5, 3)))                  # empty padded source


# ------------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------------------------------
def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def run_ragged(pkg, A, B, la, lb, cuda, pose=None, iters=40, tol=1e-9, lengths_on_device=True):
    dev_len = lambda l: None if l is None else (torch.as_tensor(np.asarray(l, np.int32)).to(cuda) if lengths_on_device else list(l))
    T, d, it = pkg.icp_ragged(torch.from_numpy(A).to(cuda), torch.from_numpy(B).to(cuda), dev_len(la), dev_len(lb), init_pose=pose,
                              max_iterations=iters, tolerance=tol)
    torch.cuda.synchronize()
    return T.cpu().numpy(), d.cpu().numpy(), it.cpu().numpy()


def standalone(pkg, A, B, lens, cuda, pose=None, iters=40, tol=1e-9):
    """{s: (T, d, it)} of icp_batch on each sample's first lens[s] points of A and B, samples of equal length together
    (every sample of a uniform launch is computed on its own)"""
    groups = {}
    for s, k in enumerate(lens):
        groups.setdefault(int(k), []).append(s)
    out = {}
    for k, ss in groups.items():
        T, d, it = pkg.icp.icp_batch(torch.from_numpy(np.ascontiguousarray(A[ss, :k])).to(cuda),
                                     torch.from_numpy(np.ascontiguousarray(B[ss, :k])).to(cuda), pose, iters, tol)
        T, d, it = T.cpu().numpy(), d.cpu().numpy(), it.cpu().numpy()
        for j, s in enumerate(ss):
            out[s] = (T[j], d[j], it[j])
    return out


def assert_bit_identical(pkg, A, B, lens, cuda, pose=None, iters=40, tol=1e-9):
    T, d, it = run_ragged(pkg, A, B, lens, lens, cuda, pose, iters, tol)
    ref = standalone(pkg, A, B, lens, cuda, pose, iters, tol)
    for s, k in enumerate(lens):
        wT, wd, wi = ref[s]
        assert it[s] == wi, f"sample {s} (length {k}): {it[s]} iterations, standalone {wi}"
        assert np.array_equal(bits(T[s]), bits(wT)), f"sample {s} (length {k}): T differs"
        assert np.array_equal(bits(d[s, :k]), bits(wd)), f"sample {s} (length {k}): distances differ"
        assert not d[s, k:].any(), f"sample {s}: distances past the length are not 0"
    return T, d, it


# ------------------------------------------------------------------------------------------------------------------------
# bit identity with icp_batch when a sample's two lengths are equal
# ------------------------------------------------------------------------------------------------------------------------
LENGTHS = {
    "full": (700, 700, lambda rng, b: [700] * b),
    "ones": (700, 900, lambda rng, b: [1] * b),
    "random": (1100, 1500, lambda rng, b: list(rng.integers(1, 1101, size=b))),
    "edges512": (1030, 1030, lambda rng, b: [511, 512, 513, 1, 1024, 1025, 1030][:b]),
    "edges4096": (4096, 4096, lambda rng, b: [4095, 4096, 2048, 3][:b]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("pose", [None, POSE], ids=["nopose", "pose"])
@pytest.mark.parametrize("pattern", list(LENGTHS))
def test_equal_lengths_give_the_bits_of_icp_batch(pkg, cuda, dtype, pose, pattern):
    n, m, draw = LENGTHS[pattern]
    rng = np.random.default_rng(len(pattern) * 7 + (pose is None))
    b = 4 if pattern == "edges4096" else 7
    lens = [int(k) for k in draw(rng, b)]
    B = rng.random((b, m, 3)).astype(dtype)
    A = np.zeros((b, n, 3), dtype)
    A[:, :] = moved_copies(rng, B, n, dtype)
    iters = 12 if pattern == "edges4096" else 40
    assert_bit_identical(pkg, A, B, lens, cuda, pose, iters)


@pytest.mark.gpu
def test_a_batch_of_4096_small_samples(pkg, cuda):
    rng = np.random.default_rng(5)
    b, n = 4096, 9
    lens = [int(k) for k in rng.integers(1, n + 1, size=b)]
    B = rng.random((b, n, 3)).astype(np.float32)
    A = moved_copies(rng, B, n, np.float32)
    _, _, it = assert_bit_identical(pkg, A, B, lens, cuda, iters=30, tol=1e-12)
    assert it.max() > 3


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_every_cloud_kind(pkg, cuda, kind):
    x, y = make_clouds(kind, 5, 1300, 1300, seed=11)
    rng = np.random.default_rng(12)
    lens = [1300, 1, 777, 1024, 513]
    A = np.concatenate([x[:2], moved_copies(rng, y[2:], 1300, np.float32)])   # unrelated clouds and rotated copies
    assert_bit_identical(pkg, A, y, lens, cuda, iters=30)


@pytest.mark.gpu
def test_reflection_planar_and_coincident_samples(pkg, cuda):
    rng = np.random.default_rng(11)
    n = 300
    B = rng.random((5, n, 3))
    A = np.empty_like(B)
    A[0] = B[0] * np.array([1.0, 1.0, -1.0]) + 0.1                       # mirrored: the optimum is a reflection
    B[1, :, 2] = 0.25                                                    # planar cloud (rank-2 H)
    A[1] = (B[1] - 0.5) @ rot([0, 0, 1], 0.4).T + 0.5
    A[2] = B[2]                                                          # identical clouds: stops in iteration 0
    A[3] = np.full((n, 3), 0.3); B[3] = np.full((n, 3), 0.7)             # coincident points: H = 0
    A[4] = rng.random((n, 3)); B[4] = rng.random((n, 3))
    lens = [300, 300, 299, 300, 150]
    for dtype in (np.float32, np.float64):
        T, d, it = assert_bit_identical(pkg, A.astype(dtype), B.astype(dtype), lens, cuda, iters=30, tol=1e-10)
        assert it[2] == 0 and d[2].max() == 0.0


# ------------------------------------------------------------------------------------------------------------------------
# unequal sizes against the oracle
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,m,la,lb", [
    (256, 7936, [256, 200, 256], [7936, 5000, 300]),        # source << destination
    (4096, 64, [4096, 3000, 64], [64, 50, 8]),             # source >> destination
    (3000, 5192, [3000, 1000, 2999], [5192, 5192, 4000]),  # n + m = 8192
])
def test_unequal_sizes_match_the_oracle(pkg, oracle, cuda, dtype, n, m, la, lb):
    rng = np.random.default_rng(n + m)
    b = len(la)
    B = rng.random((b, m, 3)).astype(dtype)
    A = rng.random((b, n, 3)).astype(dtype)
    for s in range(b):                                      # sources near their destination where they fit inside it
        k = min(la[s], lb[s])
        A[s, :k] = moved_copies(rng, B[s:s + 1], k, dtype)[0]
    iters = 25
    T, d, it = run_ragged(pkg, A, B, la, lb, cuda, iters=iters, tol=1e-9)
    for s in range(b):
        wT, wd, wi = icp_unequal(oracle, A[s, :la[s]], B[s, :lb[s]], max_iterations=iters, tolerance=1e-9)
        assert it[s] == wi, f"sample {s}: {it[s]} iterations, oracle {wi}"
        assert np.abs(d[s, :la[s]] - wd).max() <= D_TOL
        assert not d[s, la[s]:].any()
        assert np.abs(T[s] - wT).max() <= T_TOL


@pytest.mark.gpu
def test_host_lengths_and_null_lengths(pkg, cuda):
    """list lengths give the bits of CUDA lengths, and lengths equal to the padded sizes those of NULL lengths"""
    rng = np.random.default_rng(21)
    A, B = rng.random((3, 500, 3)), rng.random((3, 800, 3))
    la, lb = [500, 17, 333], [800, 800, 2]
    dev = run_ragged(pkg, A, B, la, lb, cuda)
    host = run_ragged(pkg, A, B, la, lb, cuda, lengths_on_device=False)
    for x, y in zip(dev, host):
        assert np.array_equal(bits(x), bits(y))
    full = run_ragged(pkg, A, B, [500] * 3, [800] * 3, cuda)
    null = run_ragged(pkg, A, B, None, None, cuda)
    for x, y in zip(full, null):
        assert np.array_equal(bits(x), bits(y))


# ------------------------------------------------------------------------------------------------------------------------
# padding, invalid lengths, streams and graphs, guard zones
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_padding_values_do_not_change_any_bit(pkg, cuda, dtype):
    rng = np.random.default_rng(31)
    n, m = 900, 1200
    la, lb = [900, 400, 1, 650], [1200, 700, 5, 650]
    B = rng.random((4, m, 3)).astype(dtype)
    A = moved_copies(rng, B, n, dtype)
    outs = []
    for pad in (0.0, np.nan, np.inf, -np.inf, 1e30):
        Ap, Bp = A.copy(), B.copy()
        for s in range(4):
            Ap[s, la[s]:] = pad
            Bp[s, lb[s]:] = pad
        outs.append(run_ragged(pkg, Ap, Bp, la, lb, cuda))
    for o in outs[1:]:
        for x, y in zip(outs[0], o):
            assert np.array_equal(bits(x), bits(y))
    T, d, it = outs[0]
    assert np.isfinite(T).all() and (it >= 0).all()
    for s in range(4):
        assert not d[s, la[s]:].any()


@pytest.mark.gpu
def test_invalid_lengths_touch_only_their_sample(pkg, cuda):
    rng = np.random.default_rng(41)
    n, m = 600, 700
    A, B = rng.random((6, n, 3)).astype(np.float32), rng.random((6, m, 3)).astype(np.float32)
    la, lb = [600, 300, 10, 600, 599, 1], [700, 300, 10, 700, 1, 700]
    good = run_ragged(pkg, A, B, la, lb, cuda)
    bad_a, bad_b = list(la), list(lb)
    bad_a[1], bad_b[2], bad_a[3], bad_b[4] = 0, -1, n + 1, m + 1
    T, d, it = run_ragged(pkg, A, B, bad_a, bad_b, cuda)
    for s in range(6):
        if s in (1, 2, 3, 4):
            assert np.isnan(T[s]).all() and np.isnan(d[s]).all() and it[s] == -1
        else:
            assert np.array_equal(bits(T[s]), bits(good[0][s])) and np.array_equal(bits(d[s]), bits(good[1][s]))
            assert it[s] == good[2][s]


@pytest.mark.gpu
def test_side_stream_and_graph_capture_give_the_same_bits(pkg, cuda):
    rng = np.random.default_rng(51)
    n, m = 1500, 1100
    tb = torch.from_numpy(rng.random((5, m, 3)).astype(np.float32)).to(cuda)
    ta = torch.from_numpy(moved_copies(rng, rng.random((5, n, 3)), n, np.float32)).to(cuda)
    la = torch.tensor([1500, 20, 1100, 513, 1], dtype=torch.int32, device=cuda)
    lb = torch.tensor([1100, 1100, 1100, 513, 2], dtype=torch.int32, device=cuda)
    step = lambda: pkg.icp_ragged(ta, tb, la, lb, max_iterations=30, tolerance=1e-9)
    base = [t.clone() for t in step()]
    side = torch.cuda.Stream(cuda)
    side.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(side):
        on_side = step()
    torch.cuda.current_stream(cuda).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    cap = torch.cuda.Stream(cuda)
    cap.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(cap):
        with torch.cuda.graph(graph, stream=cap):
            captured = step()
    torch.cuda.current_stream(cuda).wait_stream(cap)
    for t in captured:
        t.fill_(-7)
    graph.replay()
    torch.cuda.synchronize()
    for o in (on_side, captured):
        for x, y in zip(base, o):
            assert torch.equal(x.view(torch.int64) if x.dtype == torch.float64 else x,
                               y.view(torch.int64) if y.dtype == torch.float64 else y)


G = 2048            # guard words (4 bytes) on each side
SENT = 0x7FC0DEAD   # a NaN pattern as float32, an unmistakable value as int32


class Arena:
    """every tensor carved out of a larger sentinel-filled allocation, as in tests/test_gpu_guards.py"""

    def __init__(self, dev):
        self.dev, self.items = dev, []

    def _new(self, numel, dtype):
        words = numel * torch.empty((), dtype=dtype).element_size() // 4
        raw = torch.full((words + 2 * G,), SENT, dtype=torch.int32, device=self.dev)
        self.items.append((raw, words))
        return raw[G:G + words].view(dtype)

    def tensor(self, src):
        t = torch.as_tensor(src)
        out = self._new(t.numel(), t.dtype)
        out.copy_(t.reshape(-1).to(self.dev))
        return out.view(t.shape)

    def empty(self, shape, dtype):
        return self._new(int(np.prod(shape)), dtype).view(shape)

    def check(self, what):
        torch.cuda.synchronize()
        for raw, words in self.items:
            assert bool((raw[:G] == SENT).all()) and bool((raw[G + words:] == SENT).all()), f"{what}: a guard zone was written"


@pytest.mark.gpu
@pytest.mark.parametrize("in_f64", [0, 1])
def test_ragged_entry_point_stays_in_bounds(pkg, cuda, in_f64):
    lib = pkg._lib.lib
    vp = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
    dtype = np.float64 if in_f64 else np.float32
    rng = np.random.default_rng(61)
    b, n, m = 5, 333, 1030
    a_np, b_np = rng.random((b, n, 3)).astype(dtype), rng.random((b, m, 3)).astype(dtype)
    A = Arena(cuda)
    ta, tb = A.tensor(a_np), A.tensor(b_np)
    la, lb = A.tensor(np.array([333, 1, 200, 0, 333], np.int32)), A.tensor(np.array([1030, 1030, 7, 5, 1031], np.int32))
    pose = A.tensor(POSE)
    T, d, it = A.empty((b, 4, 4), torch.float64), A.empty((b, n), torch.float64), A.empty((b,), torch.int32)
    for lens in ((la, lb), (None, None)):
        assert lib.psd_icp_batch_ragged(vp(ta), vp(tb), in_f64, b, n, m, vp(lens[0]), vp(lens[1]), vp(pose), 9, 1e-9, vp(T), vp(d),
                                        vp(it), None) == 1
        A.check("psd_icp_batch_ragged")
    assert np.array_equal(ta.cpu().numpy(), a_np) and np.array_equal(tb.cpu().numpy(), b_np), "an input was modified"
    for args in ((b, 4097, 10, 5), (b, 4000, 4193, 5), (b, 0, 5, 5), (b, 5, 0, 5), (-1, 5, 5, 5), (b, 5, 5, 0)):
        bb, nn, mm, iters = args
        assert lib.psd_icp_batch_ragged(vp(ta), vp(tb), in_f64, bb, nn, mm, None, None, None, iters, 1e-9, vp(T), vp(d), vp(it),
                                        None) == -1
    A.check("argument errors")


# ------------------------------------------------------------------------------------------------------------------------
# end to end: pack_clouds -> icp_ragged -> apply T -> chamfer_fscore_fused with lengths
# ------------------------------------------------------------------------------------------------------------------------
def apply(T, P):
    """R p + t for T [..., 4, 4] fp64 and P [..., k, 3], elementwise (the same rounding batched and per sample)"""
    P = P.double()
    R, t = T[..., None, :3, :3], T[..., None, :3, 3]
    return P[..., 0:1] * R[..., :, 0] + P[..., 1:2] * R[..., :, 1] + P[..., 2:3] * R[..., :, 2] + t


@pytest.mark.gpu
def test_eval_chain_matches_the_per_sample_loop(pkg, cuda):
    rng = np.random.default_rng(71)
    sizes = [500, 1024, 1700, 2600, 4000, 1024]
    preds = torch.from_numpy(rng.random((len(sizes), 1024, 3)).astype(np.float32)).to(cuda)
    scans = [torch.from_numpy(moved_copies(rng, rng.random((1, k, 3)).astype(np.float32), k, np.float32)[0]).to(cuda)
             for k in sizes]
    gt, lengths = pkg.pack_clouds(scans)
    T, _, it = pkg.icp_ragged(gt, preds, lengths, tolerance=1e-10, max_iterations=60)
    aligned = apply(T, gt).float()
    r = pkg.chamfer_fscore_fused(aligned, preds, 0.001, x_lengths=lengths)
    for s, scan in enumerate(scans):
        Ts, _, its = pkg.icp_ragged(scan[None], preds[s:s + 1], tolerance=1e-10, max_iterations=60)
        assert int(its[0]) == int(it[s])
        assert torch.equal(Ts[0].view(torch.int64), T[s].view(torch.int64))
        if scan.shape[0] == 1024:
            Tu, _, _ = pkg.icp.icp_batch(scan[None], preds[s:s + 1], tolerance=1e-10, max_iterations=60)
            assert torch.equal(Tu[0].view(torch.int64), T[s].view(torch.int64))
        rs = pkg.chamfer_fscore_fused(apply(Ts[0], scan).float()[None], preds[s:s + 1], 0.001)
        k = scan.shape[0]
        assert torch.equal(rs["dist1"][0], r["dist1"][s, :k]) and torch.equal(rs["dist2"][0], r["dist2"][s])
        assert torch.equal(rs["counts"][0], r["counts"][s])
        for key in ("fscore", "precision_1", "precision_2", "chamfer"):   # fp32 divisions and sums, rounded differently
            assert torch.allclose(rs[key][0], r[key][s], rtol=1e-5, atol=0), key
