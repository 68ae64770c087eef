"""Drop-in for utils/icp.py: ``best_fit_transform(A, B)``, ``nearest_neighbor(src, dst)`` and
``icp(A, B, init_pose=None, max_iterations=20, tolerance=0.001)`` with the reference's signatures, numpy in / numpy out, plus
``icp_batch`` which aligns a whole batch of samples in one kernel launch (the reference's callers loop over the samples,
testnet.py:62-64), and ``icp_ragged`` for a batch whose samples have their own source and destination sizes.

The reference runs a sklearn KD-tree build + query, numpy reductions and a 3x3 SVD per iteration on the CPU; here the whole
iteration loop of every sample runs inside one CUDA kernel (csrc/icp.cu, psd_icp_batch), in fp64 like numpy.  There is no
CPU fallback."""
import ctypes

import numpy as np
import torch

try:
    from . import _lib
    from .sinkhorn import _lengths
except ImportError:
    import _lib
    from sinkhorn import _lengths

MAX_POINTS = 4096         # source points of one sample (padded N)
MAX_POINTS_PAIR = 8192    # source + destination points of one sample (padded N + M)


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("icp needs a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def _to_dev(x, dev):
    """[..., n, 3] numpy / torch input -> contiguous device tensor, float32 kept (exact in fp64), everything else float64."""
    t = torch.as_tensor(x)
    t = t.to(dev, torch.float32 if t.dtype == torch.float32 else torch.float64)
    return t.contiguous()


def icp_batch(A, B, init_pose=None, max_iterations=20, tolerance=0.001):
    """icp() for every sample of A, B [batch, n, 3] (numpy or torch, float32 or float64; both must share the dtype).
    Returns (T [batch,4,4] float64, distances [batch,n] float64, iterations [batch] int32) as torch tensors on the device."""
    dev = A.device if isinstance(A, torch.Tensor) and A.is_cuda else _device()
    a, b = _to_dev(A, dev), _to_dev(B, dev)
    assert a.shape == b.shape and a.dim() == 3 and a.shape[2] == 3, "A and B must both be [batch, n, 3]"
    if a.dtype != b.dtype:
        a, b = a.double(), b.double()
    batch, n, _ = a.shape
    pose = None if init_pose is None else torch.as_tensor(np.asarray(init_pose, dtype=np.float64)).to(dev).contiguous()
    if pose is not None:
        assert pose.shape == (4, 4)
    T = torch.empty(batch, 4, 4, device=dev, dtype=torch.float64)
    dist = torch.empty(batch, n, device=dev, dtype=torch.float64)
    iters = torch.zeros(batch, device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        rc = _lib.lib.psd_icp_batch(_lib.ptr(a), _lib.ptr(b), int(a.dtype == torch.float64), batch, n,
                                    None if pose is None else _lib.ptr(pose), int(max_iterations), ctypes.c_double(tolerance),
                                    _lib.ptr(T), _lib.ptr(dist), _lib.ptr(iters), _lib.stream_of(a))
    _lib.raise_on_cuda_error(rc, "psd_icp_batch")
    return T, dist, iters


def icp_ragged(A, B, a_lengths=None, b_lengths=None, init_pose=None, max_iterations=20, tolerance=0.001):
    """icp() for every sample of a ragged batch, in one launch: sample s aligns its first a_lengths[s] source points A[s] to
    its first b_lengths[s] destination points B[s].  The two sizes need not be equal: the reference's algorithm is defined
    for any sizes, only its ``assert A.shape == B.shape`` forbids them.

    A [batch, N, 3] and B [batch, M, 3] are padded (numpy or torch, float32 or float64; mixed dtypes are promoted to
    float64), with N <= 4096 and N + M <= 8192; a_lengths / b_lengths [batch] default to N / M.  Rows past the lengths are
    never read.  A list or CPU tensor of lengths is checked here (ValueError unless every length is in [1, N] / [1, M]); a
    CUDA integer tensor is used as it is, and a sample with a length out of range gets T all NaN, NaN distances and
    iteration -1 without affecting the others.  max_iterations must be >= 1.

    Returns (T [batch,4,4] float64, distances [batch,N] float64, iterations [batch] int32) on the device: T maps the source
    onto the destination, distances are those of the last NN pass (0 past a_lengths[s]).  A sample with equal lengths gets
    the bits ``icp_batch`` gives on its points alone.

    The evaluation of scans of different sizes against fixed-size predictions, with the ground truth as the moving source
    as in testnet.py:57-64, then runs in two launches::

        gt, lengths = pack_clouds(scans)                          # [B, max k, 3], [B]
        T, _, _ = icp_ragged(gt, preds, lengths, tolerance=1e-10, max_iterations=1024)
        aligned = gt.double() @ T[:, :3, :3].transpose(1, 2) + T[:, None, :3, 3]
        r = chamfer_fscore_fused(aligned.float(), preds, x_lengths=lengths)
    """
    a, b = torch.as_tensor(A), torch.as_tensor(B)
    if a.dim() != 3 or a.shape[2] != 3 or b.dim() != 3 or b.shape[2] != 3 or a.shape[0] != b.shape[0]:
        raise ValueError(f"A and B must be [batch, N, 3] and [batch, M, 3], got {tuple(a.shape)} and {tuple(b.shape)}")
    batch, n, m = a.shape[0], a.shape[1], b.shape[1]
    if n < 1 or m < 1 or n > MAX_POINTS or n + m > MAX_POINTS_PAIR:
        raise ValueError(f"icp_ragged needs 1 <= N <= {MAX_POINTS} and N + M <= {MAX_POINTS_PAIR}, got N = {n}, M = {m}")
    if max_iterations < 1:
        raise ValueError("icp_ragged needs max_iterations >= 1")
    la = None if a_lengths is None else _lengths("a_lengths", a_lengths, batch, n)
    lb = None if b_lengths is None else _lengths("b_lengths", b_lengths, batch, m)
    dev = a.device if a.is_cuda else _device()
    a, b = _to_dev(a, dev), _to_dev(b, dev)
    if a.dtype != b.dtype:
        a, b = a.double(), b.double()
    la = None if la is None else la.to(dev)
    lb = None if lb is None else lb.to(dev)
    pose = None if init_pose is None else torch.as_tensor(np.asarray(init_pose, dtype=np.float64)).to(dev).contiguous()
    if pose is not None and pose.shape != (4, 4):
        raise ValueError("init_pose must be 4x4")
    T = torch.empty(batch, 4, 4, device=dev, dtype=torch.float64)
    dist = torch.empty(batch, n, device=dev, dtype=torch.float64)
    iters = torch.empty(batch, device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        rc = _lib.lib.psd_icp_batch_ragged(_lib.ptr(a), _lib.ptr(b), int(a.dtype == torch.float64), batch, n, m, _lib.ptr(la),
                                           _lib.ptr(lb), None if pose is None else _lib.ptr(pose), int(max_iterations),
                                           ctypes.c_double(tolerance), _lib.ptr(T), _lib.ptr(dist), _lib.ptr(iters),
                                           _lib.stream_of(a))
    if rc == -1:
        raise ValueError(_lib.last_error())
    _lib.raise_on_cuda_error(rc, "psd_icp_batch_ragged")
    return T, dist, iters


def icp(A, B, init_pose=None, max_iterations=20, tolerance=0.001):
    """utils/icp.py:68-118: (T, distances, i) for one pair of [N, 3] clouds."""
    assert A.shape == B.shape
    assert max_iterations >= 1, "the reference's icp() needs at least one iteration"
    T, dist, iters = icp_batch(torch.as_tensor(A)[None], torch.as_tensor(B)[None], init_pose, max_iterations, tolerance)
    return T[0].cpu().numpy(), dist[0].cpu().numpy(), int(iters[0].item())


def best_fit_transform(A, B):
    """utils/icp.py:4-46: (T, R, t) mapping the corresponding points A onto B (3-D, evaluated in float64)."""
    assert A.shape == B.shape and A.shape[1] == 3, "the CUDA path is 3-D only"
    dev = _device()
    a = torch.as_tensor(np.asarray(A, dtype=np.float64)).to(dev)[None].contiguous()
    b = torch.as_tensor(np.asarray(B, dtype=np.float64)).to(dev)[None].contiguous()
    T = torch.empty(1, 4, 4, device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        rc = _lib.lib.psd_icp_batch(_lib.ptr(a), _lib.ptr(b), 1, 1, a.shape[1], None, 0, ctypes.c_double(0.0), _lib.ptr(T),
                                    None, None, _lib.stream_of(a))
    _lib.raise_on_cuda_error(rc, "psd_icp_batch")
    T = T[0].cpu().numpy()
    return T, T[:3, :3].copy(), T[:3, 3].copy()


def nearest_neighbor(src, dst):
    """utils/icp.py:49-65: Euclidean distance and dst index of the nearest neighbour of every src point."""
    assert src.shape == dst.shape
    dev = _device()
    s, d = _to_dev(src, dev)[None], _to_dev(dst, dev)[None]
    if s.dtype != d.dtype:
        s, d = s.double(), d.double()
    n = s.shape[1]
    dist = torch.empty(1, n, device=dev, dtype=torch.float64)
    idx = torch.empty(1, n, device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        rc = _lib.lib.psd_nn_f64(_lib.ptr(s), _lib.ptr(d), int(s.dtype == torch.float64), 1, n, d.shape[1], _lib.ptr(dist),
                                 _lib.ptr(idx), _lib.stream_of(s))
    _lib.raise_on_cuda_error(rc, "psd_nn_f64")
    return dist[0].cpu().numpy(), idx[0].cpu().numpy().astype(np.int64)
