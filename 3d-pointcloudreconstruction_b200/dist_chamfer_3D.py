"""Drop-in for metric/chamfer3D/dist_chamfer_3D.py: ``chamfer_3DDist()(xyz1, xyz2) -> dist1, dist2, idx1, idx2``
with autograd to both clouds.  Differences from the reference wrapper, none of them visible in results:
outputs are allocated on the device directly (the reference allocates on the CPU and copies,
dist_chamfer_3D.py:40-49), there is no global ``torch.cuda.set_device`` side effect (:50), idx outputs are
marked non-differentiable, a failed launch raises instead of being ignored (:52), and a cloud that arrives as the
transposed view of a contiguous [B,3,N] tensor -- what the training loop passes, ``fake.transpose(2,1)`` at train.py:163 --
is read (and its gradient written) in place through strides instead of being copied by ``.contiguous()`` (:79-80)."""
import torch
from torch import nn
from torch.autograd import Function

try:
    from . import _lib
    from .sinkhorn import _lengths
except ImportError:
    import _lib
    from sinkhorn import _lengths


def cloud_layout(t):
    """0 for a contiguous [B,N,3] cloud, 1 for the transposed view of a contiguous [B,3,N] tensor, None otherwise."""
    if t.dim() != 3 or t.shape[2] != 3:
        return None
    if t.is_contiguous():
        return 0
    b, n, _ = t.shape
    if t.stride(2) == n and t.stride(1) == 1 and (t.stride(0) == 3 * n or b == 1):
        return 1
    return None


def as_kernel_cloud(t):
    """(tensor the kernels can read in place, layout flag)."""
    lay = cloud_layout(t)
    if lay is None or t.dtype != torch.float32:
        return t.contiguous(), 0
    return t, lay


def grad_buffers(xyz1, xyz2, layout, zero=False):
    """One allocation for both gradients (adjacent, so that one fill covers them); each is returned as a [B,N,3] view with the
    memory layout of its cloud.  Returns (flat buffer, grad1, grad2)."""
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    flat = (torch.zeros if zero else torch.empty)(3 * b * (n + m), device=xyz1.device, dtype=torch.float32)
    g1, g2 = flat[: 3 * b * n], flat[3 * b * n:]
    g1 = g1.view(b, 3, n).transpose(1, 2) if layout & 1 else g1.view(b, n, 3)
    g2 = g2.view(b, 3, m).transpose(1, 2) if layout & 2 else g2.view(b, m, 3)
    return flat, g1, g2


def _kernel_pair(xyz1, xyz2):
    """Checks a cloud pair and returns (xyz1, xyz2, layout) as the kernels read them."""
    batchsize, n, dim = xyz1.size()
    assert dim == 3, "Wrong last dimension for the chamfer distance 's input! Check with .size()"
    _, m, dim = xyz2.size()
    assert dim == 3, "Wrong last dimension for the chamfer distance 's input! Check with .size()"
    for name, t in (("xyz1", xyz1), ("xyz2", xyz2)):
        if not t.is_cuda:
            raise RuntimeError(f"{name}: expected a CUDA tensor (this op has no CPU path)")
        if t.dtype != torch.float32:
            raise RuntimeError(f"{name}: expected dtype torch.float32, got {t.dtype}")
    if xyz2.size(0) != batchsize or xyz2.device != xyz1.device:
        raise RuntimeError("chamfer_3DFunction: xyz1 and xyz2 need the same batch size and device")
    xyz1, l1 = as_kernel_cloud(xyz1)
    xyz2, l2 = as_kernel_cloud(xyz2)
    return xyz1, xyz2, l1 | (l2 << 1)


class chamfer_3DFunction(Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2):
        xyz1, xyz2, layout = _kernel_pair(xyz1, xyz2)
        batchsize, n, _ = xyz1.size()
        m = xyz2.size(1)
        device = xyz1.device
        dist1 = torch.empty(batchsize, n, device=device, dtype=torch.float32)
        dist2 = torch.empty(batchsize, m, device=device, dtype=torch.float32)
        idx1 = torch.empty(batchsize, n, device=device, dtype=torch.int32)
        idx2 = torch.empty(batchsize, m, device=device, dtype=torch.int32)
        if n == 0 or m == 0 or batchsize == 0:  # the reference leaves its zero-filled outputs untouched
            dist1.zero_(); dist2.zero_(); idx1.zero_(); idx2.zero_()
        # the gradient buffers of a backward that may follow are zero-filled by the forward launch itself (the reference
        # zero-fills them on the CPU and copies, dist_chamfer_3D.py:62-66): no memset on the way back
        ctx.grads = grad_buffers(xyz1, xyz2, layout) if any(ctx.needs_input_grad) else None
        with torch.cuda.device(device):
            rc = _lib.lib.psd_chamfer_forward_zero(_lib.ptr(xyz1), _lib.ptr(xyz2), batchsize, n, m, layout, _lib.ptr(dist1),
                                                   _lib.ptr(dist2), _lib.ptr(idx1), _lib.ptr(idx2), None, 0.0, None,
                                                   _lib.ptr(ctx.grads[0]) if ctx.grads else None,
                                                   ctx.grads[0].numel() if ctx.grads else 0, _lib.stream_of(xyz1))
        if rc != 1:
            raise RuntimeError(f"chamfer_3D.forward failed (rc={rc}): {_lib.last_error()}")
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2)
        ctx.layout = layout
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, dist2, idx1, idx2

    @staticmethod
    def backward(ctx, graddist1, graddist2, gradidx1, gradidx2):
        xyz1, xyz2, idx1, idx2 = ctx.saved_tensors
        layout = ctx.layout
        b, n, _ = xyz1.shape
        m = xyz2.shape[1]
        graddist1 = graddist1.contiguous()
        graddist2 = graddist2.contiguous()
        # buffers the forward launch zero-filled; a second backward through the same graph gets fresh zeros
        grads, ctx.grads = ctx.grads, None
        _, gradxyz1, gradxyz2 = grads if grads is not None else grad_buffers(xyz1, xyz2, layout, zero=True)
        with torch.cuda.device(xyz1.device):
            rc = _lib.lib.psd_chamfer_backward_ex(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(gradxyz1), _lib.ptr(gradxyz2),
                                                  _lib.ptr(graddist1), _lib.ptr(graddist2), _lib.ptr(idx1), _lib.ptr(idx2),
                                                  b, n, m, layout, 0, _lib.stream_of(xyz1))
        if rc != 1:
            raise RuntimeError(f"chamfer_3D.backward failed (rc={rc}): {_lib.last_error()}")
        return gradxyz1, gradxyz2


class chamfer_3DDist(nn.Module):
    def __init__(self):
        super(chamfer_3DDist, self).__init__()

    def forward(self, input1, input2):
        # (the reference calls .contiguous() here; chamfer_3DFunction reads [B,N,3] and transposed [B,3,N] views in place
        # and copies only what it cannot address through strides)
        return chamfer_3DFunction.apply(input1, input2)


class chamfer_raggedFunction(Function):
    """psd_chamfer_forward_ragged / psd_chamfer_backward_ragged behind autograd (see chamfer_ragged)."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, len1, len2):
        xyz1, xyz2, layout = _kernel_pair(xyz1, xyz2)
        b, n, _ = xyz1.size()
        m = xyz2.size(1)
        device = xyz1.device
        dist1 = torch.empty(b, n, device=device, dtype=torch.float32)
        dist2 = torch.empty(b, m, device=device, dtype=torch.float32)
        idx1 = torch.empty(b, n, device=device, dtype=torch.int32)
        idx2 = torch.empty(b, m, device=device, dtype=torch.int32)
        ctx.grads = grad_buffers(xyz1, xyz2, layout) if any(ctx.needs_input_grad[:2]) else None
        p = _lib.ptr
        with torch.cuda.device(device):
            rc = _lib.lib.psd_chamfer_forward_ragged(p(xyz1), p(xyz2), b, n, m, layout, p(len1), p(len2), p(dist1), p(dist2),
                                                     p(idx1), p(idx2), None, 0.0, None, p(ctx.grads[0]) if ctx.grads else None,
                                                     ctx.grads[0].numel() if ctx.grads else 0, _lib.stream_of(xyz1))
        if rc != 1:
            raise RuntimeError(f"chamfer_ragged.forward failed (rc={rc}): {_lib.last_error()}")
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2, len1, len2)
        ctx.layout = layout
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, dist2, idx1, idx2

    @staticmethod
    def backward(ctx, graddist1, graddist2, gradidx1, gradidx2):
        xyz1, xyz2, idx1, idx2, len1, len2 = ctx.saved_tensors
        b, n, _ = xyz1.shape
        m = xyz2.shape[1]
        graddist1 = graddist1.contiguous()
        graddist2 = graddist2.contiguous()
        grads, ctx.grads = ctx.grads, None
        _, gradxyz1, gradxyz2 = grads if grads is not None else grad_buffers(xyz1, xyz2, ctx.layout, zero=True)
        p = _lib.ptr
        with torch.cuda.device(xyz1.device):
            rc = _lib.lib.psd_chamfer_backward_ragged(p(xyz1), p(xyz2), p(gradxyz1), p(gradxyz2), p(graddist1), p(graddist2),
                                                      p(idx1), p(idx2), p(len1), p(len2), b, n, m, ctx.layout,
                                                      _lib.stream_of(xyz1))
        if rc != 1:
            raise RuntimeError(f"chamfer_ragged.backward failed (rc={rc}): {_lib.last_error()}")
        return gradxyz1, gradxyz2, None, None


def ragged_lengths(x_lengths, y_lengths, b, n, m, device):
    """The per-pair lengths of a ragged call as int32 [b] tensors on `device` (None stays None), checked as
    sinkhorn_divergence checks them."""
    return tuple(None if t is None else _lengths(name, t, b, size).to(device)
                 for name, t, size in (("x_lengths", x_lengths, n), ("y_lengths", y_lengths, m)))


def chamfer_ragged(x, y, x_lengths=None, y_lengths=None):
    """Chamfer nearest neighbours of a ragged batch in one launch: ``-> dist1 [B, N], dist2 [B, M], idx1, idx2``.

    x [B, N, 3] and y [B, M, 3] are padded fp32 CUDA clouds (or transposed views of contiguous [B, 3, N] tensors, read and
    their gradients written in place, as in chamfer_3DDist).  Pair b uses only the first x_lengths[b] points of x[b] and
    y_lengths[b] points of y[b]; None means the full size, and with both None this is chamfer_3DDist.  The rows past the
    lengths are never read: they may hold anything.  dist / idx of each pair are the bits of chamfer_3DDist on the pair's
    points alone; rows past the lengths get dist 0 and idx -1 and a zero gradient, whatever the upstream gradient there.
    Gradients flow to both clouds.

    Lengths are checked as in sinkhorn_divergence: a list or CPU tensor raises ValueError unless every length is in [1, N] /
    [1, M]; a CUDA integer tensor is used as it is (no host synchronisation, so the call can be captured in a CUDA graph),
    and a pair with a length out of range gets dist NaN, idx -1 and NaN gradients without affecting the others.
    ``pack_clouds`` builds the padded batch from a list of clouds.  The per-cloud mean Chamfer distance is exact because
    padding rows are 0::

        d1, d2, _, _ = chamfer_ragged(x, y, x_len, y_len)
        cd = d1.sum(1) / x_len + d2.sum(1) / y_len
    """
    if x_lengths is None and y_lengths is None:
        return chamfer_3DFunction.apply(x, y)
    if x.dim() != 3 or y.dim() != 3 or x.size(0) != y.size(0):
        raise ValueError(f"chamfer_ragged: expected clouds [B, N, 3] and [B, M, 3], got {tuple(x.shape)} and {tuple(y.shape)}")
    l1, l2 = ragged_lengths(x_lengths, y_lengths, x.size(0), x.size(1), y.size(1), x.device)
    return chamfer_raggedFunction.apply(x, y, l1, l2)
