"""Drop-in for metric/emd/emd_module.py: ``emdModule()(xyz1, xyz2, eps, iters) -> dist, assignment``.

Same contract as the reference (emd_module.py:9-19): clouds [B, n, 3] of equal size normalised to [0, 1],
n a multiple of 1024, B <= 512; gradient only for xyz1 (xyz2 gets zeros); the assignment is approximate and
not guaranteed to be a bijection.  The 12 scratch tensors of the reference wrapper (:43-54) are not needed:
the persistent kernel keeps the auction state in shared memory and starts from the same initial state."""
import torch
from torch import nn
from torch.autograd import Function

try:
    from . import _lib, emd
except ImportError:
    import _lib
    import emd


class emdFunction(Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2, eps, iters):
        batchsize, n, _ = xyz1.size()
        _, m, _ = xyz2.size()

        assert n == m
        assert xyz1.size()[0] == xyz2.size()[0]
        assert n % 1024 == 0
        assert batchsize <= 512

        # (the reference's .cuda() moves CUDA tensors to the CURRENT device, emd_module.py:41-42; here a CUDA input stays on
        # its own device and only host tensors are moved)
        xyz1 = xyz1.contiguous().float()
        xyz1 = xyz1 if xyz1.is_cuda else xyz1.cuda()
        xyz2 = xyz2.contiguous().float().to(xyz1.device)
        dist = torch.empty(batchsize, n, device=xyz1.device, dtype=torch.float32)
        assignment = torch.empty(batchsize, n, device=xyz1.device, dtype=torch.int32)
        rc = emd.forward_fresh(xyz1, xyz2, dist, assignment, eps, iters)
        if rc != 1:
            raise RuntimeError(f"emd.forward failed (rc={rc}): {_lib.last_error()}")
        ctx.save_for_backward(xyz1, xyz2, assignment)
        ctx.mark_non_differentiable(assignment)
        return dist, assignment

    @staticmethod
    def backward(ctx, graddist, gradidx):
        xyz1, xyz2, assignment = ctx.saved_tensors
        graddist = graddist.contiguous()
        b, n, _ = xyz1.shape
        gradxyz1 = torch.empty_like(xyz1)     # one term per address: stored by the kernel, no zero fill
        with torch.cuda.device(xyz1.device):
            rc = _lib.lib.psd_emd_backward_ex(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(gradxyz1), _lib.ptr(graddist),
                                              _lib.ptr(assignment), b, n, 1, _lib.stream_of(xyz1))
        _lib.raise_on_cuda_error(rc, "emd.backward")
        gradxyz2 = torch.zeros_like(xyz2) if ctx.needs_input_grad[1] else None   # the reference returns zeros (emd_module.py:84-87)
        return gradxyz1, gradxyz2, None, None


class emdModule(nn.Module):
    def __init__(self):
        super(emdModule, self).__init__()

    def forward(self, input1, input2, eps, iters):
        return emdFunction.apply(input1, input2, eps, iters)


class emdCertifiedFunction(Function):
    """psd_emd_certified behind autograd: dist is differentiable with respect to both clouds."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, eps_end, eps_start, scale, max_iters_per_phase):
        batchsize, n, _ = xyz1.size()
        _, m, _ = xyz2.size()
        assert n == m
        assert xyz1.size()[0] == xyz2.size()[0]
        assert n % 1024 == 0
        assert batchsize <= 512

        xyz1 = xyz1.contiguous().float()
        xyz1 = xyz1 if xyz1.is_cuda else xyz1.cuda()
        xyz2 = xyz2.contiguous().float().to(xyz1.device)
        dev = xyz1.device
        dist = torch.empty(batchsize, n, device=dev, dtype=torch.float32)
        assignment = torch.empty(batchsize, n, device=dev, dtype=torch.int32)
        price = torch.empty(batchsize, n, device=dev, dtype=torch.float32)
        bounds = torch.empty(batchsize, 2, device=dev, dtype=torch.float64)
        status = torch.empty(batchsize, device=dev, dtype=torch.int32)
        p = _lib.ptr
        with torch.cuda.device(dev):
            rc = _lib.lib.psd_emd_certified(p(xyz1), p(xyz2), batchsize, n, eps_start, eps_end, scale, int(max_iters_per_phase),
                                            p(dist), p(assignment), p(price), p(bounds), p(status), _lib.stream_of(xyz1))
        if rc == -1:
            raise ValueError(_lib.last_error())
        if rc != 1:
            raise RuntimeError(f"emd_certified failed (rc={rc}): {_lib.last_error()}")
        ctx.save_for_backward(xyz1, xyz2, assignment)
        ctx.mark_non_differentiable(assignment, bounds, status)
        return dist, assignment, bounds, status

    @staticmethod
    def backward(ctx, graddist, gradidx, gradbounds, gradstatus):
        xyz1, xyz2, assignment = ctx.saved_tensors
        graddist = graddist.contiguous()
        b, n, _ = xyz1.shape
        gradxyz1 = torch.empty_like(xyz1)
        with torch.cuda.device(xyz1.device):
            rc = _lib.lib.psd_emd_backward_ex(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(gradxyz1), _lib.ptr(graddist),
                                              _lib.ptr(assignment), b, n, 1, _lib.stream_of(xyz1))
        _lib.raise_on_cuda_error(rc, "emd_certified.backward")
        gradxyz2 = None
        if ctx.needs_input_grad[1]:
            # d dist[b,j] / d xyz2[b, a_j] is minus the xyz1 term; index_add_ sums the terms of an object that several points
            # share (an assignment that is not a permutation).  An unassigned point has a zero term.
            offs = torch.arange(b, device=xyz1.device, dtype=torch.int64)[:, None] * n
            idx = (assignment.long().clamp_min(0) + offs).reshape(-1)
            gradxyz2 = torch.zeros_like(xyz2).view(-1, 3).index_add_(0, idx, gradxyz1.view(-1, 3), alpha=-1).view_as(xyz2)
        return (gradxyz1 if ctx.needs_input_grad[0] else None), gradxyz2, None, None, None, None


def emd_certified(xyz1, xyz2, eps_end=1e-4, eps_start=0.05, scale=4.0, max_iters_per_phase=20000):
    """Earth mover's distance run to a true matching, with a bound on its distance from the optimum.

    The auction of ``emdModule`` runs in epsilon-scaling phases (eps_start, eps_start / scale, ... down to eps_end), each
    one from an empty assignment and the previous phase's prices, until every point is assigned.  A certificate kernel
    then bounds the optimal matching cost from both sides by weak duality.  Same input contract as ``emdModule``
    (clouds [B, n, 3] in [0, 1], n a multiple of 1024, B <= 512); eps_end >= 1e-5.

    Returns ``(dist, assignment, bounds, status)``:
      * dist [B, n] fp32, squared distances as in ``emdModule``, differentiable w.r.t. both clouds;
      * assignment [B, n] int32, a permutation when status is 1;
      * bounds [B, 2] fp64, (lower, upper) on the optimal EMD per point, the unit of ``sqrt(dist).mean(1)``:
        lower <= true EMD <= upper, with upper - lower <= eps_end in practice;
      * status [B] int32, 1 = permutation (both bounds valid), 0 = a phase ran out of ``max_iters_per_phase`` and the result
        is not a matching (lower bound still valid, upper is NaN), or a cloud has a NaN or infinite coordinate (no
        certificate: both bounds NaN)."""
    return emdCertifiedFunction.apply(xyz1, xyz2, float(eps_end), float(eps_start), float(scale), int(max_iters_per_phase))
