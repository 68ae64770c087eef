"""Debiased Sinkhorn divergence between point clouds of any sizes, on the ``psd_sinkhorn_divergence`` kernel.

The transport loss for what the auction EMD cannot compare: clouds of different sizes (a 1024-point prediction against a
2048-point scan, 128- or 256-point ground truths), sizes that are not a multiple of 1024, and clouds outside the unit cube.  It
is smooth and has a gradient with respect to both clouds."""
import torch
from torch.autograd import Function

try:
    from . import _lib
except ImportError:
    import _lib


class sinkhornFunction(Function):
    """psd_sinkhorn_divergence behind autograd.  The forward asks the kernel for dS/dx and dS/dy only when an input needs
    a gradient (they come out of the same launch); the backward scales them by each cloud's upstream value."""

    @staticmethod
    def forward(ctx, x, y, blur, scaling):
        assert x.dim() == 3 and x.size(2) == 3, "x must be [B, N, 3]"
        assert y.dim() == 3 and y.size(2) == 3, "y must be [B, M, 3]"
        assert x.size(0) == y.size(0), "x and y must have the same batch size"
        x = x.contiguous().float()
        x = x if x.is_cuda else x.cuda()
        y = y.contiguous().float().to(x.device)
        b, n, _ = x.shape
        m = y.shape[1]
        dev = x.device
        loss = torch.empty(b, device=dev, dtype=torch.float32)
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        p = _lib.ptr
        with torch.cuda.device(dev):
            rc = _lib.lib.psd_sinkhorn_divergence(p(x), p(y), b, n, m, blur, scaling, p(loss), p(gx), p(gy), None, None,
                                                  _lib.stream_of(x))
        if rc == -1:
            raise ValueError(_lib.last_error())
        if rc != 1:
            raise RuntimeError(f"sinkhorn_divergence failed (rc={rc}): {_lib.last_error()}")
        ctx.save_for_backward(gx, gy)
        return loss

    @staticmethod
    def backward(ctx, gloss):
        gx, gy = ctx.saved_tensors
        w = gloss.reshape(-1, 1, 1)
        return (gx * w if gx is not None else None), (gy * w if gy is not None else None), None, None


def sinkhorn_divergence(x, y, blur=0.05, scaling=0.5):
    """Debiased Sinkhorn divergence S[b] between clouds x [B, N, 3] and y [B, M, 3] (fp32, CUDA; any N, M in [1, 2^20]).

    The computation is that of geomloss ``SamplesLoss("sinkhorn", p=2, blur=blur, scaling=scaling, debias=True)`` with the
    tensorized backend, applied to each cloud pair: cost |u - v|^2 / 2, uniform weights, an epsilon schedule from the
    squared diameter of both clouds down to blur^2, symmetric updates and one extrapolation step.  This is not the EMD: the
    entropic blur biases it below the optimal transport cost (about 28 % below at the default blur 0.05 / scaling 0.5 for two
    uniform 256-point clouds in the unit cube, 0.3 % at 0.002 / 0.98).  The defaults are those the reference's
    ``batch_EMD_loss`` is recalled to use (p=2, blur=0.05, scaling=0.5); they have not been checked against its source.

    Differentiable with respect to both clouds.  Deterministic bit for bit.  A pair whose points all coincide gives 0; a pair
    with a NaN or infinite coordinate gives NaN (and NaN gradients) without affecting the others.  Every other pair gives
    finite results: each ε of the schedule is raised to at least 2^-128, which changes only pairs with a diameter (or a
    blur) below 5.4e-20, and there only the first rounds, whose potentials vanish against blur² in the last ones.  Raises ValueError for
    blur <= 0, scaling outside (0, 1), or sizes outside the limits."""
    return sinkhornFunction.apply(x, y, float(blur), float(scaling))
