"""Debiased Sinkhorn divergence between point clouds of any sizes, on the ``psd_sinkhorn_divergence`` kernel.

The transport loss for what the auction EMD cannot compare: clouds of different sizes (a 1024-point prediction against a
2048-point scan, 128- or 256-point ground truths), sizes that are not a multiple of 1024, and clouds outside the unit cube.  It
is smooth and has a gradient with respect to both clouds.  A batch of clouds of different sizes, or with point weights, runs in
one launch (``x_lengths`` / ``y_lengths``, ``x_weights`` / ``y_weights``; ``pack_clouds`` builds the padded batch)."""
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
    def forward(ctx, x, y, blur, scaling, x_len=None, y_len=None, x_w=None, y_w=None):
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
            if x_len is None and y_len is None and x_w is None and y_w is None:
                rc = _lib.lib.psd_sinkhorn_divergence(p(x), p(y), b, n, m, blur, scaling, p(loss), p(gx), p(gy), None, None,
                                                      _lib.stream_of(x))
            else:
                rc = _lib.lib.psd_sinkhorn_divergence_weighted(p(x), p(y), b, n, m, p(x_len), p(y_len), p(x_w), p(y_w), blur,
                                                               scaling, p(loss), p(gx), p(gy), None, None, _lib.stream_of(x))
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
        return (gx * w if gx is not None else None), (gy * w if gy is not None else None), None, None, None, None, None, None


def _lengths(name, t, b, size):
    """Per-pair lengths as an int32 [b]: a CUDA integer tensor is taken as it is (the kernel makes a pair with a length
    outside [1, size] NaN); a list or CPU tensor is checked here."""
    if torch.is_tensor(t) and t.is_cuda:
        if t.dtype not in (torch.int32, torch.int64) or t.shape != (b,):
            raise ValueError(f"{name}: expected an integer tensor of shape [{b}], got {t.dtype} {tuple(t.shape)}")
        return t.to(torch.int32).contiguous()
    v = torch.as_tensor(t)
    if v.dtype.is_floating_point or v.dtype == torch.bool or v.shape != (b,):
        raise ValueError(f"{name}: expected {b} integer lengths, got {v.dtype} {tuple(v.shape)}")
    if b and (int(v.min()) < 1 or int(v.max()) > size):
        raise ValueError(f"{name}: every length must be in [1, {size}]")
    return v.to(torch.int32).contiguous()


def _weights(name, w, shape):
    if not torch.is_tensor(w) or tuple(w.shape) != shape:
        raise ValueError(f"{name}: expected a tensor of shape {list(shape)}")
    if w.requires_grad and torch.is_grad_enabled():
        raise ValueError(f"{name}: point weights are not differentiable; pass weights.detach()")
    return w.detach().to(torch.float32).contiguous()


def pack_clouds(clouds):
    """Pads a list of clouds [k_i, 3] (k_i >= 1, all on one device) into (x [B, max k_i, 3] with zero rows past each length,
    lengths [B] int32 on the same device) for ``sinkhorn_divergence(..., x_lengths=lengths)``."""
    if len(clouds) == 0:
        raise ValueError("pack_clouds: no clouds")
    for c in clouds:
        if c.dim() != 2 or c.size(1) != 3 or c.size(0) < 1:
            raise ValueError(f"pack_clouds: every cloud must be [k, 3] with k >= 1, got {tuple(c.shape)}")
    dev = clouds[0].device
    lengths = torch.tensor([c.size(0) for c in clouds], dtype=torch.int32)
    out = clouds[0].new_zeros(len(clouds), int(lengths.max()), 3)
    for i, c in enumerate(clouds):
        out[i, :c.size(0)] = c
    return out, lengths.to(dev)


def sinkhorn_divergence(x, y, blur=0.05, scaling=0.5, *, x_lengths=None, y_lengths=None, x_weights=None, y_weights=None):
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
    blur <= 0, scaling outside (0, 1), or sizes outside the limits.

    Ragged and weighted batches (geomloss's ``SamplesLoss(...)(α, x, β, y)``), in the same single launch:

    * ``x_lengths`` / ``y_lengths`` [B]: pair b uses only the first x_lengths[b] points of x[b] (and likewise for y); the rows
      past a length are never read and get a zero gradient.  A list or CPU tensor is checked here (ValueError unless every
      length is in [1, N] / [1, M]); a CUDA integer tensor is used as it is, and a pair with a length out of range gives NaN.
    * ``x_weights`` [B, N] / ``y_weights`` [B, M]: fp32 point weights α, β (None: uniform, 1 / length).  A weight of 0 removes
      the point as a target; the diameter still spans every participating point, as in geomloss.  The weights are not
      normalised (that each side sums to 1 is the caller's contract, as in geomloss) and not differentiable: a weight tensor
      that requires grad while grad mode is on raises ValueError.  A pair with a negative, NaN or infinite participating
      weight, or whose participating weights on one side are all 0, gives NaN.

    With weights None, each pair gives the bits of a call on its participating points alone; ``pack_clouds`` builds the
    padded batch from a list of clouds."""
    if x_lengths is None and y_lengths is None and x_weights is None and y_weights is None:
        return sinkhornFunction.apply(x, y, float(blur), float(scaling))
    assert x.dim() == 3 and x.size(2) == 3, "x must be [B, N, 3]"
    assert y.dim() == 3 and y.size(2) == 3, "y must be [B, M, 3]"
    b, n, m = x.size(0), x.size(1), y.size(1)
    extra = (None if x_lengths is None else _lengths("x_lengths", x_lengths, b, n),
             None if y_lengths is None else _lengths("y_lengths", y_lengths, b, m),
             None if x_weights is None else _weights("x_weights", x_weights, (b, n)),
             None if y_weights is None else _weights("y_weights", y_weights, (b, m)))
    dev = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    return sinkhornFunction.apply(x, y, float(blur), float(scaling), *(None if t is None else t.to(dev) for t in extra))
