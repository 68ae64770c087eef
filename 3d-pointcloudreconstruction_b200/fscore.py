"""Threshold F-score of the evaluation path (loss/loss_.py:122-140), on the CUDA op's squared distances.

``fscore(dist1, dist2, threshold)`` is the plain form (the hook commented out at metric/chamfer3D/test.py:2,9);
``chamfer_fscore_fused(xyz1, xyz2, threshold)`` runs the NN search once and takes the two thresholded counts
and the two distance sums from the kernel's epilogue instead of four extra reduction kernels."""
import torch

try:
    from . import _lib, chamfer_3D
    from .dist_chamfer_3D import ragged_lengths
except ImportError:
    import _lib
    import chamfer_3D
    from dist_chamfer_3D import ragged_lengths


def _f_from_precisions(p1, p2):
    f = 2 * p1 * p2 / (p1 + p2)
    f[torch.isnan(f)] = 0
    return f


def fscore(dist1, dist2, threshold=0.0001):
    """dist1: [B, N] x->y squared NN distances, dist2: [B, M] y->x.  Returns (fscore, precision_1, precision_2)
    per cloud, precision_1 over dist1 and precision_2 over dist2 (strict '<', as loss_.py:132-133)."""
    p1 = torch.mean((dist1 < threshold).float(), dim=1)
    p2 = torch.mean((dist2 < threshold).float(), dim=1)
    return _f_from_precisions(p1, p2), p1, p2


def chamfer_fscore_fused(xyz1, xyz2, threshold=0.0001, layout=0, *, x_lengths=None, y_lengths=None):
    """layout: bit mask of psd_chamfer_forward_ex (1: xyz1 is [B,3,N], 2: xyz2 is [B,3,M]).
    One launch: returns dict(dist1, dist2, idx1, idx2, sums[B,2], counts[B,2], fscore[B], precision_1[B],
    precision_2[B], chamfer[B] = mean(dist1)+mean(dist2) per cloud).
    x_lengths / y_lengths [B]: a ragged batch (see chamfer_ragged): pair b uses the first x_lengths[b] / y_lengths[b] points,
    and the precisions and ``chamfer`` divide by those lengths."""
    b = xyz1.shape[0]
    n = xyz1.shape[2] if layout & 1 else xyz1.shape[1]
    m = xyz2.shape[2] if layout & 2 else xyz2.shape[1]
    dev = xyz1.device
    if x_lengths is not None or y_lengths is not None:
        return _fscore_ragged(xyz1, xyz2, threshold, layout, b, n, m, *ragged_lengths(x_lengths, y_lengths, b, n, m, dev))
    xyz1 = xyz1.contiguous()
    xyz2 = xyz2.contiguous()
    dist1 = torch.empty(b, n, device=dev, dtype=torch.float32)
    dist2 = torch.empty(b, m, device=dev, dtype=torch.float32)
    idx1 = torch.empty(b, n, device=dev, dtype=torch.int32)
    idx2 = torch.empty(b, m, device=dev, dtype=torch.int32)
    acc = torch.zeros(b, 4, device=dev, dtype=torch.float32)  # [:, :2] sums (fp32), [:, 2:] counts (int32 bits)
    sums = acc[:, :2].contiguous()
    counts = torch.zeros(b, 2, device=dev, dtype=torch.int32)
    rc = chamfer_3D.forward_ex(xyz1, xyz2, dist1, dist2, idx1, idx2, layout=layout, sums=sums, fs_thr=threshold,
                               fs_count=counts)
    _lib.raise_on_cuda_error(rc, "chamfer_3D.forward_ex")
    p1 = counts[:, 0].float() / n
    p2 = counts[:, 1].float() / m
    return {
        "dist1": dist1, "dist2": dist2, "idx1": idx1, "idx2": idx2, "sums": sums, "counts": counts,
        "fscore": _f_from_precisions(p1, p2), "precision_1": p1, "precision_2": p2,
        "chamfer": sums[:, 0] / n + sums[:, 1] / m,
    }


def _fscore_ragged(xyz1, xyz2, threshold, layout, b, n, m, len1, len2):
    dev = xyz1.device
    xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()
    for name, t in (("xyz1", xyz1), ("xyz2", xyz2)):
        _lib.check_tensor(name, t, torch.float32, 3)
    dist1 = torch.empty(b, n, device=dev, dtype=torch.float32)
    dist2 = torch.empty(b, m, device=dev, dtype=torch.float32)
    idx1 = torch.empty(b, n, device=dev, dtype=torch.int32)
    idx2 = torch.empty(b, m, device=dev, dtype=torch.int32)
    sums = torch.zeros(b, 2, device=dev, dtype=torch.float32)
    counts = torch.zeros(b, 2, device=dev, dtype=torch.int32)
    p = _lib.ptr
    with torch.cuda.device(dev):
        rc = _lib.lib.psd_chamfer_forward_ragged(p(xyz1), p(xyz2), b, n, m, layout, p(len1), p(len2), p(dist1), p(dist2), p(idx1),
                                                 p(idx2), p(sums), threshold, p(counts), None, 0, _lib.stream_of(xyz1))
    if rc == -1:
        raise ValueError(_lib.last_error())
    _lib.raise_on_cuda_error(rc, "psd_chamfer_forward_ragged")
    nc = float(n) if len1 is None else len1.float()
    mc = float(m) if len2 is None else len2.float()
    p1 = counts[:, 0].float() / nc
    p2 = counts[:, 1].float() / mc
    return {
        "dist1": dist1, "dist2": dist2, "idx1": idx1, "idx2": idx2, "sums": sums, "counts": counts,
        "fscore": _f_from_precisions(p1, p2), "precision_1": p1, "precision_2": p2,
        "chamfer": sums[:, 0] / nc + sums[:, 1] / mc,
    }
