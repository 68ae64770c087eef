"""ctypes loader for libpsd_b200.so (the C ABI declared in include/psd_b200.h).

PyTorch is only plumbing here: tensors give device pointers, the current stream and a device guard.
The library must exist -- there is deliberately no eager/CPU fallback."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSD_B200_LIB") or os.path.join(_HERE, "libpsd_b200.so")  # env override: A/B builds of the same ABI

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python 3d-pointcloudreconstruction_b200/build.py` "
        "(nvcc, sm_100a). This package has no CPU or eager fallback."
    )

lib = ctypes.CDLL(LIB_PATH)

_vp = ctypes.c_void_p
_ci = ctypes.c_int
_cf = ctypes.c_float

# every export of include/psd_b200.h with its argument types (all return int unless noted)
_SIGNATURES = {
    "psd_chamfer_forward": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp],
    "psd_chamfer_forward_ex": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _cf, _vp, _ci, _ci, _vp],
    "psd_chamfer_forward_zero": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _cf, _vp, _vp, ctypes.c_longlong, _vp],
    "psd_chamfer_backward": [_vp] * 8 + [_ci, _ci, _ci, _vp],
    "psd_chamfer_backward_ex": [_vp] * 8 + [_ci, _ci, _ci, _ci, _ci, _vp],
    "psd_chamfer_forward_ragged": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _cf, _vp, _vp,
                                   ctypes.c_longlong, _vp],
    "psd_chamfer_backward_ragged": [_vp] * 10 + [_ci, _ci, _ci, _ci, _vp],
    "psd_emd_forward": [_vp, _vp, _ci, _ci, _ci] + [_vp] * 12 + [_cf, _ci, _vp],
    "psd_emd_forward_fresh": [_vp, _vp, _ci, _ci, _vp, _vp, _cf, _ci, _vp],
    "psd_emd_forward_cluster": [_vp, _vp, _ci, _ci, _vp, _vp, _vp, _vp, _cf, _ci, _ci, _vp],
    "psd_emd_backward": [_vp, _vp, _vp, _vp, _vp, _ci, _ci, _vp],
    "psd_emd_backward_ex": [_vp, _vp, _vp, _vp, _vp, _ci, _ci, _ci, _vp],
    "psd_emd_dual_bound": [_vp, _vp, _ci, _ci, _vp, _vp, _vp, _vp, _vp],
    "psd_emd_certified": [_vp, _vp, _ci, _ci, _cf, _cf, _cf, _ci, _vp, _vp, _vp, _vp, _vp, _vp],
    "psd_emd_certified_cluster": [_vp, _vp, _ci, _ci, _cf, _cf, _cf, _ci, _vp, _vp, _vp, _vp, _vp, _ci, _vp],
    "psd_emd_mean_loss_forward": [_vp, _vp, _ci, _ci, _vp, _vp, _cf, _ci, _vp, _vp, _vp],
    "psd_emd_mean_loss_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _ci, _ci, _vp],
    "psd_sinkhorn_divergence": [_vp, _vp, _ci, _ci, _ci, _cf, _cf, _vp, _vp, _vp, _vp, _vp, _vp],
    "psd_sinkhorn_divergence_cluster": [_vp, _vp, _ci, _ci, _ci, _cf, _cf, _vp, _vp, _vp, _vp, _vp, _ci, _vp],
    "psd_sinkhorn_divergence_weighted": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _cf, _cf, _vp, _vp, _vp, _vp, _vp, _vp],
    "psd_sinkhorn_divergence_weighted_cluster": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _cf, _cf, _vp, _vp, _vp, _vp, _vp,
                                                 _ci, _vp],
    "psd_chamfer_forward_host": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp],
    "psd_fp32_fma_peak": [_cf, ctypes.POINTER(_cf), _vp],
    "psd_chamfer_stats": [ctypes.POINTER(ctypes.c_longlong), _ci],
    "psd_chamfer_nn_variant": [_ci],
    "psd_chamfer_mean_loss_forward": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "psd_chamfer_mean_loss_forward_zero": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_longlong, _vp],
    "psd_chamfer_mean_loss_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _ci, _ci, _ci, _vp],
    "psd_chamfer_mean_loss_backward_ex": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _ci, _ci, _ci, _ci, _ci, _vp],
    "psd_chamfer_loss_step_host": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _vp],
    "psd_chamfer_loss_step_host_ex": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _ci, _ci, _vp],
    "psd_chamfer_loss_step_pred_dev": [_vp, _ci, _vp, _ci, _ci, _ci, _vp, _vp, _ci, _ci, _vp],
    "psd_host_step_graphs": [_ci],
    "psd_emd_solo_mode": [_ci],
    "psd_emd_grid_mode": [_ci],
    "psd_chamfer_tc_ctas": [_ci],
    "psd_proj_min_dist": [_vp, _vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp],
    "psd_icp_batch": [_vp, _vp, _ci, _ci, _ci, _vp, _ci, ctypes.c_double, _vp, _vp, _vp, _vp],
    "psd_icp_batch_ragged": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp, _ci, ctypes.c_double, _vp, _vp, _vp, _vp],
    "psd_nn_f64": [_vp, _vp, _ci, _ci, _ci, _ci, _vp, _vp, _vp],
    "psd_farthest_point_sample": [_vp, _ci, _ci, _ci, _ci, _vp, _vp],
    "psd_cont_proj": [_vp, _ci, _ci, _ci, _ci, ctypes.c_float, _vp, _vp],
    "psd_cont_proj_backward": [_vp, _vp, _ci, _ci, _ci, _ci, ctypes.c_float, _vp, _vp],
    "psd_debug_tc_prof": [_vp],
    "psd_debug_tc_filter": [_vp, _vp, _ci, _ci, _ci, _vp, _vp, _vp, _vp, _vp, _ci, _vp],
}
lib.psd_version.restype = _ci
lib.psd_last_error.restype = ctypes.c_char_p
for _n, _a in _SIGNATURES.items():
    getattr(lib, _n).argtypes = _a
    getattr(lib, _n).restype = _ci

EXPORTS = ("psd_version", "psd_last_error") + tuple(_SIGNATURES)


def last_error() -> str:
    return lib.psd_last_error().decode("utf-8", "replace")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_of(t) -> ctypes.c_void_p:
    """torch's current stream on the tensor's device (the reference launches on the legacy default stream;
    the current stream is identical behaviour there and correct everywhere else)."""
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def check_tensor(name, t, dtype, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (this op has no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous tensor")
    if ndim is not None and t.dim() != ndim:
        raise RuntimeError(f"{name}: expected {ndim} dimensions, got {t.dim()}")


def raise_on_cuda_error(rc: int, what: str):
    """The reference printf()s and returns 0 on a launch error and Python ignores it
    (dist_chamfer_3D.py:52); here the 0 is still returned to the caller of the native-module mirror, but
    the autograd wrappers turn it into an exception."""
    if rc == 0:
        raise RuntimeError(f"{what} failed: {last_error()}")
