"""B200-native point-set distance ops (Chamfer NN fwd/bwd, auction EMD) -- drop-in for the
`metric/chamfer3D` and `metric/emd` extensions of sunhui-3D/3D-PointCloudReconstruction.

The directory can be used in two ways:
  * put it on ``sys.path`` where the reference puts ``metric/chamfer3D`` and ``metric/emd``
    (loss/loss.py:3-4): ``from dist_chamfer_3D import chamfer_3DDist``, ``import emd_module`` and even
    ``import chamfer_3D`` / ``import emd`` (the native-module names) resolve to this implementation;
  * or load it as a package through ``psd_b200.load()`` at the repository root.
There is no CPU fallback: importing `_lib` raises if libpsd_b200.so is missing.
"""
from . import _lib  # noqa: F401  (fails loudly when the CUDA library is absent)
from . import chamfer_3D, emd  # native-module mirrors (pybind names of the reference)
from . import proj_loss        # loss/proj_loss.py mirror (get_loss_proj, grid_dist)
from . import icp              # utils/icp.py mirror (icp, best_fit_transform, nearest_neighbor) + icp_batch, icp_ragged
from . import projection       # utils/projection.py mirror (cont_proj, apply_kernel)
from . import utils            # utils/utils.py sampling helpers (farthest_point_sample, index_points)
from . import loss_            # loss/loss_.py mirror (cd, distChamfer, batch_NN_loss, fscore) on the CUDA op
from .dist_chamfer_3D import chamfer_3DDist, chamfer_3DFunction, chamfer_ragged
from .emd_module import emdFunction, emdModule, emd_certified
from .fscore import fscore, chamfer_fscore_fused
from .icp import icp_ragged
from .loss import Loss, chamfer_loss_step_host, ChamferLossPipeline
from .metrics import Metrics, certified_emd_distance
from .sinkhorn import pack_clouds, sinkhornFunction, sinkhorn_divergence

__all__ = [
    "chamfer_3D", "emd", "proj_loss", "icp", "projection", "utils", "loss_", "chamfer_3DDist", "chamfer_3DFunction", "chamfer_ragged", "emdFunction", "emdModule",
    "fscore", "chamfer_fscore_fused", "Loss", "chamfer_loss_step_host", "ChamferLossPipeline", "Metrics",
    "emd_certified", "certified_emd_distance", "sinkhornFunction", "sinkhorn_divergence", "pack_clouds",
    "icp_ragged",
]
