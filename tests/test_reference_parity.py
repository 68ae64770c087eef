"""GPU parity against the REFERENCE ITSELF: outputs of the reference's chamfer3D / emd CUDA extensions, compiled unmodified
for sm_100a and run on a B200 (tests/golden/make_golden.py --ref), are stored with their inputs in tests/golden/*_ref.npz
(meta source == "reference_cuda"); this library's kernels run on the same inputs and must reproduce them."""
import glob
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _stored(op):
    files = sorted(glob.glob(os.path.join(GOLDEN, f"{op}_*_ref.npz")))
    assert files, f"no stored reference outputs for {op}"
    return [os.path.basename(f) for f in files]


def _load(name):
    z = np.load(os.path.join(GOLDEN, name))
    meta = json.loads(str(z["meta"]))
    assert meta["source"] == "reference_cuda", name
    return z, meta


@pytest.mark.parametrize("variant", [1, 3], ids=["ffma", "tensor_core"])
@pytest.mark.parametrize("name", _stored("chamfer"))
def test_chamfer_matches_reference_extension(pkg, oracle, cuda, name, variant):
    """Both NN kernels (psd_chamfer_nn_variant: 1 = FFMA, 3 = tcgen05) bit-equal to the reference extension's dist / idx."""
    z, _ = _load(name)
    x, y = z["xyz1"], z["xyz2"]
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    old = pkg._lib.lib.psd_chamfer_nn_variant(variant)
    try:
        d1, d2, i1, i2 = pkg.chamfer_3DDist()(tx, ty)
        torch.cuda.synchronize()
    finally:
        pkg._lib.lib.psd_chamfer_nn_variant(old)
    for got, k in zip((d1, d2, i1, i2), ("dist1", "dist2", "idx1", "idx2")):
        assert np.array_equal(got.cpu().numpy(), z[k]), f"{k} differs from the reference extension"
    w = oracle.chamfer_forward(x, y, nthreads=4)
    assert np.array_equal(w[2], z["idx1"]) and np.array_equal(w[0], z["dist1"]), "oracle != reference"
    # gradients along the reference's indices: both sides accumulate with float atomics -> 1e-5 relative
    rng = np.random.default_rng(b * n + m)
    g1 = rng.random((b, n), dtype=np.float32); g2 = rng.random((b, m), dtype=np.float32)
    oa = torch.zeros_like(tx); ob = torch.zeros_like(ty)
    assert pkg.chamfer_3D.backward(tx, ty, oa, ob, torch.from_numpy(g1).to(cuda), torch.from_numpy(g2).to(cuda),
                                   torch.from_numpy(z["idx1"]).to(cuda), torch.from_numpy(z["idx2"]).to(cuda)) == 1
    torch.cuda.synchronize()
    wa, wb = oracle.chamfer_backward(x, y, g1, g2, z["idx1"], z["idx2"])
    for got, want in ((oa, wa), (ob, wb)):
        assert float(np.abs(got.cpu().numpy() - want).max()) <= 1e-5 * float(np.abs(want).max())


@pytest.mark.parametrize("name", _stored("emd"))
def test_emd_matches_reference_extension(pkg, oracle, cuda, name):
    z, meta = _load(name)
    x, y, eps, iters = z["xyz1"], z["xyz2"], meta["eps"], meta["iters"]
    dist, ass = pkg.emdModule()(torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda), eps, iters)
    torch.cuda.synchronize()
    dist, ass = dist.cpu().numpy(), ass.cpu().numpy()
    wd, wa = oracle.emd_forward(x, y, eps, iters, nthreads=2)[:2]
    # the stored runs had no GetMax race in the reference (no multi-winner event): identical assignment, bit-identical
    # distances
    assert meta["exact"] and meta["multi_winner_events"] == 0, name
    assert np.array_equal(ass, z["assignment"]) and np.array_equal(dist, z["dist"])
