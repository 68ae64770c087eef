"""The boundary on both sides (VERDICT r1 missing 5): pybind/psd_pybind.cpp compiled into the reference's two native module
names (`chamfer_3D`, `emd`) over the C ABI, called with the argument lists of the reference's wrappers
(metric/chamfer3D/dist_chamfer_3D.py, metric/emd/emd_module.py: caller-allocated outputs and scratch tensors), compared with
the outputs of the reference's own CUDA extensions stored in tests/golden/*_ref.npz and with the CPU oracle."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "3d-pointcloudreconstruction_b200", "pybind", "_build")


def test_pybind_modules_are_built_and_export_the_reference_names():
    """CPU check: both modules exist (built by __graft_entry__.build()) and export forward / backward.  Imported in a
    subprocess so that the module name `emd` / `chamfer_3D` cannot collide with anything loaded in this session."""
    for name in ("chamfer_3D", "emd"):
        assert os.path.exists(os.path.join(BUILD, name + ".so")), f"{name}.so missing: run python 3d-pointcloudreconstruction_b200/build.py --pybind"
    code = ("import sys, torch; sys.path.insert(0, %r); import chamfer_3D, emd; "
            "assert callable(chamfer_3D.forward) and callable(chamfer_3D.backward) and callable(emd.forward) and callable(emd.backward); "
            "print(chamfer_3D.__file__)" % BUILD)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert BUILD in out.stdout


_WORKER = r'''
import glob, json, os, sys
import numpy as np, torch
ROOT, BUILD = sys.argv[1:3]
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, BUILD)                                                # native modules: THIS repo's pybind build
import chamfer_3D, emd
assert os.path.dirname(chamfer_3D.__file__) == BUILD and os.path.dirname(emd.__file__) == BUILD
from conftest import make_clouds
from oracle import oracle as O
O.build_c()
dev = torch.device("cuda:0")
z = lambda *s, dt=torch.float32: torch.zeros(*s, device=dev, dtype=dt)


def chamfer(x, y):
    """chamfer_3DFunction.forward of dist_chamfer_3D.py: zero-filled outputs, forward into them."""
    b, n, m = x.shape[0], x.shape[1], y.shape[1]
    tx, ty = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    out = [z(b, n), z(b, m), z(b, n, dt=torch.int32), z(b, m, dt=torch.int32)]
    assert chamfer_3D.forward(tx, ty, *out) == 1
    return tx, ty, out


def emd_forward(x, y, eps, iters):
    """emdFunction.forward of emd_module.py: the 12 caller-initialised state / scratch tensors, then the native forward."""
    b, n = x.shape[:2]
    tx, ty = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    dist, ass = z(b, n), z(b, n, dt=torch.int32) - 1
    s = [z(b, n), z(b, n, dt=torch.int32) - 1, z(b, n, dt=torch.int32), z(b, n), z(b, n), z(b * n, dt=torch.int32),
         z(512, dt=torch.int32), z(512, dt=torch.int32), z(512, dt=torch.int32), z(b * n, dt=torch.int32)]
    assert emd.forward(tx, ty, dist, ass, *s, eps, iters) == 1
    return tx, ty, dist, ass


# ---- chamfer: the stored outputs of the reference's own extension, bit for bit
for f in sorted(glob.glob(os.path.join(GOLDEN, "chamfer_*_ref.npz"))):
    g = np.load(f)
    _, _, out = chamfer(g["xyz1"], g["xyz2"])
    torch.cuda.synchronize()
    for got, k in zip(out, ("dist1", "dist2", "idx1", "idx2")):
        assert np.array_equal(got.cpu().numpy(), g[k]), (f, k)
# ---- chamfer forward bits and the gradients of mean(dist1) + mean(dist2) (chamfer_3DFunction.backward) == oracle
x, y = make_clouds("uniform", 8, 1024, 1500, seed=3)
tx, ty, (d1, d2, i1, i2) = chamfer(x, y)
gx, gy = torch.zeros_like(tx), torch.zeros_like(ty)
g1 = np.full(d1.shape, 1.0 / d1.numel(), np.float32); g2 = np.full(d2.shape, 1.0 / d2.numel(), np.float32)
assert chamfer_3D.backward(tx, ty, gx, gy, torch.from_numpy(g1).to(dev), torch.from_numpy(g2).to(dev), i1, i2) == 1
torch.cuda.synchronize()
w = O.chamfer_forward(x, y, nthreads=8)
for got, want in zip((d1, d2, i1, i2), w):
    assert np.array_equal(got.cpu().numpy(), want), "chamfer forward"
wg1, wg2 = O.chamfer_backward(x, y, g1, g2, w[2], w[3])
assert np.allclose(gx.cpu().numpy(), wg1, rtol=1e-5, atol=1e-9) and np.allclose(gy.cpu().numpy(), wg2, rtol=1e-5, atol=1e-9)
# ---- EMD: the stored outputs of the reference's own extension (runs without a GetMax race in the reference: exact)
for f in sorted(glob.glob(os.path.join(GOLDEN, "emd_*_ref.npz"))):
    g = np.load(f); meta = json.loads(str(g["meta"]))
    _, _, dist, ass = emd_forward(g["xyz1"], g["xyz2"], meta["eps"], meta["iters"])
    torch.cuda.synchronize()
    assert meta["exact"], f
    assert np.array_equal(ass.cpu().numpy(), g["assignment"]) and np.array_equal(dist.cpu().numpy(), g["dist"]), f
# ---- EMD forward == oracle, and the gradient of sqrt(dist).mean(1).mean() through emdFunction.backward's native call
a, b_ = make_clouds("uniform", 4, 1024, 1024, seed=5)
ta, tb, dist, ass = emd_forward(a, b_, 0.005, 50)
torch.cuda.synchronize()
wd, wa = O.emd_forward(a, b_, 0.005, 50, nthreads=4)[:2]
assert np.array_equal(ass.cpu().numpy(), wa) and np.array_equal(dist.cpu().numpy(), wd)
gd = ((1.0 / 4 / 1024) / (2 * np.sqrt(wd))).astype(np.float32)
ga = torch.zeros_like(ta)
assert emd.backward(ta, tb, ga, torch.from_numpy(gd).to(dev), ass) == 1
torch.cuda.synchronize()
assert np.allclose(ga.cpu().numpy(), O.emd_backward(a, b_, gd, wa), rtol=1e-5, atol=1e-9)
# the shape checks of the native module are the reference's (emd_cuda.cu:236-249): -1, nothing raised at this level
bad = torch.rand(1, 1000, 3, device=dev)
s = [z(1, 1000), z(1, 1000, dt=torch.int32), z(1, 1000), z(1, 1000, dt=torch.int32), z(1, 1000, dt=torch.int32), z(1, 1000), z(1, 1000),
     z(1000, dt=torch.int32), z(512, dt=torch.int32), z(512, dt=torch.int32), z(512, dt=torch.int32), z(1000, dt=torch.int32)]
assert emd.forward(bad, bad, *s, 0.005, 5) == -1
print("PYBIND_OK")
'''


@pytest.mark.gpu
def test_pybind_modules_reproduce_the_reference_extensions(cuda):
    out = subprocess.run([sys.executable, "-c", _WORKER, ROOT, BUILD], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "PYBIND_OK" in out.stdout, (out.stdout[-1500:], out.stderr[-3000:])
