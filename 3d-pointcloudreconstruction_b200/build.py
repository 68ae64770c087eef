"""Build libpsd_b200.so in-tree with plain nvcc for sm_100a (no torch headers: the library is a pure C ABI)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libpsd_b200.so")
SOURCES = ["chamfer.cu", "chamfer_nn_tc.cu", "emd.cu", "proj.cu", "icp.cu", "fps.cu", "splat.cu", "sinkhorn.cu", "psd_capi.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    # no --use_fast_math: IEEE sqrt/div, denormals kept, -fmad only where written explicitly matters
]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "psd_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str = OUT, defines=()) -> str:
    """out / defines: A/B builds of the same ABI (loaded through the PSD_B200_LIB environment variable)."""
    if out == OUT and not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = ([nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-D" + d for d in defines] + ["-o", out] +
           [os.path.join(CSRC, s) for s in SOURCES])
    subprocess.check_call(cmd)
    return out


PYBIND_DIR = os.path.join(HERE, "pybind")


def build_pybind(verbose: bool = False) -> str:
    """Compile pybind/psd_pybind.cpp into the reference's two native module names, `chamfer_3D` and `emd`, linked against
    libpsd_b200.so (rpath = this directory).  The modules land in pybind/_build/ (git-ignored, shipped to the GPU box); put
    that directory on sys.path and the reference's unmodified dist_chamfer_3D.py / emd_module.py import them."""
    build()
    from torch.utils.cpp_extension import load

    out = os.path.join(PYBIND_DIR, "_build")
    src = os.path.join(PYBIND_DIR, "psd_pybind.cpp")
    for name, macro in (("chamfer_3D", "-DPSD_BIND_CHAMFER"), ("emd", "-DPSD_BIND_EMD")):
        bdir = os.path.join(out, "obj_" + name)
        os.makedirs(bdir, exist_ok=True)
        so = os.path.join(out, name + ".so")
        if os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(src), os.path.getmtime(OUT)):
            continue
        load(name=name, sources=[src], build_directory=bdir, is_python_module=False, verbose=verbose,
             extra_cflags=["-O2", macro], extra_include_paths=[os.path.join(HERE, "..", "include")],
             extra_ldflags=["-L" + HERE, "-lpsd_b200", "-Wl,-rpath," + HERE], with_cuda=True)
        import shutil
        shutil.copy2(os.path.join(bdir, name + ".so"), so)
    return out


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
    if "--pybind" in sys.argv:
        print(build_pybind(verbose="-v" in sys.argv))
