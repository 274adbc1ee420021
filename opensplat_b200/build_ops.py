"""In-tree build of the libtorch operator layer (g++; torch headers only here, never in the .cu files):
opensplat_b200/lib/libopensplat_b200_ops.so = ProjectGaussians / RasterizeGaussians / SphericalHarmonics
autograd classes + torch.ops registration, linked against libgsplat_b200.so.
`python -m opensplat_b200.build_ops`"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import torch

from . import build as build_cuda

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "ops")
OUT = os.path.join(HERE, "lib", "libopensplat_b200_ops.so")
TORCH = os.path.dirname(torch.__file__)
CXX = os.environ.get("CXX", "g++")
FLAGS = ["-std=c++17", "-O2", "-fPIC", "-DUSE_CUDA", "-D_GLIBCXX_USE_CXX11_ABI=1", "-w",
         f"-I{TORCH}/include", f"-I{TORCH}/include/torch/csrc/api/include", "-I/usr/local/cuda/include",
         f"-I{SRC}"]
SOURCES = ["project_gaussians.cpp", "rasterize_gaussians.cpp", "spherical_harmonics.cpp", "fused_extras.cpp",
           "register.cpp"]


def shared_stdcxx_flags():
    """-L of a directory whose libstdc++.so resolves to the SHARED runtime.  This image's default g++ wrapper has a
    dangling libstdc++.so symlink and silently falls back to libstdc++.a; a second, statically linked copy of the
    iostream/locale machinery inside a .so that lives next to libtorch's shared one crashes as soon as a number is
    formatted (e.g. a TORCH_CHECK message)."""
    import glob
    for cand in sorted(glob.glob("/usr/lib/gcc/x86_64-linux-gnu/*/libstdc++.so"), reverse=True):
        if os.path.exists(cand):   # follows the symlink
            return ["-L" + os.path.dirname(cand)]
    return []


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(SRC, f) for f in os.listdir(SRC) if os.path.isfile(os.path.join(SRC, f))]
    deps.append(os.path.join(HERE, "..", "include", "gsplat_b200.h"))
    return any(os.path.getmtime(p) > t for p in deps)


def build(force=False):
    build_cuda.build()
    if not force and not needs_build():
        return OUT
    obj_dir = os.path.join(HERE, "build", "ops")
    os.makedirs(obj_dir, exist_ok=True)

    def cc(name):
        obj = os.path.join(obj_dir, name.replace(".cpp", ".o"))
        r = subprocess.run([CXX] + FLAGS + ["-c", os.path.join(SRC, name), "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"{CXX} failed for {name}:\n{r.stderr[-4000:]}")
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(cc, SOURCES))
    lib_dir = os.path.join(HERE, "lib")
    cmd = [CXX, "-shared", "-o", OUT] + objs + shared_stdcxx_flags() + [
        f"-L{lib_dir}", "-lgsplat_b200", "-Wl,-rpath,$ORIGIN", f"-L{TORCH}/lib", f"-Wl,-rpath,{TORCH}/lib",
        "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda", "-L/usr/local/cuda/lib64", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stderr[-4000:]}")
    return OUT


TEST_SRC = os.path.join(HERE, "..", "tests", "native", "model_forward_op.cpp")
TEST_OUT = os.path.join(HERE, "..", "tests", "native", "_build", "libopensplat_b200_test_ops.so")


def build_test_ops(force=False):
    """Test-only binding of gsb::modelForward (tests/native/model_forward_op.cpp) ->
    tests/native/_build/libopensplat_b200_test_ops.so, linked against the operator library built above."""
    build()
    if not force and os.path.exists(TEST_OUT) and all(
            os.path.getmtime(d) <= os.path.getmtime(TEST_OUT) for d in (TEST_SRC, OUT)):
        return TEST_OUT
    os.makedirs(os.path.dirname(TEST_OUT), exist_ok=True)
    lib_dir = os.path.join(HERE, "lib")
    cmd = [CXX] + FLAGS + ["-shared", TEST_SRC, "-o", TEST_OUT] + shared_stdcxx_flags() + [
        f"-L{lib_dir}", "-lopensplat_b200_ops", "-lgsplat_b200", "-Wl,-rpath,$ORIGIN/../../../opensplat_b200/lib",
        f"-L{TORCH}/lib", f"-Wl,-rpath,{TORCH}/lib", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda",
        "-L/usr/local/cuda/lib64", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"test ops build failed:\n{r.stderr[-4000:]}")
    return TEST_OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
