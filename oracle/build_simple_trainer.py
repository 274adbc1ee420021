"""Compiles the reference's simple_trainer.cpp UNCHANGED against the gsplat_b200 operator layer
(opensplat_b200/csrc/ops headers + libopensplat_b200_ops.so + libgsplat_b200.so) -> oracle/_ref/simple_trainer_b200: the
reference's caller running THIS project's operators, not product.  What tests/golden/make_golden_b200.py records from
it is therefore a regression baseline of this project's operators under that caller, not independent reference data.

Only possible where the reference source tree exists (REF: same variable and default as oracle/Makefile).
The source file is compiled from a scratch copy under oracle/_ref/obj so that its quoted #includes resolve to THIS
repo's operator headers instead of the reference's own (quoted includes search the includer's directory
first); nothing from the reference is copied into the repo.  cxxopts / OpenCV (FetchContent / system
dependencies of the reference that are unavailable offline) are replaced by the minimal shims in shims/.
"""
import os
import shutil
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(os.environ.get("REF", "/root/reference"), "simple_trainer.cpp")
OUT = os.path.join(ROOT, "oracle", "_ref", "simple_trainer_b200")


def build():
    if not os.path.exists(REF):
        return OUT if os.path.exists(OUT) else None
    sys.path.insert(0, ROOT)
    from opensplat_b200 import build_ops
    build_ops.build()
    shared_stdcxx_flags = build_ops.shared_stdcxx_flags
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    tmp = os.path.join(ROOT, "oracle", "_ref", "obj", "simple_trainer")
    os.makedirs(tmp, exist_ok=True)
    shutil.copy(REF, os.path.join(tmp, "simple_trainer.cpp"))
    T = os.path.dirname(torch.__file__)
    ops = os.path.join(ROOT, "opensplat_b200", "csrc", "ops")
    shims = os.path.join(ROOT, "shims")
    lib = os.path.join(ROOT, "opensplat_b200", "lib")
    cmd = ["g++", "-std=c++17", "-O2", "-DUSE_CUDA", "-D_GLIBCXX_USE_CXX11_ABI=1", "-w",
           f"-I{ops}", f"-I{shims}", f"-I{T}/include", f"-I{T}/include/torch/csrc/api/include",
           "-I/usr/local/cuda/include", os.path.join(tmp, "simple_trainer.cpp"), os.path.join(shims, "cv_utils.cpp"),
           "-o", OUT] + shared_stdcxx_flags() + [f"-L{lib}", "-lopensplat_b200_ops", "-lgsplat_b200", "-Wl,-rpath,$ORIGIN/../../opensplat_b200/lib",
           f"-L{T}/lib", f"-Wl,-rpath,{T}/lib", "-Wl,--no-as-needed", "-ltorch", "-ltorch_cpu", "-ltorch_cuda",
           "-lc10", "-lc10_cuda", "-L/usr/local/cuda/lib64", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("simple_trainer build failed:\n" + r.stderr[-6000:])
    return OUT


if __name__ == "__main__":
    print(build())
