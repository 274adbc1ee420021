"""Compiles the reference's model.cpp UNCHANGED (with -DUSE_CUDA) against the gsplat_b200 operator layer ->
oracle/_ref/libopensplat_model_b200.so, together with this repo's test driver tests/native/model_driver.cpp (with
GSB_DRIVER_FUSED; torch.ops.opensplat_b200_model.{train, train_fused, after_train, save}) and linked against
libopensplat_b200_ops.so / libgsplat_b200.so: the reference's caller running THIS project's operators, not product.
What tests/golden/make_golden_b200.py records from it is therefore a regression baseline of this project's operators
under that caller, not independent reference data.

This is the drop-in check for the real caller of the hot path (SURVEY.md 8b: model.cpp:147-218 must compile
unchanged): Model::forward / mainLoss / optimizersStep / afterTrain / save run as written, with
ProjectGaussians / RasterizeGaussians / SphericalHarmonics resolving to opensplat_b200/csrc/ops.

Only possible where the reference source tree exists (REF: same variable and default as oracle/Makefile).
model.cpp and model.hpp are compiled from a scratch copy under oracle/_ref/obj so that their quoted #includes of the three
operator headers (and gsplat.hpp / tile_bounds.hpp / constants.hpp) resolve to THIS repo's versions instead of the
reference's own (quoted includes search the includer's directory first); every other reference header and
tensor_math.cpp / optim_scheduler.cpp / ssim.cpp are compiled where they lie.  Nothing from the reference is copied
into the repo.  nanoflann / nlohmann / OpenCV calib3d (FetchContent / system dependencies, absent offline, unused
by model.cpp) are the name-only stand-ins in shims/model_deps/."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("REF", "/root/reference")
OUT = os.path.join(ROOT, "oracle", "_ref", "libopensplat_model_b200.so")


def build(force=False):
    if not os.path.exists(os.path.join(REF, "model.cpp")):
        return OUT if os.path.exists(OUT) else None
    sys.path.insert(0, ROOT)
    from opensplat_b200 import build_ops
    build_ops.build()
    driver = os.path.join(ROOT, "tests", "native", "model_driver.cpp")
    deps = [driver, build_ops.OUT, os.path.join(REF, "model.cpp"), os.path.join(REF, "model.hpp"), __file__]
    if not force and os.path.exists(OUT) and all(os.path.getmtime(d) <= os.path.getmtime(OUT) for d in deps):
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    tmp = os.path.join(ROOT, "oracle", "_ref", "obj", "model_b200")
    os.makedirs(tmp, exist_ok=True)
    for f in ("model.cpp", "model.hpp"):
        shutil.copy(os.path.join(REF, f), os.path.join(tmp, f))
    T = os.path.dirname(torch.__file__)
    ops = os.path.join(ROOT, "opensplat_b200", "csrc", "ops")
    flags = ["-std=c++17", "-O2", "-fPIC", "-DUSE_CUDA", "-D_GLIBCXX_USE_CXX11_ABI=1", "-w",
             f"-I{tmp}", f"-I{ops}", f"-I{os.path.join(ROOT, 'shims', 'model_deps')}", f"-I{T}/include",
             f"-I{T}/include/torch/csrc/api/include", "-I/usr/local/cuda/include", f"-I{REF}"]
    srcs = [(os.path.join(tmp, "model.cpp"), []), (os.path.join(REF, "tensor_math.cpp"), []),
            (os.path.join(REF, "optim_scheduler.cpp"), []), (os.path.join(REF, "ssim.cpp"), []),
            (driver, ["-DGSB_DRIVER_LIB=opensplat_b200_model", "-DGSB_DRIVER_FUSED"])]
    cxx = os.environ.get("CXX", "g++")

    def cc(item):
        src, extra = item
        obj = os.path.join(tmp, os.path.basename(src).replace(".cpp", ".o"))
        r = subprocess.run([cxx] + flags + extra + ["-c", src, "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"compile failed for {src}:\n{r.stderr[-6000:]}")
        return obj
    with ThreadPoolExecutor(max_workers=5) as ex:
        objs = list(ex.map(cc, srcs))
    lib = os.path.join(ROOT, "opensplat_b200", "lib")
    cmd = [cxx, "-shared", "-o", OUT] + objs + build_ops.shared_stdcxx_flags() + [
        f"-L{lib}", "-lopensplat_b200_ops", "-lgsplat_b200", "-Wl,-rpath,$ORIGIN/../../opensplat_b200/lib", f"-L{T}/lib",
        f"-Wl,-rpath,{T}/lib", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda",
        "-L/usr/local/cuda/lib64", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr[-6000:])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
