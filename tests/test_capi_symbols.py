"""CPU-only: the C-ABI shared library builds for sm_100a, loads, and exports every symbol that
include/gsplat_b200.h declares (no compute calls -- there is no GPU in the build container)."""
import ctypes
import os
import re

from opensplat_b200 import build, capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    txt = open(os.path.join(ROOT, "include", "gsplat_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gsb_[a-z0-9_]+)\s*\(", txt)))


def test_library_builds_and_exports_every_declared_symbol():
    so = build.build()
    assert os.path.exists(so)
    L = ctypes.CDLL(so)
    names = _declared()
    assert len(names) >= 16
    for n in names:
        assert hasattr(L, n), f"{n} declared in gsplat_b200.h but not exported"


def test_python_binding_covers_header():
    bound = set(capi.exported_symbols())
    for n in _declared():
        assert n in bound or n in capi._OPT_SIGS, f"{n} not bound in capi.py"


def test_version_and_no_cpu_fallback():
    import pytest
    import torch
    L = capi.lib()
    assert L.gsb_version() >= 100
    from opensplat_b200 import ops
    with pytest.raises(capi.GsbError):  # CPU tensors are rejected, never silently computed on the host
        ops.compute_sh_forward(0, 0, torch.zeros(4, 3), torch.zeros(4, 1, 3))


def test_cubin_is_sm100a_and_uses_tma_bulk_copy():
    import subprocess
    so = build.build()
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out  # cp.async.bulk in the blend kernels


def test_cxx_libraries_use_the_shared_libstdcxx():
    """A C++ .so that carries its own statically linked copy of libstdc++'s iostream / locale code next to the
    shared one libtorch uses crashes as soon as it formats a number on a stream created by the other copy (seen
    here: the image's default g++ wrapper has a dangling libstdc++.so symlink and silently falls back to
    libstdc++.a).  build_ops.shared_stdcxx_flags() / oracle/Makefile STDCXX_DIR prevent it; this pins it."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libs = [os.path.join(root, "opensplat_b200", "lib", "libopensplat_b200_ops.so"),
            os.path.join(root, "oracle", "_ref", "libopensplat_model_b200.so"),
            os.path.join(root, "oracle", "_ref", "libopensplat_ref_cpu.so"),
            os.path.join(root, "oracle", "_ref", "libopensplat_ref_model.so")]
    checked = 0
    for lib in libs:
        if not os.path.exists(lib):
            continue
        out = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True).stdout
        assert "_ZNSo9_M_insertIlEERSoT_" not in out, f"{lib} embeds a static copy of libstdc++ (ostream::_M_insert<long>)"
        checked += 1
    assert checked >= 1


def _prototypes():
    """{name: (return type, [parameter types])} parsed from include/gsplat_b200.h (comments stripped)."""
    txt = open(os.path.join(ROOT, "include", "gsplat_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"\b(int|size_t|const char \*)\s*(gsb_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", txt, flags=re.S):
        params = " ".join(params.split())
        plist = [] if params in ("", "void") else [p.strip() for p in params.split(",")]
        protos[name] = (ret, plist)
    return protos


def _ctype_of(decl):
    """ctypes class of one C parameter declaration of the header."""
    import ctypes as C
    if "*" in decl:
        return C.c_void_p
    base = decl.rsplit(" ", 1)[0].replace("const ", "").strip()
    return {"int": C.c_int, "int32_t": C.c_int, "float": C.c_float, "size_t": C.c_size_t, "long long": C.c_longlong,
            "unsigned": C.c_uint, "unsigned int": C.c_uint, "gsb_stream_t": C.c_void_p}[base]


def test_ctypes_signatures_match_the_header_prototypes():
    """Every binding in capi._SIGS has the arity and the scalar/pointer classes of its prototype in
    include/gsplat_b200.h (an int bound as a float, or a dropped argument, would otherwise only show as garbage on
    the GPU box)."""
    import ctypes as C
    protos = _prototypes()
    assert len(protos) >= 50, len(protos)
    sigs = dict(capi._SIGS)
    sigs.update(capi._OPT_SIGS)
    checked = 0
    for name, (ret, plist) in protos.items():
        assert name in sigs, name
        restype, argtypes = sigs[name]
        assert len(argtypes) == len(plist), (name, len(argtypes), len(plist), plist)
        for i, (a, decl) in enumerate(zip(argtypes, plist)):
            want = _ctype_of(decl)
            if want is C.c_void_p:     # pointers and the stream handle: bound as void* (or a typed pointer)
                assert a is C.c_void_p or issubclass(a, C._Pointer), (name, i, decl, a)
            else:
                assert a is want, (name, i, decl, a, want)
        want_ret = {"int": C.c_int, "size_t": C.c_size_t, "const char *": C.c_char_p}[ret]
        assert restype is want_ret, (name, restype, want_ret)
        checked += 1
    assert checked == len(protos)
