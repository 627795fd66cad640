"""In-tree build of the CUDA shared library (sm_100a) and of the C++ host-shim self test.

`nvcc` cross-compiles without a GPU.  The library links the CUDA runtime statically and has no
torch / Python dependency: it is the C-ABI of include/shyft_b200.h and nothing else.
"""
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libshyft_b200.so")

# -fmad=false: the cell stacks follow the reference's operation order; contracting a*b+c into FMA changes the last bit
# of intermediate results, which can flip the discrete decisions the reference's results are defined by (Kirchner
# accept/reject, Brent branches, gamma_snow thresholds).  See DESIGN.md "FMA policy".
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off",
              "-cudart", "static"]


def _sources():
    out = [os.path.join(ROOT, "include", "shyft_b200.h")]
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".hpp")):
            out.append(os.path.join(CSRC, f))
    return out


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built")
    return p


def build_library(force=False, verbose=False):
    """Compile shyft_b200/csrc/sb2_capi.cu -> shyft_b200/libshyft_b200.so for sm_100a."""
    if not force and not _stale(LIB, _sources()):
        return LIB
    tmp = LIB + ".tmp%d" % os.getpid()   # written aside and renamed: a concurrent reader never sees a half-written library
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-shared", "-o", tmp, os.path.join(CSRC, "sb2_capi.cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    try:
        subprocess.check_call(cmd, cwd=CSRC)
        os.replace(tmp, LIB)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return LIB


def build_host_shim_test(force=False):
    """g++ build of the C++ host shim self test (include/shyft_b200/region_model.hpp over the C ABI).  In a read-only checkout a
    missing or stale executable is built into a temporary directory instead of tests/cpp; returns the executable's path."""
    src = os.path.join(ROOT, "tests", "cpp", "shim_selftest.cpp")
    out = os.path.join(ROOT, "tests", "cpp", "shim_selftest")
    if not os.path.exists(src):
        return None
    deps = [src, os.path.join(ROOT, "include", "shyft_b200.h"), os.path.join(ROOT, "include", "shyft_b200", "region_model.hpp"), LIB]
    if force or _stale(out, deps):
        if not os.access(os.path.dirname(out), os.W_OK):
            out = os.path.join(tempfile.mkdtemp(prefix="shyft_b200_shim_"), "shim_selftest")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", out, src, "-L", HERE, "-lshyft_b200",
                               "-Wl,-rpath," + HERE, "-Wl,-rpath,$ORIGIN/../../shyft_b200"])
    return out


def pybind_module_path():
    import sysconfig
    return os.path.join(HERE, "_shyft_b200_cpp" + sysconfig.get_config_var("EXT_SUFFIX"))


def build_pybind_module(force=False):
    """g++ build of the pybind11 module over the C++ shim (shyft_b200/pybind/module.cpp -> shyft_b200/_shyft_b200_cpp.*.so)."""
    import sysconfig

    import pybind11
    src = os.path.join(HERE, "pybind", "module.cpp")
    out = pybind_module_path()
    deps = [src, os.path.join(ROOT, "include", "shyft_b200.h"), os.path.join(ROOT, "include", "shyft_b200", "region_model.hpp"), LIB]
    if force or _stale(out, deps):
        tmp = out + ".tmp%d" % os.getpid()
        try:
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-I", pybind11.get_include(),
                                   "-I", sysconfig.get_paths()["include"], "-I", os.path.join(ROOT, "include"), "-o", tmp, src,
                                   "-L", HERE, "-lshyft_b200", "-Wl,-rpath,$ORIGIN"])
            os.replace(tmp, out)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return out
