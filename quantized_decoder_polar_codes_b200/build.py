"""In-tree build of the two native artefacts (they travel to the GPU box with the snapshot):

  libpolar_b200.so                  nvcc, sm_100a only   -- the C ABI of include/polar_b200.h + all kernels
  _libPolarDecoder<ext>.so          g++ / pybind11       -- host mirror of the reference's pybind11 module

Usage: python -m quantized_decoder_polar_codes_b200.build [--force]
"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libpolar_b200.so")
EXT = os.path.join(HERE, "_libPolarDecoder" + sysconfig.get_config_var("EXT_SUFFIX"))

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false",            # fp64 families: no contraction (SURVEY App. B7)
              "-Xcompiler", "-fPIC", "-shared"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources(exts):
    out = [os.path.join(ROOT, "include", "polar_b200.h")]
    for f in sorted(os.listdir(CSRC)):
        if f.endswith(exts):
            out.append(os.path.join(CSRC, f))
    return out


# translation units of libpolar_b200.so: (object name, source, extra flags, headers it depends on besides its source)
_COMMON = ["pb_internal.h", "pb_generic.cuh"]
_UNITS = [("capi", "pb_capi.cu", [], None)]          # None = every header
_UNITS += [("k%d" % t, "pb_kernels.cu", ["-DPB_TU=%d" % t], _COMMON + ["pb_scl_lut.cuh"]) for t in (1, 2, 3, 4)]
_UNITS += [("k%d" % t, "pb_kernels.cu", ["-DPB_TU=%d" % t], _COMMON + ["pb_path_warp.cuh"]) for t in (5, 6, 7, 8)]
_UNITS += [("k9", "pb_kernels.cu", ["-DPB_TU=9"], _COMMON)]
_UNITS += [("lutgen", "pb_lutgen.cu", [], ["pb_lutgen.cuh"])]
OBJDIR = os.path.join(HERE, "build")


def build_cuda(force=False, verbose=False):
    """Compile the translation units in parallel (one nvcc per object), then link."""
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJDIR, exist_ok=True)
    allhdr = _sources((".cuh", ".h"))
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])
    jobs, objs = [], []
    for name, src, extra, deps in _UNITS:
        obj = os.path.join(OBJDIR, name + ".o")
        objs.append(obj)
        dep = [os.path.join(CSRC, src)] + (allhdr if deps is None else [os.path.join(CSRC, d) for d in deps])
        if force or _newer(obj, dep):
            jobs.append([nvcc] + flags + extra + ["-c", os.path.join(CSRC, src), "-o", obj])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            def run(c):
                import time
                t0 = time.time()
                rc = subprocess.call(c)
                if verbose:
                    print("[build] %s: %.0f s" % (os.path.basename(c[-1]), time.time() - t0), flush=True)
                return rc
            for rc, cmd in zip(ex.map(run, jobs), jobs):
                if rc != 0:
                    raise subprocess.CalledProcessError(rc, cmd)
    if jobs or _newer(LIB, objs):
        subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs)
    return LIB


def pybind11_include():
    """pybind11's header directory: the pybind11 package's, else the copy torch ships (torch is a dependency anyway, so a
    Python environment without the pybind11 package still builds)"""
    try:
        import pybind11
        return pybind11.get_include()
    except ImportError:
        import torch
        inc = os.path.join(os.path.dirname(torch.__file__), "include")
        if not os.path.isfile(os.path.join(inc, "pybind11", "pybind11.h")):
            raise RuntimeError("pybind11 headers not found: neither the pybind11 package nor torch's copy is installed")
        return inc


def build_pybind(force=False):
    src = os.path.join(CSRC, "pb_pybind.cpp")
    if force or _newer(EXT, [src, os.path.join(ROOT, "include", "polar_b200.h"), LIB]):
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
               "-I" + sysconfig.get_paths()["include"], "-I" + pybind11_include(), src,
               "-L" + HERE, "-lpolar_b200", "-Wl,-rpath,$ORIGIN", "-o", EXT]
        subprocess.check_call(cmd)
    return EXT


def build_all(force=False, verbose=False):
    return build_cuda(force, verbose), build_pybind(force)


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="-v" in sys.argv))
