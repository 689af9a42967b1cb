"""Builds the sm_100a CUDA library and its pybind11 layer IN-TREE.

  centernet_b200/lib/libcenternet_b200.so   <- nvcc, every csrc/*.cu   (the C ABI)
  centernet_b200/_C<ext>.so                 <- g++,  csrc/pybind.cpp    (thin binding)

Run as ``python centernet_b200/build.py`` (add ``--force`` to rebuild).  nvcc
cross-compiles without a GPU, so this also runs in the CPU-only build container.
"""
import glob
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libcenternet_b200.so")
EXT = os.path.join(HERE, "_C" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-cudart", "static"] + os.environ.get("CNB_NVCC_DEFINES", "").split()


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return r.stdout + r.stderr


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    cus = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    hdrs = glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(HERE, "..", "include", "*.h"))
    objs = []
    rebuilt = False
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for cu in cus:
        obj = os.path.join(objdir, os.path.basename(cu)[:-3] + ".o")
        objs.append(obj)
        if force or _newer(obj, [cu] + hdrs):
            cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", cu, "-o", obj]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            rebuilt = True
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), out))
        if verbose:
            print(out)
    if rebuilt or not os.path.exists(LIB):
        _run([NVCC, "-shared", "-cudart", "static", "-o", LIB] + objs)
    src = os.path.join(CSRC, "pybind.cpp")
    if force or rebuilt or _newer(EXT, [src] + hdrs):
        import pybind11
        _run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", src,
              "-I" + pybind11.get_include(), "-I" + sysconfig.get_paths()["include"],
              "-L" + LIBDIR, "-lcenternet_b200", "-Wl,-rpath,$ORIGIN/lib", "-o", EXT])
    return LIB, EXT


if __name__ == "__main__":
    lib, ext = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built", lib)
    print("built", ext)
