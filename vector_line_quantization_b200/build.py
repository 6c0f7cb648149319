"""In-tree build of the two shared libraries of the package (no JIT cache: the .so files travel with the repo snapshot).

  lib/libvlq_b200.so  hand-written sm_100a CUDA kernels behind the C-ABI of include/vlq_b200.h       (nvcc)
  lib/libvlq_host.so  C++ host layer: faiss::Index-shaped classes + C wrapper include/vlq_index_c.h   (g++, links the above)

Usage:  python -m vector_line_quantization_b200.build [--force] [--verbose]
"""
import concurrent.futures as cf
import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build", "obj")
INCLUDE = os.path.join(ROOT, "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr", "-Xptxas", "-v",
]
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-Wall", "-Wno-unused-function", "-pthread"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA path cannot be built (there is no CPU fallback)")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd, verbose, log=None):
    out = subprocess.run(cmd, capture_output=True, text=True)
    if log is not None:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + out.stdout + out.stderr)
    if out.returncode != 0:
        raise RuntimeError("build step failed:\n%s\n%s%s" % (" ".join(cmd), out.stdout, out.stderr))
    if verbose:
        sys.stderr.write(out.stdout + out.stderr)


def build_cuda(force=False, verbose=False):
    os.makedirs(OBJDIR, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    hdrs = glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(INCLUDE, "*.h")) + [__file__]
    jobs = []
    objs = []
    for s in srcs:
        o = os.path.join(OBJDIR, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        if force or _newer(o, [s] + hdrs):
            jobs.append(([nvcc] + NVCC_FLAGS + ["-I", INCLUDE, "-c", s, "-o", o], o + ".log"))
    with cf.ThreadPoolExecutor(max_workers=8) as ex:
        list(ex.map(lambda j: _run(j[0], verbose, j[1]), jobs))
    lib = os.path.join(LIBDIR, "libvlq_b200.so")
    if force or jobs or _newer(lib, objs):
        _run([nvcc, "-shared", "-o", lib] + objs + ["-lcudart"], verbose)
    return lib


def build_host(force=False, verbose=False):
    srcs = sorted(glob.glob(os.path.join(HOST, "*.cpp")))
    if not srcs:
        return None
    # the host layer includes csrc/pq4.cuh (the 4-bit code format is shared with the device code)
    hdrs = (glob.glob(os.path.join(HOST, "*.h")) + glob.glob(os.path.join(INCLUDE, "*.h")) +
            [os.path.join(CSRC, "pq4.cuh"), __file__])
    lib = os.path.join(LIBDIR, "libvlq_host.so")
    cuda_lib = os.path.join(LIBDIR, "libvlq_b200.so")
    if force or _newer(lib, srcs + hdrs + [cuda_lib]):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        _run([cxx] + CXX_FLAGS + ["-shared", "-I", INCLUDE, "-I", HOST, "-o", lib] + srcs +
             ["-L", LIBDIR, "-lvlq_b200", "-Wl,-rpath,$ORIGIN"], verbose)
    return lib


def build_all(force=False, verbose=False):
    a = build_cuda(force, verbose)
    b = build_host(force, verbose)
    return a, b


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
