"""In-tree build of libgds_b200.so (CUDA kernels + C ABI) and the host-side C++ mirror.

nvcc cross-compiles sm_100a without a GPU.  The .so stays in-tree (git-ignored) so it travels to
the GPU box with the snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libgds_b200.so")
HOST_BIN = os.path.join(HERE, "gds_host_test")
HOST_LIB = os.path.join(HERE, "libgds_host.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-pthread", "-shared"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _find_nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgds_b200.so cannot be built (there is no CPU fallback)")


def build_cuda(force=False, verbose=False):
    csrc = os.path.join(HERE, "csrc")
    srcs = [os.path.join(csrc, f) for f in sorted(os.listdir(csrc))]
    srcs.append(os.path.join(ROOT, "include", "gds.h"))
    if not force and not _newer(LIB, srcs):
        return LIB
    cmd = [_find_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB, os.path.join(csrc, "gds_api.cu")]
    subprocess.check_call(cmd)
    return LIB


def build_kernel_harness(force=False):
    """tests/kernels/libkernel_harness.so: the scan, radix sort and K5/K6 kernels behind C wrappers
    for tests/test_kernels.py.  Test infrastructure, never loaded by the package."""
    kdir = os.path.join(ROOT, "tests", "kernels")
    src = os.path.join(kdir, "kernel_harness.cu")
    out = os.path.join(kdir, "libkernel_harness.so")
    csrc = os.path.join(HERE, "csrc")
    srcs = [src] + [os.path.join(csrc, f) for f in sorted(os.listdir(csrc))]
    if not force and not _newer(out, srcs):
        return out
    subprocess.check_call([_find_nvcc()] + NVCC_FLAGS + ["-o", out, src])
    return out


def build_host(force=False):
    hdir = os.path.join(HERE, "host")
    if not os.path.isdir(hdir):
        return None
    srcs = [os.path.join(dp, f) for dp, _, fs in os.walk(hdir) for f in fs]
    srcs.append(os.path.join(ROOT, "include", "gds.h"))
    cpps = [s for s in srcs if s.endswith(".cpp")]
    if not cpps:
        return None
    if not force and not _newer(HOST_BIN, srcs + [LIB]) and not _newer(HOST_LIB, srcs + [LIB]):
        return HOST_BIN
    # the system g++ (the image's CXX wrapper links libstdc++ statically, which must not be
    # dlopen()ed into a process that already has libstdc++)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    common = [cxx, "-O2", "-std=c++17", "-Wall", "-fPIC", "-pthread",
              "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(hdir, "include")]
    link = ["-L" + HERE, "-lgds_b200", "-lz", "-Wl,-rpath,$ORIGIN"]
    lib_srcs = [s for s in cpps if not s.endswith("host_test_main.cpp")]
    bin_srcs = [s for s in cpps if not s.endswith("host_c_api.cpp")]
    subprocess.check_call(common + ["-shared", "-o", HOST_LIB] + lib_srcs + link)
    subprocess.check_call(common + ["-o", HOST_BIN] + bin_srcs + link)
    return HOST_BIN


if __name__ == "__main__":
    build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_host(force="--force" in sys.argv)
    print("built", LIB)
