"""Builds libsdbg.so (the sm_100a kernels + C ABI) in-tree with nvcc. No JIT cache: the .so lives
under serenedb_b200/_lib/ so it travels to the GPU box with the repo snapshot."""
import atexit
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libsdbg.so")
SOURCES = [os.path.join(CSRC, "sdbg_abi.cu"), os.path.join(CSRC, "posting_format.cpp")]
DEPS = SOURCES + [os.path.join(CSRC, f) for f in ("bm25_kernels.cuh", "bm25_stream.cuh", "bm25_merge.cuh", "column_kernels.cuh", "device_common.cuh",
                                                   "posting_format.hpp")] + [
    os.path.join(os.path.dirname(HERE), "include", "sdbg.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-cudart", "static"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a. Returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        if os.path.exists(LIB_PATH):
            return LIB_PATH  # GPU box without sources changed: use the shipped build
        raise RuntimeError("nvcc not found and no prebuilt libsdbg.so")
    lib_path = LIB_PATH
    if os.access(LIB_DIR if os.path.isdir(LIB_DIR) else HERE, os.W_OK):
        os.makedirs(LIB_DIR, exist_ok=True)
    else:
        # read-only tree, e.g. when the import finds the sources newer than the library: the rebuilt library goes to a
        # private temporary directory, never into the tree. The build step itself (build_adapters, the oracle) still
        # writes the tree.
        tmp_dir = tempfile.mkdtemp(prefix="sdbg-")
        atexit.register(shutil.rmtree, tmp_dir, True)
        lib_path = os.path.join(tmp_dir, "libsdbg.so")
    tmp = lib_path + ".tmp"
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp] + SOURCES + ["-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, lib_path)
    if verbose:
        print(res.stderr)
    return lib_path


HOST_DIR = os.path.join(HERE, "host")
SELFTEST = os.path.join(LIB_DIR, "adapter_selftest")


def build_adapters(force=False):
    """Compile the C++ adapters (GpuTopKIterator : irs::DocIterator, GpuAggScan) against the mock
    reference headers and link them with libsdbg.so into a self-test binary."""
    srcs = [os.path.join(HOST_DIR, f) for f in ("adapter_selftest.cpp", "gpu_adapters.cpp")]
    deps = srcs + [os.path.join(HOST_DIR, f) for f in ("gpu_adapters.hpp", "irs_mock.hpp")] + [LIB_PATH]
    if not force and os.path.exists(SELFTEST) and all(os.path.getmtime(d) <= os.path.getmtime(SELFTEST) for d in deps):
        return SELFTEST
    gxx = shutil.which("g++")
    if gxx is None:
        if os.path.exists(SELFTEST):
            return SELFTEST
        raise RuntimeError("g++ not found")
    cmd = [gxx, "-std=c++20", "-O2", "-Wall", "-Wextra", "-o", SELFTEST] + srcs + ["-L" + LIB_DIR, "-lsdbg", "-Wl,-rpath,$ORIGIN"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
    return SELFTEST


if __name__ == "__main__":
    print(build(force=True, verbose=True))
