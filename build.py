"""Build helpers: everything is compiled IN-TREE with explicit commands so the
built .so files travel to the GPU box with the gpurun snapshot.

  build_cuda()        nvcc -> go-snark-study_b200/lib/libb200snark.so   (the product: sm_100a only)
  build_host_arith()  g++  -> go-snark-study_b200/lib/libb200_host_arith.so (CPU unit-test vehicle)
  build_oracle()      gcc  -> oracle/_build/liboracle.so             (test infrastructure)
  stage_ref_binary()  copies the reference's prebuilt Go CLI to oracle/_ref/ when /root/reference exists
"""
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "go-snark-study_b200")
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
ORACLE = os.path.join(ROOT, "oracle")
HOSTTEST = os.path.join(ROOT, "tests", "host")     # CPU test vehicles for the kernel headers (g++, no CUDA)

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUDA_SOURCES = ["capi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _all_sources(exts=(".cu", ".cuh", ".cpp", ".h")):
    out = []
    for d in (CSRC, os.path.join(ROOT, "include"), HOSTTEST):
        if os.path.isdir(d):
            out += [os.path.join(d, f) for f in os.listdir(d) if f.endswith(exts)]
    return out


def _run(cmd, log=None):
    p = subprocess.run(cmd, capture_output=True, text=True)
    if log:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + p.stdout + p.stderr)
    if p.returncode != 0:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-8000:])
        raise RuntimeError("build failed: " + " ".join(cmd))
    return p


def build_cuda(force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200snark.so")
    if not force and not _newer(target, _all_sources(exts=(".cu", ".cuh", ".h"))):   # the .cpp files are CPU test vehicles
        return target
    if not os.path.exists(NVCC):
        if os.path.exists(target):
            return target          # GPU box without a toolchain change: use the shipped build
        raise RuntimeError("nvcc not found and no prebuilt libb200snark.so")
    cmd = [NVCC, *NVCC_FLAGS, "-I", os.path.join(ROOT, "include"), "-I", CSRC,
           "-o", target, *[os.path.join(CSRC, s) for s in CUDA_SOURCES]]
    _run(cmd, log=os.path.join(LIBDIR, "nvcc_build.log"))
    return target


def build_host_arith(force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200_host_arith.so")
    if not force and not _newer(target, _all_sources()):
        return target
    cmd = ["g++", "-O2", "-std=c++17", "-x", "c++", "-shared", "-fPIC", "-Wno-psabi", "-I", CSRC,
           "-o", target, os.path.join(HOSTTEST, "host_arith_test.cpp")]
    _run(cmd)
    return target


def build_host_kernels(force=False):
    """g++ build of the per-thread bucket kernels over csrc/host_stub (CPU test vehicle, tests/test_host_kernels.py)."""
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200_host_kernels.so")
    if not force and not _newer(target, _all_sources() + [os.path.join(HOSTTEST, "host_stub", "cuda_runtime.h")]):
        return target
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-x", "c++", "-shared", "-fPIC", "-Wno-psabi", "-I", os.path.join(HOSTTEST, "host_stub"),
           "-I", HOSTTEST, "-I", CSRC, "-o", target, os.path.join(HOSTTEST, "host_kernel_test.cpp")]
    _run(cmd)
    return target


def build_host_verify_batch(force=False):
    """g++ build of the batch-verification kernels of csrc/verify_batch.cuh over tests/host/host_stub (CPU test vehicle,
    tests/test_host_verify_batch.py)."""
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200_host_verify_batch.so")
    if not force and not _newer(target, _all_sources() + [os.path.join(HOSTTEST, "host_stub", "cuda_runtime.h")]):
        return target
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-x", "c++", "-shared", "-fPIC", "-Wno-psabi", "-I", os.path.join(HOSTTEST, "host_stub"),
           "-I", HOSTTEST, "-I", CSRC, "-o", target, os.path.join(HOSTTEST, "host_verify_batch_test.cpp")]
    _run(cmd)
    return target


def build_host_pinocchio_verify_batch(force=False):
    """g++ build of the Pinocchio verification kernels of csrc/verify_batch_pinocchio.cuh over tests/host/host_stub (CPU
    test vehicle, tests/test_host_pinocchio_verify_batch.py)."""
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200_host_pinocchio_verify_batch.so")
    if not force and not _newer(target, _all_sources() + [os.path.join(HOSTTEST, "host_stub", "cuda_runtime.h")]):
        return target
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-x", "c++", "-shared", "-fPIC", "-Wno-psabi", "-I", os.path.join(HOSTTEST, "host_stub"),
           "-I", HOSTTEST, "-I", CSRC, "-o", target, os.path.join(HOSTTEST, "host_pinocchio_verify_batch_test.cpp")]
    _run(cmd)
    return target


def build_shard_partition(force=False):
    """g++ build of csrc/shard_partition.h behind a C entry point (CPU test vehicle, tests/test_shard_partition.py)."""
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libb200_shard_partition.so")
    srcs = [os.path.join(HOSTTEST, "shard_partition_test.cpp"), os.path.join(CSRC, "shard_partition.h")]
    if not force and not _newer(target, srcs):
        return target
    _run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, "-o", target, srcs[0]])
    return target


def build_oracle(force=False):
    out = os.path.join(ORACLE, "_build")
    os.makedirs(out, exist_ok=True)
    target = os.path.join(out, "liboracle.so")
    srcs = [os.path.join(ORACLE, "ref_c.c")]
    if not os.path.exists(srcs[0]):
        return None
    if not force and not _newer(target, srcs):
        return target
    _run(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", target, *srcs])
    return target


def stage_ref_binary():
    """The reference is Go (no toolchain here), but it ships a prebuilt CLI
    (go-snark-cli, build-cli.sh:3-4).  Stage it under oracle/_ref/ (git-ignored,
    NOT gpurun-ignored) so GPU-box tests can have real Go code verify our proofs."""
    src = "/root/reference/go-snark-cli"
    dst_dir = os.path.join(ORACLE, "_ref")
    dst = os.path.join(dst_dir, "go-snark-cli")
    if os.path.exists(src):
        os.makedirs(dst_dir, exist_ok=True)
        if not os.path.exists(dst) or os.path.getsize(dst) != os.path.getsize(src):
            shutil.copy(src, dst)
            os.chmod(dst, 0o755)
    return dst if os.path.exists(dst) else None


if __name__ == "__main__":
    print(build_host_arith(force=True))
    print(build_oracle(force=True))
    print(stage_ref_binary())
    print(build_cuda(force=True))
