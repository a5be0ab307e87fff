"""Builds libgwasdev.so (CUDA kernels + C-ABI) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgwasdev.so")
SWEEP_LIB = os.path.join(HERE, "libgwasdev_sweep.so")
HOST_LIB = os.path.join(HERE, "libgwaspp_host.so")
HOST_CLI = os.path.join(HERE, "gwas_b200")
SOURCES = ["store.cu", "ingest.cu", "marginal.cu", "pairwise.cu", "pairwise_mma.cu", "multi_device.cu", "permute.cu", "ld.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr", "-I", os.path.join(ROOT, "include")]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    if not os.path.exists(HOST_LIB) or not os.path.exists(HOST_CLI):
        return True
    t = min(t, os.path.getmtime(HOST_LIB), os.path.getmtime(HOST_CLI))
    host = os.path.join(HERE, "host")
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(host, f) for f in os.listdir(host)] \
        + [os.path.join(ROOT, "include", "gwasdev.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, sweep: bool = False) -> str:
    """sweep=True builds libgwasdev_sweep.so instead: the same sources with -DGWASDEV_SWEEP, i.e. with the extra kernel
    configurations, the GWASDEV_*_CFG environment parsing and the role timers that the tuning scripts under tools/ use
    (load it with GWASDEV_LIB=<path>). The product library has none of them."""
    if sweep:
        return _build_lib(SWEEP_LIB, ["-DGWASDEV_SWEEP"], "build_sweep", verbose)
    if not force and not needs_build():
        return LIB
    _build_lib(LIB, [], "build", verbose)
    build_host()
    return LIB


def _build_lib(lib: str, extra: list, objdir: str, verbose: bool) -> str:
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, objdir), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, objdir, src.replace(".cu", ".o"))
        cmd = [nvcc(), *NVCC_FLAGS, *extra, "-ccbin", "g++", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode:
            sys.stderr.write(out)
        if pr.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [nvcc(), "-shared", "-ccbin", "g++", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib, *objs, "-lz", "-ldl"]
    subprocess.check_call(link)
    return lib


def build_host() -> str:
    """C++ host mirror of the reference's GenoTable / test-class API (libgwaspp_host.so) and the small
    harness executable (gwas_b200), both above the C-ABI."""
    host = os.path.join(HERE, "host")
    inc = ["-I", os.path.join(ROOT, "include"), "-I", host]
    common = ["g++", "-std=c++17", "-O2", "-Wall", *inc]
    subprocess.check_call([*common, "-fPIC", "-shared", "-o", HOST_LIB, os.path.join(host, "device_geno_table.cpp"),
                           os.path.join(host, "test_functions.cpp"), "-L", HERE, "-lgwasdev", "-Wl,-rpath,$ORIGIN"])
    subprocess.check_call([*common, "-o", HOST_CLI, os.path.join(host, "gwas_b200.cpp"), "-L", HERE, "-lgwaspp_host",
                           "-lgwasdev", "-Wl,-rpath,$ORIGIN"])
    return HOST_LIB


if __name__ == "__main__":
    if "--variant" in sys.argv:      # experiment build: libgwasdev_<name>.so with extra -D flags (tools/time_screen.py --lib ...)
        name = sys.argv[sys.argv.index("--variant") + 1]
        defs = [a for a in sys.argv[1:] if a.startswith("-D")]
        print(_build_lib(os.path.join(HERE, f"libgwasdev_{name}.so"), defs, f"build_{name}", "-v" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, sweep="--sweep" in sys.argv))
