"""Builds libnimble_b200.so and the static libnimble_b200.a (C ABI, include/nimble_b200.h) in-tree with nvcc for sm_100a. No torch involved."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libnimble_b200.so")
AR = os.path.join(HERE, "libnimble_b200.a")   # the static library north_star names: same objects, for a host that links it in (INTEGRATION.md)
CLI = os.path.join(HERE, "nimble")
SOURCES = ["library.cpp", "index_build.cpp", "fastq.cpp", "bam.cpp", "bam_group.cu", "kernels.cu", "engine.cu", "index_build_gpu.cu", "roofs.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-extended-lambda",
         "-Xcompiler", "-fPIC,-pthread,-Wall,-Wno-unused-function", "-cudart", "shared"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in ("host.hpp", "kernels.cuh", "khash.h", "kmap.cuh", "inflate.hpp", "pgunzip.hpp", "deflate_fast.hpp", "bam_group.hpp")] + [os.path.join(HERE, "..", "include", "nimble_b200.h")]
    if force or _stale(SO, deps):
        objs = []
        for s in srcs:
            o = os.path.join(CSRC, os.path.basename(s) + ".o")
            if force or _stale(o, deps):
                cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
                subprocess.check_call(cmd)
            objs.append(o)
        subprocess.check_call([NVCC, "-shared", "-cudart", "shared", "-o", SO] + objs + ["-lz", "-lpthread", "-ldl"])
        if os.path.exists(AR):
            os.remove(AR)
        subprocess.check_call(["ar", "rcs", AR] + objs)
    main = os.path.join(CSRC, "nimble_main.cpp")
    if os.path.exists(main) and (force or _stale(CLI, [main, SO])):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", CLI, main, "-L" + HERE, "-lnimble_b200", "-Wl,-rpath,$ORIGIN"])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
