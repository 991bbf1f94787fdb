"""Builds libdanbo_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m danbo_b200.build         (or: from danbo_b200 import build; build.build())
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdanbo_b200.so")
SOURCES = ["version.cu", "field.cu", "field_mma.cu", "composite.cu", "mlp_tcgen05.cu", "backward_mlp.cu", "backward_field.cu", "mlp_bwd_tcgen05.cu", "anerf.cu", "anerf_bwd.cu", "loss.cu", "graphnet.cu", "pose.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "--expt-extended-lambda"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if force:                                               # from clean: no stale object can end up in the library
        for f in os.listdir(CSRC):
            if f.endswith(".o"):
                os.remove(os.path.join(CSRC, f))
        if os.path.exists(LIB):
            os.remove(LIB)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out.decode())
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
