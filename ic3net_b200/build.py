"""Build libic3net_b200.so in-tree with nvcc for sm_100a.

    python -m ic3net_b200.build [--force]

The shared library is a plain C-ABI object (include/ic3net_b200.h); it links only
against the CUDA runtime and is loaded by ic3net_b200/_lib.py through ctypes.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libic3net_b200.so")
SOURCES = ["c_api.cu", "pp_env.cu", "tj_env.cu", "policy.cu", "policy_tc.cu", "bptt_tc.cu", "returns.cu", "optim.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "ic3net_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    extra = os.environ.get("IC3_NVCC_EXTRA", "").split()      # extra nvcc flags for local experiments
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
        if verbose:
            print(out)
    cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs + ["-lcudart"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
