"""Builds libregt_b200.so in-tree with nvcc for sm_100a (no torch dependency, plain C-ABI)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.normpath(os.path.join(HERE, "..", ".."))
OUT = os.path.join(HERE, "..", "lib")
SOURCES = ["api_core.cu", "plan.cu", "spmm.cu", "weights.cu", "cell.cu", "cell_g.cu", "cell_f.cu", "head.cu", "head_f.cu", "input_grad.cu", "api.cu", "cell_tc.cu", "head_tc.cu", "gemm_tma.cu", "peer.cu", "loop.cu", "combine.cu", "umma_selftest.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", HERE]


def lib_path() -> str:
    return os.path.normpath(os.path.join(OUT, "libregt_b200.so"))


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OUT, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    deps = srcs + [os.path.join(HERE, "common.cuh"), os.path.join(ROOT, "include", "regt_b200.h")]
    deps += [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith(".cuh")]
    target = lib_path()
    if not force and os.path.exists(target) and all(os.path.getmtime(d) <= os.path.getmtime(target) for d in deps):
        return target
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(OUT, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        if not force and os.path.exists(o) and all(os.path.getmtime(d) <= os.path.getmtime(o) for d in [s] + deps[len(srcs):]):
            continue
        cmd = [nvcc, *NVCC_FLAGS, "-c", s, "-o", o] + (["-Xptxas", "-v"] if verbose else [])
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
        if verbose:
            print(out)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", target, *objs, "-lcudart", "-lcuda"])
    return target


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
