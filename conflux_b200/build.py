"""conflux_b200/build.py -- compiles the CUDA sources in-tree into conflux_b200/libconflux_b200.so (sm_100a only).

nvcc cross-compiles without a GPU; the built .so travels to the GPU box with the repo snapshot."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libconflux_b200.so")
SOURCES = ["gemm.cu", "ozaki.cu", "panel.cu", "rows.cu", "trsm.cu", "lu.cu", "validate.cu", "solve.cu", "chol.cu", "dbg.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-O3",
         "-ccbin", "g++", "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "conflux_b200.h"))
    objs = []
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(bdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src} ---\n{out}\n")
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-lnccl", "-Xlinker", "--no-as-needed"]
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
