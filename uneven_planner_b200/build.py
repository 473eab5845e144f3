"""In-tree build of libualm.so (CUDA kernels + C ABI + host tools) for sm_100a with nvcc.

Usage: python -m uneven_planner_b200.build [--force]
The .so is written next to the sources (uneven_planner_b200/libualm.so): it is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libualm.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

CU_SOURCES = ["ualm_api.cu", "ualm_front_end.cu"]   # parity path, device front-end + C ABI: -fmad=false (bit-identical to the host)
CU_SOURCES_FMA = ["ualm_tp.cu"]       # throughput path (precision 32 / 65): FMA contraction on, CUDA libm
CXX_SOURCES = ["host_tools.cpp", "kino_astar.cpp"]
HEADERS = ["ualm_kernels.cuh", "map_cell.h", "map_prep.h", "../../include/ualm_detmath.h", "ualm_tp_kernels.cuh", "ualm_tp_samples.cuh", "ualm_tp_host.h", "dubins.h", "kino_search.h",
           "ualm_front_end.h"]



def _flags(fma=False):
    # -fmad=false: no FMA contraction, so every double result is bit-identical to the CPU oracle's
    # (gcc -ffp-contract=off); fp64 division and sqrt are IEEE by default (no fast-math anywhere).
    # The throughput translation unit (fma=True) is compiled with contraction on.
    return ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17"] + ([] if fma else ["-fmad=false"]) + \
           ["-Xcompiler", "-fPIC,-O3" + ("" if fma else ",-ffp-contract=off"), "-I", os.path.join(ROOT, "include"), "-I", CSRC,
            "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _digest():
    h = hashlib.sha256()
    for name in CU_SOURCES + CU_SOURCES_FMA + CXX_SOURCES + HEADERS + ["../../include/ualm.h"]:
        p = os.path.join(CSRC, name)
        if os.path.exists(p):
            with open(p, "rb") as f:
                h.update(f.read())
    h.update(" ".join(_flags() + _flags(True)).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    stamp = OUT + ".stamp"
    dig = _digest()
    if not force and os.path.exists(OUT) and os.path.exists(stamp) and open(stamp).read() == dig:
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    log, objs, procs = "", [], []
    for src, fma in [(s_, False) for s_ in CU_SOURCES + CXX_SOURCES] + [(s_, True) for s_ in CU_SOURCES_FMA]:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [NVCC] + _flags(fma) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    ok = True
    for cmd, pr in procs:
        out, _ = pr.communicate()
        log += " ".join(cmd) + "\n" + out
        ok = ok and pr.returncode == 0
    if ok:
        cmd = [NVCC, "-shared", "-o", OUT] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        log += " ".join(cmd) + "\n" + res.stdout + res.stderr
        ok = res.returncode == 0
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write(log)
    if not ok:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building libualm.so")
    if verbose:
        print(log)
    with open(stamp, "w") as f:
        f.write(dig)
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", OUT)
