"""Build libeps_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m edge_proposal_sets_b200.build [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libeps_b200.so")
SOURCES = ["eps_abi.cu", "cn_aa.cu", "topk.cu", "spmm.cu", "gcn_norm.cu", "linkpred_simt.cu", "linkpred_tc.cu", "twohop_score.cu", "comm.cu", "pair_hadamard.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "eps.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in sources():
        obj = os.path.join(HERE, "build", os.path.basename(src) + ".o")
        cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("EPS_EXTRA_NVCC_FLAGS", "").split(), "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {os.path.basename(src)}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    with open(os.path.join(HERE, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-lcudart", "-ldl"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
