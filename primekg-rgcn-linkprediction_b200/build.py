"""In-tree build of the C-ABI library ``csrc/librgcn_b200.so`` with nvcc for sm_100a.

``python primekg-rgcn-linkprediction_b200/build.py`` (or ``__graft_entry__.build()``).  The built
``.so`` stays next to the sources so it travels to the GPU box with the repo snapshot.
nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "librgcn_b200.so")
SOURCES = ["lib.cu", "csr_build.cu", "aggregate.cu", "decoder.cu", "transform.cu", "rank.cu", "p2p.cu", "rowsparse.cu", "basis.cu", "layer.cu", "fused_layer.cu", "probe.cu", "optim.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas=-v",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; the RGCN B200 library cannot be built")
    return nvcc


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stamp() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for fn in sorted(os.listdir(root)):
            if fn.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, fn), "rb") as f:
                    h.update(fn.encode())
                    h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp_file = os.path.join(CSRC, ".build_stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()
    objs = []

    def compile_one(src):
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, _sources()))
    objs = [o for o, _ in results]
    with open(os.path.join(CSRC, "ptxas_info.txt"), "w") as f:
        for (_, log), src in zip(results, _sources()):
            f.write(f"==== {src}\n{log}\n")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
