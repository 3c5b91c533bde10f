"""In-tree build of the C-ABI CUDA library (sm_100a only).

`python -m graphneuralnetwork_b200.build` or `__graft_entry__.build()` compiles every
`csrc/*.cu` with nvcc for `-gencode arch=compute_100a,code=sm_100a -lineinfo` and links
`graphneuralnetwork_b200/libgnn_b200.so`.  The library has no torch dependency: it is the
drop-in boundary of include/gnn_b200.h and is loaded with ctypes (`_lib.py`).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OBJ = PKG / "csrc" / "build"
LIB = PKG / "libgnn_b200.so"
SOURCES = ["api.cu", "spmm.cu", "sage.cu", "gat.cu", "graph.cu", "peer.cu", "sampler.cu", "sddmm.cu", "semantic.cu",
           "metapath.cu", "node_union.cu", "spgemm.cu"]
HEADERS = ["common.cuh", "rowreduce.cuh", "spmm_kernels.cuh", "../../include/gnn_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (no CPU fallback exists)")


def _digest(paths) -> str:
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for p in paths:
        h.update(Path(p).read_bytes())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile and link libgnn_b200.so; incremental on a content hash of sources+headers."""
    nvcc = _nvcc()
    OBJ.mkdir(parents=True, exist_ok=True)
    hdr_paths = [CSRC / h for h in HEADERS]
    jobs = []
    objs = []
    for src in SOURCES:
        sp = CSRC / src
        op = OBJ / (src + ".o")
        stamp = OBJ / (src + ".sha")
        dig = _digest([sp] + hdr_paths)
        objs.append(op)
        if not force and op.exists() and stamp.exists() and stamp.read_text() == dig:
            continue
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", str(sp), "-o", str(op)]
        jobs.append((cmd, stamp, dig))

    def run(job):
        cmd, stamp, dig = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        stamp.write_text(dig)
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for out in ex.map(run, jobs):
                if verbose and out:
                    print(out, file=sys.stderr)
    if jobs or not LIB.exists():
        cmd = [nvcc, "-shared", "-o", str(LIB)] + [str(o) for o in objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
