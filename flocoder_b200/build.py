"""Build the C-ABI library in-tree:  python -m flocoder_b200.build

nvcc cross-compiles for sm_100a without a GPU.  Output: flocoder_b200/_C/libflocoder_b200.so
(git-ignored, but it travels to the GPU box with the repo snapshot).
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
OUT_DIR = os.path.join(HERE, "_C")
LIB = os.path.join(OUT_DIR, "libflocoder_b200.so")
SOURCES = ["api.cu", "kernels_simt.cu", "conv_umma.cu", "fused.cu", "fused_attn.cu", "selftest.cu", "rk45.cu", "jvp.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


NVCC_FLAGS += [f for f in os.environ.get("FLO_NVCC_EXTRA", "").split() if f]     # e.g. -DFLO_DBG_... for experiments


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".h", ".cuh", ".inc")):
                with open(os.path.join(root, name), "rb") as f:
                    h.update(name.encode())
                    h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    stamp = os.path.join(OUT_DIR, "build.sha256")
    digest = _digest()
    if not force and os.path.isfile(LIB) and os.path.isfile(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = find_nvcc()
    objs = [os.path.join(OUT_DIR, s.replace(".cu", ".o")) for s in SOURCES]

    def compile_one(pair):
        src, obj = pair
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, zip(SOURCES, objs)))
    log = []
    for src, r in results:
        log.append(f"==== {src}\n{r.stdout}{r.stderr}")
        if r.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(OUT_DIR, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    link = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
