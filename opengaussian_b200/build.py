"""Builds opengaussian_b200/csrc/libogs_b200.so for sm_100a with nvcc (no torch headers involved).

``python -m opengaussian_b200.build`` or ``build()``; incremental (mtime based).  The .so is kept
in-tree (git-ignored) so that it travels to the GPU box with the snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(CSRC, "libogs_b200.so")
OBJ = os.path.join(CSRC, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "--expt-relaxed-constexpr", "-Xptxas", "-v"]
# translation units; preprocess.cu / binning.cu carry the bit-exact arithmetic contract (no FMA contraction), knn.cu
# computes its distances in the direct form with every operation rounded on its own
UNITS = {
    "preprocess.cu": ["--fmad=false"],
    "binning.cu": ["--fmad=false"],
    "radix.cu": [],
    "blend_fwd.cu": [],
    "blend_bwd.cu": [],
    "preprocess_bwd.cu": [],
    "kmeans_seg.cu": [],
    "peer.cu": [],
    "nvls.cu": [],
    "kmeans.cu": [],
    "mask_stats.cu": [],
    "separation.cu": [],
    "mask_iou.cu": [],
    "adam.cu": [],
    "footprint.cu": [],
    "subsets.cu": [],
    "knn.cu": ["--fmad=false"],
    "capi.cu": [],
}


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "ogs_b200.h"))
    headers.append(os.path.abspath(__file__))
    nvcc = _nvcc()
    dev_flags = os.environ.get("OGS_NVCC_FLAGS", "").split()   # developer tuning knobs (-DPB=64 ...); pass force=True with them
    jobs = []
    objs = []
    for src, extra in UNITS.items():
        sp = os.path.join(CSRC, src)
        if not os.path.exists(sp):
            continue
        op = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(op)
        if force or _stale(op, [sp] + headers):
            jobs.append(([nvcc] + ARCH + COMMON + extra + dev_flags + ["-c", sp, "-o", op], op))

    def run(job):
        cmd, op = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = op.replace(".o", ".ptxas.log")
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if verbose:
            print(r.stderr)
        return op

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            list(ex.map(run, jobs))
    if force or jobs or _stale(OUT, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", OUT] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
