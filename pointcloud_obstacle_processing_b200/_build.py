"""In-tree builds: libpcop.so (CUDA, sm_100a) and libpcop_synth.so (host-only generators).

nvcc cross-compiles without a GPU, so this runs on the CPU-only dev box; the resulting .so files
travel to the GPU box with the repo snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpcop.so")
SYNTH_SRC = os.path.join(HERE, "synth", "synth.cpp")
SYNTH_LIB = os.path.join(HERE, "synth", "libpcop_synth.so")

CU_SOURCES = ["pcop_api.cu", "batch.cu", "radix_sort.cu", "stage_crop.cu", "stage_voxel.cu", "stage_voxel_fused.cu", "stage_voxel_part.cu", "stage_sor.cu", "stage_plane.cu",
              "stage_cluster.cu", "stage_cluster_small.cu", "stage_occupancy.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",          # no FMA contraction anywhere: float predicates must match the oracle bit for bit
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_cuda(force=False, verbose=False):
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "pcop.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    jobs = []
    for src in CU_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _newer(o, [s] + headers):
            extra = os.environ.get("PCOP_NVCC_EXTRA", "").split()  # e.g. -DPCOP_ECE_DEBUG_CLK for tools/ece_phases.py
            jobs.append([nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        logs = list(ex.map(run, jobs))
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in CU_SOURCES]
    if jobs or force or _newer(LIB, objs):
        run([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"])
    if verbose:
        for l in logs:
            sys.stderr.write(l)
    return LIB


def build_synth(force=False):
    if force or _newer(SYNTH_LIB, [SYNTH_SRC]):
        subprocess.check_call(["g++", "-O2", "-fPIC", "-std=c++17", "-shared", "-o", SYNTH_LIB, SYNTH_SRC])
    return SYNTH_LIB


def build_all(force=False, verbose=False):
    build_synth(force)
    return build_cuda(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
