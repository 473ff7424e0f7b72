"""In-tree nvcc build of libgaussianavatars_b200.so (sm_100a only; cross-compiles without a GPU).

    python -m gaussianavatars_b200.build [--force]

preprocess.cu is compiled with --fmad=false (bit-reproducible keys, see its header); everything else with
default contraction.  The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgaussianavatars_b200.so")
OBJ_DIR = os.path.join(HERE, "csrc", "_obj")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
SOURCES = {
    "api.cu": [],
    "preprocess.cu": ["--fmad=false"],
    "preprocess_bwd.cu": [],
    "binning.cu": [],
    "tile_sort.cu": [],
    "densify.cu": [],
    "regularize.cu": [],
    "nvls.cu": [],
    "blend.cu": [],
    "face_frame.cu": [],
    "flame.cu": [],
    "loss.cu": [],
    "optim.cu": [],
}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _newest_header():
    inc = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    inc.append(os.path.join(HERE, "..", "include", "gab200_rasterizer.h"))
    return max(os.path.getmtime(p) for p in inc)


def build_native(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_time = _newest_header()
    jobs = []
    for src, extra in SOURCES.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        stale = force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_time)
        if stale:
            cmd = [_nvcc(), *ARCH, *COMMON, *extra, "-ccbin", "/usr/bin/g++", "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for out in ex.map(run, jobs):
                if verbose and out:
                    print(out)
    objs = [os.path.join(OBJ_DIR, s.replace(".cu", ".o")) for s in SOURCES]
    if jobs or not os.path.exists(LIB):
        # only the symbols of include/gab200_rasterizer.h are exported (version script); cudart is linked statically
        link = [_nvcc(), *ARCH, "-shared", "-ccbin", "/usr/bin/g++", "-o", LIB, *objs, "-Xlinker",
                "--version-script=" + os.path.join(CSRC, "exports.map")]
        run(link)
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
