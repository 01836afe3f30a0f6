"""Build libspn_b200.so (the C-ABI library of include/spn_b200.h, spn_jpeg.h, spn_nerf.h, spn_posed.h, spn_match.h, spn_retrieval.h and spn_verify.h) in-tree with nvcc for sm_100a.

    python superpoint-nerf-pytorch_b200/build.py [--force]

No torch involvement: plain `nvcc -shared`.  The .so is git-ignored but travels to the GPU box with gpurun.
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
SO = HERE / "libspn_b200.so"
SOURCES = ["spn_api.cu", "conv_fp32.cu", "conv_tc.cu", "conv_fold.cu", "conv_split.cu", "front_tc.cu", "head_tc.cu", "geometry.cu", "nms.cu", "desc.cu", "eval.cu", "labels.cu", "jpeg.cu", "match.cu", "retrieval.cu", "verify.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def needs_build() -> bool:
    if not SO.exists():
        return True
    t = SO.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [HERE.parent / "include" / "spn_b200.h",
                                                                HERE.parent / "include" / "spn_jpeg.h",
                                                                HERE.parent / "include" / "spn_nerf.h",
                                                                HERE.parent / "include" / "spn_posed.h",
                                                                HERE.parent / "include" / "spn_match.h",
                                                                HERE.parent / "include" / "spn_retrieval.h",
                                                                HERE.parent / "include" / "spn_verify.h", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return SO
    objs = []
    bdir = HERE / "build"
    bdir.mkdir(exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = bdir / (src + ".o")
        cmd = ["nvcc", *[f for f in NVCC_FLAGS if f != "--use_fast_math=false"], "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed (see output above)")
    subprocess.check_call(["nvcc", "-shared", "-o", str(SO), *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static",
                           "-Xcompiler", "-fPIC"])
    return SO


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
