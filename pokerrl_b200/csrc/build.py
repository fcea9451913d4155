"""Builds pokerrl_b200/lib/libpokerrl_b200.so with nvcc for sm_100a (in-tree, no JIT cache).

    python -m pokerrl_b200.csrc.build            # or: python pokerrl_b200/csrc/build.py [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB_DIR = os.path.join(os.path.dirname(HERE), "lib")
LIB = os.path.join(LIB_DIR, "libpokerrl_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", HERE]

# translation unit -> extra flags.  The CFR sweeps must not contract multiply-adds (bit parity with numpy).
SOURCES = {
    "prl_common.cu": [],
    "cfr_levels.cu": ["-fmad=false"],
    "hand_eval.cu": [],
    "cfr_twocard.cu": [],
    "cfr_board.cu": ["--expt-relaxed-constexpr"],
    "env_kernels.cu": [],
    "lbr_rollout.cu": [],
    "allin_dense.cu": [],
    "h2h.cu": [],
}


def _stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    headers = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(ROOT, "include", "pokerrl_b200.h"))
    objs, rebuilt = [], False
    for src, extra in SOURCES.items():
        s = os.path.join(HERE, src)
        o = os.path.join(obj_dir, src.replace(".cu", ".o").replace(".cpp", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [NVCC] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            print(" ".join(cmd))
            subprocess.check_call(cmd)
            rebuilt = True
    if rebuilt or not os.path.exists(LIB):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs
        print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
