"""Build ``libhrp_b200.so`` (the C-ABI library declared in ``include/hrp.h``) in-tree with nvcc.

Run as ``python highway-rope-ppo_b200/build.py`` or through ``__graft_entry__.build()``.
sm_100a only; nvcc cross-compiles without a GPU present.
"""
from __future__ import annotations

import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libhrp_b200.so")
SOURCES = ["hrp_env.cu", "hrp_env_fast.cu", "hrp_api.cu", "hrp_ppo.cu", "hrp_mlp_tc.cu", "hrp_comm.cu", "hrp_episodes.cu",
           "hrp_norm.cu", "hrp_graph.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
# per-file additions.  hrp_env.cu: approximate fp32 division / sqrt and flush-to-zero in the fused step kernel --
# NOT --use_fast_math, which would also turn the sinf / cosf / sincosf of the embedding epilogue into SFU
# approximations that lose their error bound at the 2 pi angles RoPE / DistPE reach.  The epilogue's float32 operation
# order is kept by explicit __f*_rn intrinsics (exact whatever these flags say); the fp64 validation instantiation is
# not affected by them.  The PPO files stay IEEE.
# hrp_env_fast.cu is hrp_env.cu built with the highway-fast-v0 collision pass, so it takes the same flags.
EXTRA_FLAGS = {"hrp_env.cu": ["-ftz=true", "-prec-div=false", "-prec-sqrt=false"]}
EXTRA_FLAGS["hrp_env_fast.cu"] = EXTRA_FLAGS["hrp_env.cu"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = _sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(ROOT, "include", "hrp.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    base = [nvcc] + NVCC_FLAGS + ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    if os.environ.get("HRP_PHASE_CLOCKS") == "1":   # profiling build: per-phase SM clocks of the GEMM kernels (tools/gemm_one.py)
        base += ["-DHRP_PHASE_CLOCKS"]
    if verbose:
        base += ["-Xptxas", "-v"]
    jobs = []
    for src in _sources():   # one translation unit per process, in parallel
        name = os.path.basename(src)
        obj = os.path.join(obj_dir, name[:-3] + ".o")
        cmd = base + EXTRA_FLAGS.get(name, []) + ["-c", src, "-o", obj]
        jobs.append((name, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for name, obj, proc in jobs:
        out, _ = proc.communicate()
        if verbose or proc.returncode != 0:
            sys.stderr.write(out)
        failed |= proc.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libhrp_b200.so")
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-cudart", "static", "-o", LIB_PATH]
    res = subprocess.run(link + [obj for _, obj, _ in jobs], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed linking libhrp_b200.so")
    for _, obj, _ in jobs:   # the objects are intermediates: only the .so ships
        os.remove(obj)
    os.rmdir(obj_dir)
    return LIB_PATH


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
