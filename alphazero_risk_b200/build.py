"""Builds libaz_b200.so (the CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python -m alphazero_risk_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(PKG, "_obj")
LIB = os.path.join(PKG, "libaz_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]
# per translation unit flags: the game / tree code must round exactly like the reference's
# x86 build (no FMA contraction); the network kernels may fuse.
# A unit may include another .cu whose bytes must stay as they are (profiles/traffic.json keys its ncu captures by source hashes):
# INCLUDED lists those files, so that a change to them rebuilds the unit.
UNITS = {
    "az_env_rollout.cu": ["-fmad=false"],    # az_env.cu (included unchanged) + the rollout with the land bytes kept in the pool slot
    "az_mcts_value6.cu": ["-fmad=false"],    # az_mcts.cu (included unchanged) + az_mcts_create's six-output check
    "az_nn.cu": [],
    "az_nn_tc_value6.cu": [],                # az_nn_tc.cu (included unchanged) + the six-output value tail
    "az_tc_gemm.cu": [],
    "az_nn_train.cu": ["-fmad=false"],   # training step: plain fp32, same roundings whatever the compiler would contract
    "az_ckpt.cpp": [],       # host only: TensorFlow V2 checkpoint bundles
    "az_env6.cu": ["-fmad=false"],   # six-player extension of the environment (SIXPLAYER.md), integer only
    "az_mcts6.cu": ["-fmad=false"],  # six-player search: reference roundings (no FMA contraction), like az_mcts.cu
    "az_dist.cu": [],        # NCCL weight broadcast + statistics gather (NCCL itself is dlopen'ed at run time)
}


INCLUDED = {"az_env_rollout.cu": ["az_env.cu"], "az_mcts_value6.cu": ["az_mcts.cu"], "az_nn_tc_value6.cu": ["az_nn_tc.cu"]}


def _newer(src_files, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_files)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers += [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    objs, procs = [], []
    for unit, extra in UNITS.items():
        src = os.path.join(CSRC, unit)
        if not os.path.exists(src):
            continue
        obj = os.path.join(OBJ, os.path.splitext(unit)[0] + ".o")
        objs.append(obj)
        if force or _newer([src] + [os.path.join(CSRC, f) for f in INCLUDED.get(unit, [])] + headers, obj):
            cmd = [nvcc] + ARCH + COMMON + extra + os.environ.get("AZ_B200_NVCC_FLAGS", "").split() + \
                  (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((unit, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for unit, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- %s\n%s\n" % (unit, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or not os.path.exists(LIB):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcuda", "-ldl"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
