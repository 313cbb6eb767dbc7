"""Build the native library (nvcc, sm_100a) in-tree: mujoco_rl_manipulate_unknown_objects_b200/libgripper_sim_b200.so.

The build container has no GPU; nvcc cross-compiles.  The .so is git-ignored but travels to the GPU box with the
repository snapshot.  `python -m mujoco_rl_manipulate_unknown_objects_b200.build` rebuilds when a source is newer.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgripper_sim_b200.so")
SOURCES = ["gripper_sim.cu", "policy_kernels.cu", "train_kernels.cu", "replay_kernels.cu", "mjcf_compiler.cpp", "dev_model.cpp"]
HEADERS = ["model.h", "sim_kernels.cuh", "env_kernels.cuh", "env_lockstep.cuh", "render_kernels.cuh",
           os.path.join("..", "..", "include", "b200_gripper_sim.h")]
# -prec-div=false / -prec-sqrt=false / -ftz=true: divisions and square roots are the hardware's 2-ulp approximations and
# denormals flush to zero.  The physics kernel divides and normalises on every dependent chain (quaternions, contact frames,
# Cholesky pivots, the MPR portal), and the IEEE-exact sequences (~8 instructions + a slow path each) were 12 % of the step
# (profiles/r2k_flags.log: 18.9 -> 21.2 M substeps/s); every parity test passes unchanged with them.  NOT -use_fast_math: its
# sin/cos/pow intrinsics change trajectories beyond the parity bounds (8 tests fail).
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "-shared", "-diag-suppress", "550,177", "-prec-div=false", "-prec-sqrt=false", "-ftz=true"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    files = [os.path.join(CSRC, f) for f in SOURCES + HEADERS if os.path.exists(os.path.join(CSRC, f))] + [os.path.abspath(__file__)]  # the flags live here
    return any(os.path.getmtime(f) > t for f in files)


LAST_BUILD = {"compiled": [], "reused": [], "nvcc_s": 0.0, "flags": []}  # what the last build_native() call did


def build_native(force=False, verbose=False):
    """Compiles the library when a source is newer than it (or force=True, or GRAFT_FORCE_BUILD=1 in the environment).
    LAST_BUILD records what happened: sources compiled, artefacts reused, seconds spent in nvcc."""
    import time
    force = force or os.environ.get("GRAFT_FORCE_BUILD", "") not in ("", "0")
    srcs = [os.path.join(CSRC, f) for f in SOURCES if os.path.exists(os.path.join(CSRC, f))]
    LAST_BUILD.update(compiled=[], reused=[], nvcc_s=0.0, flags=NVCC_FLAGS)
    if not force and not needs_build():
        LAST_BUILD["reused"] = [os.path.relpath(LIB, os.path.dirname(HERE))]
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB + ".tmp"] + srcs
    t0 = time.perf_counter()
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    LAST_BUILD["nvcc_s"] = round(time.perf_counter() - t0, 2)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout)
    if verbose:
        print(r.stdout)
    os.replace(LIB + ".tmp", LIB)
    LAST_BUILD["compiled"] = [os.path.relpath(f, os.path.dirname(HERE)) for f in srcs]
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
