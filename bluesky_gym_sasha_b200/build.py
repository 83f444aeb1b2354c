"""Builds libbsg_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m bluesky_gym_sasha_b200.build [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("BSG_LIB_OUT") or os.path.join(HERE, "libbsg_b200.so")      # BSG_LIB_OUT: A/B builds
SOURCES = ["api.cu", "env_step.cu", "cd_tiled.cu", "host_pool.cu", "obs_noise.cu", "traf_airspace.cu", "traf_events.cu", "render.cu", "cd_order.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "bsg.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])
    flags += os.environ.get("BSG_EXTRA_NVCC_FLAGS", "").split()
    if os.environ.get("BSG_LIB_OUT"):
        objdir = os.path.join(HERE, "build", "ab_" + os.path.basename(LIB))
        os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:                       # one nvcc per translation unit, in parallel
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        procs.append((src, obj, subprocess.Popen([nvcc] + flags + ["-c", "-o", obj, os.path.join(CSRC, src)],
                                                 stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libbsg_b200.so")
    # (the arch is named at the link step too: without it nvcc adds an empty default-arch stub cubin to the fat binary)
    res = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + [o for _, o, _ in procs] + ["-lcudart"],
                         capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("link of libbsg_b200.so failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
