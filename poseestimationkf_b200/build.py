"""Builds poseestimationkf_b200/libposekf_b200.so for sm_100a with nvcc (in-tree, so that the
library travels with the repository snapshot).  `python -m poseestimationkf_b200.build [--force]`.
The translation units (one device module each) compile in parallel into a temporary directory and are then linked."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libposekf_b200.so")
SOURCES = [os.path.join(CSRC, f) for f in ("posekf_capi.cu", "replay_general_innovation.cu")]
DEPENDS = SOURCES + [os.path.join(CSRC, f) for f in ("ekf_math.cuh", "device_util.cuh", "replay_kernels.cuh", "ops_kernels.cuh",
                                                     "replay_launch.cuh")] + [
    os.path.join(PKG_DIR, "..", "include", "posekf.h")]

# -fmad=false: only the explicit fma_() calls of ekf_math.cuh fuse.  The scalar kernels, the packed (f32x2
# intrinsics, never contracted) kernels and the g++ -ffp-contract=off host build then execute the same
# roundings, which is what makes their results bit-identical.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false", "--shared",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build the sm_100a library (there is no CPU fallback)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in DEPENDS)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile if the library is missing or older than its sources; returns the library path."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    compile_flags = [f for f in NVCC_FLAGS if f != "--shared"]
    with tempfile.TemporaryDirectory(prefix="posekf_build_") as tmp:
        objs = [os.path.join(tmp, os.path.basename(src) + ".o") for src in SOURCES]
        cmds = [[nvcc] + compile_flags + ["-c", "-o", obj, src] for src, obj in zip(SOURCES, objs)]
        procs = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for cmd in cmds]
        outs = [p.communicate()[0] for p in procs]
        link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-o", LIB_PATH] + objs
        ok = all(p.returncode == 0 for p in procs)
        if ok:
            lp = subprocess.run(link, capture_output=True, text=True)
            ok = lp.returncode == 0
            outs.append(lp.stdout + lp.stderr)
            cmds.append(link)
    log = "".join(" ".join(c) + "\n" + o for c, o in zip(cmds, outs))
    with open(os.path.join(PKG_DIR, "build_ptxas.log"), "w") as fh:
        fh.write(log)
    if not ok:
        raise RuntimeError("nvcc failed:\n" + log)
    if verbose:
        print(log)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
