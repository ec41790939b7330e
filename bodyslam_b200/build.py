"""In-tree build of libbodyslam_b200.so (nvcc, sm_100a only).

`python -m bodyslam_b200.build` or `bodyslam_b200.build.build()`.  The shared object lands next
to this file so that it travels with the repo snapshot to the GPU box (it is git-ignored).
-fmad=false: the TSDF and percentile arithmetic must round exactly like the CPU oracle, which is
compiled with -ffp-contract=off; every kernel here is HBM-bound, so contraction buys nothing.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbodyslam_b200.so")
SOURCES = ["bslam_tsdf.cu", "bslam_image.cu", "bslam_colorize_f32.cu", "bslam_extract.cu", "bslam_vbg.cu", "bslam_raycast.cu", "bslam_odometry.cu",
           "bslam_mesh_raycast.cu"]


def nvcc_path() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found (needed to build libbodyslam_b200.so)")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "bodyslam_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    host_cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
           "-fmad=false", "-shared", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-ccbin", host_cxx,
           "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", LIB]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
