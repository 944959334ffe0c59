"""Builds libpn2_b200.so (sm_100a only) in-tree next to the sources.

    python build.py [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so travels with the tree (git-ignored, not gpurun-ignored).
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SOURCES = ["abi.cu", "fps.cu", "gather_group.cu", "ball_query.cu", "interpolate.cu", "lift.cu", "row_mlp.cu", "row_mlp_tc.cu", "train_mlp.cu", "grid.cu", "scatter_det.cu", "voxel.cu", "sphere.cu"]
SOURCES.append("scene_blocks.cu")  # whole-scene block tiling, sampling and votes
HEADERS = ["common.cuh", "row_mlp_tile.cuh", os.path.join(ROOT, "include", "pn2_abi.h")]
OUT = os.path.join(HERE, "libpn2_b200.so")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", HERE]


def _nvcc():
    """nvcc on PATH, else under CUDA_HOME (default /usr/local/cuda), so a login without the CUDA bin directory builds too."""
    return shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


def _digest(paths):
    h = hashlib.sha256()
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    hdrs = [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    obj_dir = os.path.join(HERE, "build")
    os.makedirs(obj_dir, exist_ok=True)
    hdr_digest = _digest(hdrs)

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.basename(src) + ".o")
        stamp = obj + ".sha"
        want = _digest([src]) + hdr_digest
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == want:
            return obj, False
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        with open(stamp, "w") as f:
            f.write(want)
        return obj, True

    with ThreadPoolExecutor(max_workers=8) as ex:
        results = list(ex.map(compile_one, srcs))
    objs = [o for o, _ in results]
    if force or any(changed for _, changed in results) or not os.path.exists(OUT):
        subprocess.check_call([_nvcc(), "-shared", "-Wno-deprecated-gpu-targets", "-o", OUT] + objs + ["-lcudart"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
