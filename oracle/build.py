"""Build recipe for the oracle (test infrastructure, never shipped in the product path).

  python oracle/build.py            -> oracle/_build/liboracle.so   (CPU restatement, gcc)
  python oracle/build.py --ref      -> oracle/_ref/ref_cuda.so      (the reference's own four .cu files,
                                       compiled where they lie under /root/reference with the flags of
                                       utils/setup.py:19-20 (-O2), plus oracle/ref_shim.cu, our extern "C"
                                       forwarding shim that replaces only the THC-era .cpp glue)

The reference sources are never copied into this repository; --ref is a no-op when
/root/reference is absent (the GPU box uses the prebuilt oracle/_ref/ref_cuda.so).
"""
import hashlib
import os
import subprocess
import sys
import sysconfig
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = "/root/reference/utils/src"


def _newer(target, deps):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps if os.path.exists(d))


def build_oracle(force=False):
    """Rebuilds only when the source or the flags change (a content stamp, not mtimes, so a copied tree stays valid).
    When the tree is read-only and holds no current build, the library goes to a fresh temporary directory."""
    src = os.path.join(HERE, "pn2_oracle.c")
    # -ffp-contract=off: the only fused operations are the explicit fmaf() calls.
    # -mfma so fmaf() is one instruction; x86-64-v3 class hosts only.
    flags = ["-O2", "-std=c11", "-ffp-contract=off", "-mfma", "-mavx2", "-fopenmp", "-shared", "-fPIC"]
    with open(src, "rb") as f:
        h = hashlib.sha256(f.read())
    h.update(" ".join(flags).encode())
    want = h.hexdigest()
    out_dir = os.path.join(HERE, "_build")
    out = os.path.join(out_dir, "liboracle.so")
    stamp = out + ".sha"
    if not force and os.path.exists(out) and os.path.exists(stamp) and open(stamp).read() == want:
        return out
    try:
        os.makedirs(out_dir, exist_ok=True)
        writable = os.access(out_dir, os.W_OK)
    except OSError:
        writable = False
    if not writable:
        out_dir = tempfile.mkdtemp(prefix="pn2_oracle_")
        out = os.path.join(out_dir, "liboracle.so")
        stamp = out + ".sha"
    subprocess.check_call(["gcc"] + flags + [src, "-o", out, "-lm"])
    with open(stamp, "w") as f:
        f.write(want)
    return out


def build_ref(force=False):
    """Compile the reference's CUDA kernels verbatim for sm_100a (cross-compiles without a GPU)."""
    out_dir = os.path.join(HERE, "_ref")
    out = os.path.join(out_dir, "ref_cuda.so")
    if not os.path.isdir(REF_SRC):
        return out if os.path.exists(out) else None
    os.makedirs(out_dir, exist_ok=True)
    srcs = [os.path.join(REF_SRC, f) for f in
            ("sampling_gpu.cu", "ball_query_gpu.cu", "group_points_gpu.cu", "interpolate_gpu.cu")]
    shim = os.path.join(HERE, "ref_shim.cu")
    if not force and _newer(out, srcs + [shim]):
        return out
    import torch  # headers only: the reference's *_gpu.h include torch/ATen headers
    tinc = os.path.join(os.path.dirname(torch.__file__), "include")
    incs = ["-I", REF_SRC, "-I", tinc, "-I", os.path.join(tinc, "torch", "csrc", "api", "include"),
            "-I", sysconfig.get_paths()["include"]]
    objs = []
    procs = []
    for s in srcs + [shim]:
        o = os.path.join(out_dir, os.path.basename(s) + ".o")
        objs.append(o)
        cmd = ["nvcc", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-c", s, "-o", o] + incs
        procs.append(subprocess.Popen(cmd))
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed building the reference kernels")
    subprocess.check_call(["nvcc", "-shared", "-o", out] + objs + ["-lcudart"])
    for o in objs:
        os.remove(o)
    return out


if __name__ == "__main__":
    force = "--force" in sys.argv
    print(build_oracle(force))
    if "--ref" in sys.argv:
        print(build_ref(force))
