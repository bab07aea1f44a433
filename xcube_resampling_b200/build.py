"""In-tree build of ``libxrs.so`` (hand-written CUDA for sm_100a) with nvcc.

``python -m xcube_resampling_b200.build`` or ``__graft_entry__.build()``.
The shared object is written next to this file so that it travels with the
source tree; it is git-ignored (``*.so``).
"""

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
OBJ_DIR = os.path.join(HERE, "_obj")
LIB_PATH = os.path.join(HERE, "libxrs.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", 
          "--expt-relaxed-constexpr", f"-I{INCLUDE}", f"-I{CSRC}"]

# Per-file flags.  Kernels whose results are compared bit-for-bit with the
# reference's numba / numpy arithmetic are built without FMA contraction.
SOURCES = {
    "capi.cu": [],
    "rectify.cu": ["-fmad=false"],
    "rectify_ij.cu": ["-fmad=false"],
    "bands.cu": ["-fmad=false"],
    "coords.cu": ["-fmad=false"],
    "gather.cu": ["-fmad=false"],
    "gather_dual.cu": ["-fmad=false"],
    "resample.cu": ["-fmad=false"],
    "resample_fast.cu": ["-fmad=false"],
    "reproject.cu": [],  # projection math may contract; the numpy-parity part uses _rn intrinsics
    "decode.cu": [],  # CF scaling uses _rn intrinsics
}


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libxrs.so cannot be built")
    return exe


def _stamp(src: str, flags) -> str:
    h = hashlib.sha256()
    h.update(" ".join(flags).encode())
    for path in [src] + sorted(os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE) if f.endswith(".h")) + sorted(
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))
    ):
        with open(path, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _compile_one(nvcc, name, extra, verbose, obj_dir=None):
    src = os.path.join(CSRC, name)
    obj = os.path.join(obj_dir or OBJ_DIR, name.replace(".cu", ".o"))
    flags = ARCH + COMMON + extra
    stamp_path = obj + ".stamp"
    stamp = _stamp(src, flags)
    if os.path.exists(obj) and os.path.exists(stamp_path) and open(stamp_path).read() == stamp:
        return obj, False
    cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose and res.stderr:
        sys.stderr.write(res.stderr)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed for {name}:\n{res.stdout}\n{res.stderr}")
    with open(stamp_path, "w") as fh:
        fh.write(stamp)
    return obj, True


def build(verbose: bool = False, force: bool = False, variant: str | None = None, defines=()) -> str:
    """Compile and link ``libxrs.so``.  ``variant`` + ``defines`` (e.g. ``("-DXRS_K1_MINBLOCKS=3",)``) build
    an experimental ``libxrs_<variant>.so`` beside it (own object directory); ``XRS_LIB=<path>`` makes
    ``_lib.load()`` pick it up -- used to compare kernel variants in one GPU session."""
    nvcc = _nvcc()
    obj_dir = OBJ_DIR if not variant else OBJ_DIR + "_" + variant
    lib_path = LIB_PATH if not variant else os.path.join(HERE, f"libxrs_{variant}.so")
    os.makedirs(obj_dir, exist_ok=True)
    if force:
        for f in os.listdir(obj_dir):
            os.remove(os.path.join(obj_dir, f))
    present = {n: f + list(defines) for n, f in SOURCES.items() if os.path.exists(os.path.join(CSRC, n))}
    with ThreadPoolExecutor(max_workers=len(present)) as pool:
        results = list(pool.map(lambda kv: _compile_one(nvcc, kv[0], kv[1], verbose, obj_dir), present.items()))
    objs = [o for o, _ in results]
    changed = any(c for _, c in results)
    if changed or not os.path.exists(lib_path):
        cmd = [nvcc] + ARCH + ["-shared", "-Xcompiler", "-fPIC", "-o", lib_path] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return lib_path


if __name__ == "__main__":
    _variant = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")), None)
    _defines = tuple(a for a in sys.argv if a.startswith("-D"))
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv, variant=_variant, defines=_defines))
