"""Build libvidar_b200.so in-tree with nvcc for sm_100a.

The library has no torch dependency (C ABI, include/vidar_b200.h): it is compiled
directly with nvcc and linked against the static CUDA runtime, so the built .so travels
with the repo snapshot to the GPU box.  `python -m vidar_b200.build` rebuilds it.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvidar_b200.so")
STAMP = os.path.join(HERE, ".libvidar_b200.stamp")

SOURCES = ["core.cu", "msda.cu", "linear_tc.cu", "dvr.cu", "latent_render.cu", "latent_proj.cu", "ray_head.cu", "sca_glue.cu", "knn.cu", "eval.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libvidar_b200.so)")


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest():
    h = hashlib.sha256()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]      # every included header
    files = _sources() + headers + [os.path.join(ROOT, "include", "vidar_b200.h")]
    for f in sorted(files):
        with open(f, "rb") as fh:
            h.update(os.path.relpath(f, ROOT).encode())      # machine-independent
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current():
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    try:
        with open(STAMP) as fh:
            return fh.read().strip() == _digest()
    except OSError:
        return False


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ into vidar_b200/libvidar_b200.so."""
    if not force and is_current():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    tmp = LIB + ".tmp"       # link next to the target, then rename: the library on disk is never half-written
    cmd = [nvcc, "-shared", "-o", tmp, *objs, "-cudart", "static",
           "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB)
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
