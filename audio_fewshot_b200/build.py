"""In-tree build of libafs_b200.so (the C-ABI library declared in include/afs_b200.h).

nvcc cross-compiles for sm_100a without a GPU; each .cu is compiled to an object
in parallel and linked into audio_fewshot_b200/_C/libafs_b200.so.  The .so is
git-ignored but travels to the GPU box with the repo snapshot.

    python -m audio_fewshot_b200.build [--force] [--verbose]
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
OUT_DIR = os.path.join(PKG_DIR, "_C")
LIB_PATH = os.path.join(OUT_DIR, "libafs_b200.so")
STAMP_PATH = os.path.join(OUT_DIR, "build.stamp")
INCLUDE = os.path.join(REPO_ROOT, "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "-I", INCLUDE, "-I", CSRC,
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build libafs_b200.so")
    return exe


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _fingerprint():
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    files = _sources() + sorted(
        os.path.join(d, f) for d in (CSRC, INCLUDE) for f in os.listdir(d) if f.endswith((".cuh", ".h"))
    )
    for p in files:
        h.update(p.encode())
        with open(p, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def is_current():
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP_PATH)):
        return False
    with open(STAMP_PATH) as fh:
        return fh.read().strip() == _fingerprint()


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library. Returns its path."""
    if not force and is_current():
        return LIB_PATH
    os.makedirs(OUT_DIR, exist_ok=True)
    nvcc = _nvcc()
    log_path = os.path.join(OUT_DIR, "ptxas.log")

    def compile_one(src):
        obj = os.path.join(OUT_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, _sources()))
    objs = []
    with open(log_path, "w") as log:
        for src, obj, r in results:
            log.write("==== %s\n%s\n%s\n" % (os.path.basename(src), r.stdout, r.stderr))
            if verbose:
                sys.stderr.write(r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s\n%s" % (src, r.stdout, r.stderr))
            objs.append(obj)
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-o", LIB_PATH, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(STAMP_PATH, "w") as fh:
        fh.write(_fingerprint())
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
