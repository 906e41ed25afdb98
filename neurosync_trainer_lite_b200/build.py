"""In-tree build of the CUDA library (``_lib/libnsf.so``) with nvcc for sm_100a.

``python -m neurosync_trainer_lite_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles
without a GPU; the resulting ``.so`` is git-ignored but travels to the GPU box with the snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libnsf.so")
SOURCES = ["nsf_plan.cpp", "nsf_kernels.cu", "nsf_autocorr_mma.cu", "nsf_stft_tc.cu", "nsf_convert.cu", "nsf_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xptxas=-v", "-Xcompiler", "-fPIC,-O3,-fvisibility=hidden",
    "-x", "cu", "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build neurosync_trainer_lite_b200/_lib/libnsf.so)")


def _digest():
    """Hash of the sources and flags.  Only file NAMES relative to the repo enter the hash (never the
    absolute path), so the library built in one checkout is recognised as current in a copy of it."""
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if not f.startswith(".")]
    files.append(os.path.join(ROOT, "include", "nsf.h"))
    for p in files:
        with open(p, "rb") as fh:
            h.update(os.path.relpath(p, ROOT).replace(os.sep, "/").encode() + b"\0" + fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _is_current(stamp, digest):
    if not (os.path.exists(LIB_PATH) and os.path.exists(stamp)):
        return False
    with open(stamp) as fh:
        return fh.read().strip() == digest


def build(force=False, verbose=False):
    """Build (if the stamp does not match the sources) and return the library path.

    Safe under concurrent callers (torchrun starts one process per GPU): an exclusive file lock
    serialises builders, objects and the shared library are written under temporary names and moved into
    place with an atomic rename, so no process can ever dlopen a half-written file."""
    import fcntl
    import tempfile
    os.makedirs(LIB_DIR, exist_ok=True)
    stamp = os.path.join(LIB_DIR, "libnsf.sha256")
    digest = _digest()
    if not force and _is_current(stamp, digest):
        return LIB_PATH
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _is_current(stamp, digest):      # another process built it while we waited
                return LIB_PATH
            tmp = tempfile.mkdtemp(prefix=".build-", dir=LIB_DIR)
            try:
                from concurrent.futures import ThreadPoolExecutor

                def compile_one(src):
                    obj = os.path.join(tmp, os.path.splitext(src)[0] + ".o")
                    cmd = [_nvcc(), *NVCC_FLAGS, "-I", os.path.join(ROOT, "include"), "-I", CSRC,
                           "-DNSF_BUILDING=1", "-c", os.path.join(CSRC, src), "-o", obj]
                    res = subprocess.run(cmd, capture_output=True, text=True)
                    return src, obj, cmd, res

                objs = []
                with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
                    for src, obj, cmd, res in pool.map(compile_one, SOURCES):     # translation units in parallel
                        if verbose or res.returncode != 0:
                            sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
                        if res.returncode != 0:
                            raise RuntimeError(f"nvcc failed on {src}")
                        objs.append(obj)
                lib_tmp = os.path.join(tmp, "libnsf.so")
                cmd = [_nvcc(), "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                       "-o", lib_tmp, *objs]
                res = subprocess.run(cmd, capture_output=True, text=True)
                if res.returncode != 0:
                    sys.stderr.write(res.stdout + res.stderr)
                    raise RuntimeError("link failed")
                if os.path.exists(stamp):
                    os.remove(stamp)                          # never leave a stamp that vouches for an older library
                os.replace(lib_tmp, LIB_PATH)                 # atomic within the directory
                for obj in objs:                              # keep the objects next to the library (cuobjdump / ptxas notes)
                    os.replace(obj, os.path.join(LIB_DIR, os.path.basename(obj)))
                stamp_tmp = os.path.join(tmp, "libnsf.sha256")
                with open(stamp_tmp, "w") as fh:
                    fh.write(digest)
                os.replace(stamp_tmp, stamp)
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
