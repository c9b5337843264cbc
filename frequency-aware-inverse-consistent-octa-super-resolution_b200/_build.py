"""Build ``libb200wave.so`` in-tree with nvcc for sm_100a.

    python -m b200wave._build            (or ``__graft_entry__.build()``)

The library is a plain C-ABI shared object (``include/b200wave.h``): no torch
headers, no pybind -- the Python side binds it with ctypes.  cudart is linked
statically so the ``.so`` loads on a box without a toolkit on the loader path
(and on the GPU-less build container for the symbol-export test).
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB_DIR = os.path.join(PKG_DIR, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libb200wave.so")
STAMP = os.path.join(LIB_DIR, "libb200wave.stamp")

SOURCES = ["api.cu", "dwt.cu", "dwt_stream_afb.cu", "dwt_stream_sfb.cu", "dwt_tma_afb.cu", "dwt_tma_sfb.cu", "dwt1d.cu", "swt.cu", "swt_inverse.cu", "ssim.cu", "ssim_f64.cu", "freq.cu", "tv.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
    "-cudart", "static",
]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def _source_hash():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files += [os.path.join(INCLUDE, f) for f in sorted(os.listdir(INCLUDE))]
    for f in files:
        with open(f, "rb") as fh:
            h.update(os.path.basename(f).encode())   # not the absolute path: the tree is copied to other machines
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_fresh():
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == _source_hash()


BOUNDS_LIB_PATH = os.path.join(LIB_DIR, "libb200wave_bounds.so")
# the sources compiled with -DB200W_BOUNDS: the kernels that run by default (stream, owner and TMA kernels)
BOUNDS_SOURCES = ["dwt_stream_afb.cu", "dwt_stream_sfb.cu", "dwt_tma_afb.cu", "dwt_tma_sfb.cu"]


def build_bounds(verbose=False):
    """The B200W_BOUNDS debug build (device-side bounds checks on every shared / global access of the DWT kernels, see
    csrc/common.cuh) as a second library, ``_lib/libb200wave_bounds.so``; used by tests through B200W_LIBRARY."""
    nvcc = find_nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found")
    os.makedirs(LIB_DIR, exist_ok=True)
    stamp = os.path.join(LIB_DIR, "libb200wave_bounds.stamp")
    want = _source_hash() + "+bounds"
    if os.path.exists(BOUNDS_LIB_PATH) and os.path.exists(stamp) and open(stamp).read().strip() == want:
        return BOUNDS_LIB_PATH
    build()   # the sources without checks (api, direct kernels, SSIM, ...) come from the regular build
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            path = _build_locked(nvcc, verbose, extra=["-DB200W_BOUNDS"], out_path=BOUNDS_LIB_PATH, suffix=".bounds.o",
                                 only=BOUNDS_SOURCES)
            with open(stamp, "w") as fh:
                fh.write(want)
            return path
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def build(force=False, verbose=False):
    """Compile every ``csrc/*.cu`` into ``_lib/libb200wave.so``; returns its path.  Safe against concurrent callers
    (one process per GPU under torchrun): an exclusive file lock serialises them and the library is moved into place
    atomically, so nobody ever loads a half-written file."""
    if not force and is_fresh():
        return LIB_PATH
    nvcc = find_nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libb200wave.so (set NVCC=/path/to/nvcc)")
    os.makedirs(LIB_DIR, exist_ok=True)
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and is_fresh():   # somebody else built it while we waited
                return LIB_PATH
            return _build_locked(nvcc, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(nvcc, verbose, extra=(), out_path=None, suffix=".o", only=None):
    objs = []
    procs = []
    for src in SOURCES:
        if only is not None and src not in only:   # a variant build reuses the regular object of this source
            objs.append(os.path.join(LIB_DIR, src.replace(".cu", ".o")))
            continue
        obj = os.path.join(LIB_DIR, src.replace(".cu", suffix))
        cmd = [nvcc] + NVCC_FLAGS + list(extra) + ["-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        if src == "api.cu":   # the binary carries the hash of the tree it was built from (b200w_build_hash)
            cmd.insert(1, '-DB200W_BUILD_HASH="%s"' % _source_hash())
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if verbose and out:
            print(out, file=sys.stderr)
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
    if out_path is not None:
        tmp = out_path + ".tmp.%d" % os.getpid()
        link = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                "-Xcompiler", "-fPIC", "-o", tmp] + objs
        res = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n%s" % res.stdout)
        os.replace(tmp, out_path)
        return out_path
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    link = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
            "-Xcompiler", "-fPIC", "-o", tmp] + objs
    res = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s" % res.stdout)
    os.replace(tmp, LIB_PATH)
    with open(STAMP, "w") as fh:
        fh.write(_source_hash())
    return LIB_PATH


if __name__ == "__main__":
    if "--bounds" in sys.argv:
        print(build_bounds(verbose="-v" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
