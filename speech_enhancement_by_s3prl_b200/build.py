"""Build ``libse_b200.so`` in-tree with nvcc for sm_100a (no torch / libtorch linkage).

``python -m speech_enhancement_by_s3prl_b200.build`` or ``build_library()``.  The shared
object is written next to this file so that it travels with the source tree; it is
rebuilt when any file under ``csrc/`` or ``include/`` is newer than the library.
"""
import glob
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libse_b200.so")
HASH_PATH = LIB_PATH + ".sha256"
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libse_b200.so cannot be built (there is no CPU fallback)")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def source_hash():
    """sha256 over csrc/ and include/ (file names + contents): mtimes do not survive the copy to the GPU box."""
    import hashlib
    h = hashlib.sha256()
    for path in sorted(glob.glob(os.path.join(CSRC, "*")) + glob.glob(os.path.join(ROOT, "include", "*.h"))):
        if os.path.isfile(path):
            h.update(os.path.basename(path).encode())
            with open(path, "rb") as f:
                h.update(f.read())
    return h.hexdigest()


def is_stale():
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != source_hash()


def build_library(force=False, verbose=False, extra_flags=(), out_path=None):
    """extra_flags / out_path: experiment builds (e.g. -DSE_GEO512_K3_MINB=1 into another file, loaded via SE_B200_LIB)."""
    if out_path is None and not force and not is_stale():
        return LIB_PATH
    build_dir = os.path.join(PKG_DIR, "build")
    os.makedirs(build_dir, exist_ok=True)
    # one builder at a time (every rank of a torchrun job may find the library stale at once); the others wait here and
    # then find it fresh
    import fcntl
    with open(os.path.join(build_dir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if out_path is None and not force and not is_stale():
                return LIB_PATH
            return _build_locked(build_dir, verbose, extra_flags, out_path)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _object_key(src, extra_flags):
    """Hash of one translation unit's inputs: the source, every header of csrc/ and include/, and the flags."""
    import hashlib
    h = hashlib.sha256(" ".join(extra_flags).encode())
    deps = [src] + sorted(glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) +
                          glob.glob(os.path.join(ROOT, "include", "*.h")))
    for path in deps:
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def _build_locked(build_dir, verbose, extra_flags, out_path):
    """Compile the translation units whose inputs changed (objects are cached by content hash) and link."""
    nvcc = _nvcc()
    objs, procs = [], []
    for src in sources():
        stem = os.path.basename(src)[:-3]
        obj = os.path.join(build_dir, f"{stem}.{_object_key(src, extra_flags)}.o")
        objs.append(obj)
        if os.path.exists(obj) and not verbose:
            continue
        for old in glob.glob(os.path.join(build_dir, f"{stem}.*.o")):
            os.remove(old)
        tmp = f"{obj}.{os.getpid()}.tmp"
        cmd = [nvcc, *ARCH_FLAGS, "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", *extra_flags,
               "-I", os.path.join(ROOT, "include"), "-c", src, "-o", tmp]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, tmp, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = None
    for src, tmp, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            failed = failed or src
            if os.path.exists(tmp):
                os.remove(tmp)
        else:
            os.replace(tmp, obj)
    if failed:
        raise RuntimeError(f"nvcc failed on {failed}")
    target = out_path or LIB_PATH
    tmp = f"{target}.{os.getpid()}.tmp"
    subprocess.check_call([nvcc, *ARCH_FLAGS, "-shared", "-o", tmp, *objs, "-lcudart"])
    os.replace(tmp, target)
    if out_path is None:
        with open(HASH_PATH, "w") as f:
            f.write(source_hash())
    return target


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
