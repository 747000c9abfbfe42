"""Build libselfrec_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python -m selfrec_b200.build [--force] [--verbose]

The shared library has no torch dependency: plain `extern "C"` entry points declared in
include/selfrec_b200.h.  It is git-ignored but travels to the GPU box with the snapshot.
"""
import fcntl
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libselfrec_b200.so")
STAMP = os.path.join(HERE, "libselfrec_b200.stamp")  # no leading dot: it has to travel with the .so
LOCK = os.path.join(HERE, "libselfrec_b200.lock")

SOURCES = ["capi.cu", "spmm.cu", "bpr.cu", "infonce.cu", "score_topk.cu", "score_topk_tc.cu", "engine.cu", "sharded.cu", "graphbuild.cu", "sampler.cpp", "dataset.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall",
    "--shared",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libselfrec_b200.so)")


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, "selfrec_b200.h")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(os.path.relpath(f, ROOT).encode())  # not the absolute path: a moved tree keeps its build
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as fh:
        return fh.read().strip() != _digest()


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a into selfrec_b200/libselfrec_b200.so."""
    if not force and not needs_build():
        return LIB
    # several ranks of one job may get here at once: one builds, the others wait and find it done
    with open(LOCK, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    objs = []
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.rsplit(".", 1)[0] + ".o")
        objs.append(obj)
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
               "-Xcompiler", "-fPIC,-O3,-Wall", "-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"[selfrec_b200.build] {src} failed:\n{out}\n")
        elif verbose or out.strip():
            sys.stderr.write(f"[selfrec_b200.build] {src}:\n{out}\n")
    if failed:
        raise RuntimeError("nvcc failed; see messages above")
    tmp = LIB + f".tmp{os.getpid()}"
    link = [nvcc, "--shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout)
    os.replace(tmp, LIB)  # a process that already mapped the old library keeps its inode
    with open(STAMP + ".tmp", "w") as fh:
        fh.write(_digest())
    os.replace(STAMP + ".tmp", STAMP)
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
