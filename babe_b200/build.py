"""Build libbabe_b200.so (sm_100a) in-tree with nvcc.

    python -m babe_b200.build [--force] [--verbose]

The shared library is a plain C-ABI (include/babe_b200.h); it links only
against the CUDA runtime.  It is git-ignored but travels to the GPU box with
the repository snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbabe_b200.so")
SOURCES = ["api.cu", "stft_ops.cu", "stft_fused.cu", "fit_ops.cu", "cqt_ops.cu", "net_ops.cu", "row_noise.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _source_hash():
    """Content hash of everything the library is built from (mtimes do not survive the
    snapshot copy to the GPU box; a spurious rebuild there would cost minutes)."""
    import hashlib
    h = hashlib.sha256()
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    files.append(os.path.join(ROOT, "include", "babe_b200.h"))
    for f in files:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()


def _stale():
    if not os.path.exists(LIB) or not os.path.exists(LIB + ".srchash"):
        return True
    return open(LIB + ".srchash").read().strip() != _source_hash()


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in _sources():
        obj = os.path.join(HERE, "build", os.path.basename(src) + ".o")
        cmd = [nvcc, "-O3", "-std=c++17", "-lineinfo", *ARCH, "-Xcompiler", "-fPIC",
               "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            failed = True
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-shared", *ARCH, "-o", LIB, *objs, "-lcudart"]
    subprocess.check_call(cmd)
    with open(LIB + ".srchash", "w") as f:
        f.write(_source_hash())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
