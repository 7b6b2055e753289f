"""Build libtwxi.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m topowx_b200.build [--force] [-v] [--prof]

The .so is git-ignored but travels to the GPU box with the repo snapshot.  nvcc cross-compiles without a GPU.
A build is skipped only when the stamp next to the library (SHA-256 over every source / header, the nvcc flags and the
nvcc version) matches, so a stale prebuilt library is never reused silently.
The rejected kriging variants of round 1 (one warp per problem, right-looking register-resident) are archived under
tools/experiments/ and are not part of the library.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtwxi.so")
SOURCES = ["api.cu", "knn.cu", "setup.cu", "ked.cu", "gwr.cu", "fixer.cu", "peak.cu", "vario.cu", "xval.cu", "record.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]          # never fast-math: FP64 parity


def _nvcc():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.isabs(p) and os.path.exists(p) or not os.path.isabs(p)):
            return p
    return "nvcc"


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stamp(flags, sources):
    h = hashlib.sha256()
    try:
        h.update(subprocess.check_output([_nvcc(), "--version"]))
    except Exception:
        h.update(b"nvcc?")
    h.update(" ".join(flags).encode())
    deps = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    deps = [os.path.join(CSRC, f) for f in deps] + [os.path.join(HERE, "..", "include", "twxi.h")]
    for d in deps:
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    h.update(" ".join(sources).encode())
    return h.hexdigest()


def needs_build(target=LIB, flags=None, sources=None):
    flags = NVCC_FLAGS if flags is None else flags
    sources = _sources() if sources is None else sources
    if not os.path.exists(target) or not os.path.exists(target + ".stamp"):
        return True
    with open(target + ".stamp") as f:
        return f.read().strip() != _stamp(flags, sources)


def build_lib(force=False, verbose=False, extra=(), out=None, tag=""):  # noqa: C901
    """extra/out/tag: instrumented developer builds (e.g. extra=["-DTWXI_KED_PROFILE"], out="libtwxi_prof.so")."""
    target = os.path.join(HERE, out) if out else LIB
    flags = NVCC_FLAGS + list(extra)
    sources = _sources()
    if not force and not needs_build(target, flags, sources):
        return target
    objs = []
    procs = []
    for src in sources:
        obj = os.path.join(CSRC, src.replace(".cu", tag + ".o"))
        cmd = [_nvcc()] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out_txt, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out_txt)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s" % src)
    cmd = [_nvcc(), "-shared", "-o", target] + objs + ["-lcudart"]
    subprocess.check_call(cmd)
    with open(target + ".stamp", "w") as f:
        f.write(_stamp(flags, sources))
    return target


if __name__ == "__main__":
    if "--prof" in sys.argv:
        print(build_lib(force=True, extra=["-DTWXI_KED_PROFILE"], out="libtwxi_prof.so", tag="_prof"))
    else:
        print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
