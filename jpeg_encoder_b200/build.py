"""Builds libjpegenc_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import glob
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libjpegenc_b200.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "-shared",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cpp")))


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CSRC, "*.inc")) + glob.glob(os.path.join(PKG, "..", "include", "*.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra=()):
    """Compile every CUDA source for sm_100a into one shared library. nvcc cross-compiles without a GPU."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    bdir = os.path.join(PKG, "build")
    os.makedirs(bdir, exist_ok=True)
    for s in sources():
        o = os.path.join(bdir, os.path.basename(s) + ".o")
        objs.append(o)
        cmd = [nvcc, "-c", s, "-o", o] + [f for f in NVCC_FLAGS if f != "-shared"] + list(extra)
        if verbose:
            print(" ".join(cmd))
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    failed = False
    for s, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed on %s:\n%s\n" % (s, out))
        elif verbose and out.strip():
            print(out)
    if failed:
        raise RuntimeError("nvcc build failed")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
