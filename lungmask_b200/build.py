"""Builds lungmask_b200/liblungmask_b200.so (sm_100a only) with nvcc, in-tree.

    python -m lungmask_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "liblungmask_b200.so")
SOURCES = ["conv_tc.cu", "forward_misc.cu", "preproc.cu", "postproc.cu", "shard.cu", "engine.cu", "decode.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "lungmask_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=True):
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, out))
        if verbose and out.strip():
            print(out)
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
