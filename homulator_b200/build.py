"""In-tree build of the C-ABI library and the CLI with nvcc for sm_100a (no JIT cache, no torch extension).

    python -m homulator_b200.build        # or: from homulator_b200.build import build; build()

Outputs (git-ignored, shipped to the GPU box by gpurun):
    homulator_b200/libhomulator_b200.so   the C ABI declared in include/homulator_b200.h
    homulator_b200/Homulator.run          the drop-in CLI
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libhomulator_b200.so")
CLI = os.path.join(HERE, "Homulator.run")
CU = ["ntt.cu", "ewe.cu", "bconv_umma.cu", "context.cu", "hostpath.cu", "shard.cu", "replay.cu", "cli.cu"]
CPP = ["config.cpp", "params.cpp", "planner.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _newest_source():
    t = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            t = max(t, os.path.getmtime(os.path.join(root, f)))
    return t


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError("build failed: " + cmd[0])
    return r.stdout + r.stderr


def build(force=False, verbose=False):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        if os.path.exists(LIB):
            return LIB  # GPU box without a toolkit: use the prebuilt library that travelled with the snapshot
        raise RuntimeError("nvcc not found and no prebuilt libhomulator_b200.so")
    if not force and os.path.exists(LIB) and os.path.exists(CLI) and os.path.getmtime(LIB) >= _newest_source():
        return LIB
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    objs = []
    common = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
    procs = []
    for f in CU + CPP:
        o = os.path.join(bdir, f + ".o")
        objs.append(o)
        cmd = [nvcc] + ARCH + common + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, f), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + out)
            raise RuntimeError("build failed")
        if verbose:
            sys.stderr.write(out)
    _run([nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart", "-ldl"])
    _run([nvcc] + ARCH + common + [os.path.join(CSRC, "main.cpp"), "-o", CLI, "-L" + HERE, "-lhomulator_b200",
                                   "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
