"""Builds the in-tree native libraries.

  libmcb200.so            the product: C ABI (include/mcb.h) + sm_100a kernels (csrc/*.cu, csrc/*.cpp)
  (oracle/ is built by oracle/Makefile; see __graft_entry__.build)

nvcc cross-compiles for sm_100a without a GPU.  Flags that matter for parity with the reference's fp32 arithmetic:
  -fmad=false          no FMA contraction of a*b+c (the oracle is built with -ffp-contract=off, SURVEY.md A.2)
  default -prec-div=true -prec-sqrt=true -ftz=false (never --use_fast_math)
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmcb200.so")
SOURCES = ["mcb_api.cu", "mcb_lower.cpp", "mcb_jit.cpp"]
HEADERS = [os.path.join("..", "..", "tools", "headless_main.cpp"), os.path.join("..", "..", "include", "marching.h"),
           os.path.join("..", "..", "include", "evaluator.h"), "mcb_kernels.cuh", "mcb_jit.h", "mcb_bytecode.h", "mcb_pow.h", "mcb_trig.h", "mcb_interval.h", "mcb_tables.h", "mcb_tri_words.inc", "mcb_lower.h",
           os.path.join("..", "..", "include", "mcb.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
         "-Xcompiler", "-fPIC,-O2,-ffp-contract=off", "--shared", "-cudart", "shared"]


def stale():
    if not os.path.exists(LIB) or not os.path.exists(os.path.join(HERE, "mcb_headless")):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS) or os.path.getmtime(__file__) > t


def source_stamp():
    """sha256 over every source the library is built from, in a fixed order (mcb_build_stamp() returns it)."""
    import hashlib
    h = hashlib.sha256()
    names = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".cpp", ".h")) or f == "mcb_tri_words.inc")
    for f in names + [os.path.join("..", "..", "include", "mcb.h")]:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    stamp = source_stamp()
    stamp_file = os.path.join(CSRC, "mcb_build_stamp.inc")
    old = open(stamp_file).read() if os.path.exists(stamp_file) else ""
    if old != '"%s"\n' % stamp:
        with open(stamp_file, "w") as o:
            o.write('"%s"\n' % stamp)
        force = True  # a source changed since the library was built, whatever the mtimes say
    if not force and not stale():
        return LIB
    # mcb_pow.h, mcb_trig.h and mcb_bytecode.h also travel inside the library as text: the run-time compiled evaluator
    # (mcb_jit.cpp) includes them through NVRTC
    for name, inc, tag in (("mcb_pow.h", "mcb_pow_src.inc", "MCBPOWSRC"), ("mcb_trig.h", "mcb_trig_src.inc", "MCBTRIGSRC"),
                           ("mcb_bytecode.h", "mcb_bytecode_src.inc", "MCBBCSRC")):
        with open(os.path.join(CSRC, name)) as f, open(os.path.join(CSRC, inc), "w") as o:
            o.write('R"%s(' % tag + f.read() + ')%s"\n' % tag)
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building libmcb200.so")
    build_headless()
    return LIB


def build_headless():
    """mcb_headless: the reference's main.cpp wiring without the GUI (tools/headless_main.cpp), on the C++ drop-in headers."""
    root = os.path.dirname(HERE)
    exe = os.path.join(HERE, "mcb_headless")
    cmd = [os.environ.get("CXX", "g++"), "-std=c++14", "-O2", "-Wall", "-I", os.path.join(root, "include"),
           os.path.join(root, "tools", "headless_main.cpp"), "-o", exe, "-L", HERE, "-lmcb200", "-Wl,-rpath,$ORIGIN", "-pthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building mcb_headless")
    return exe


if __name__ == "__main__":
    build(force=True, verbose="-v" in sys.argv)
    print(LIB)
