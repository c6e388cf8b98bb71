"""Build libjaero_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libjaero_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math"]
# (source, extra flags). The demodulator kernels keep IEEE mul/add separate so that double arithmetic
# rounds exactly as the CPU reference does (x86-64 has no implicit FMA contraction).
UNITS = [
    ("capi.cu", []),
    ("capi_batch.cu", []),
    ("capi_burst.cu", []),
    ("capi_frames.cu", []),
    ("capi_ingest.cu", []),
    ("host_design.cpp", []),                 # host C++ only: nvcc hands it to the host compiler with the flags above
    ("viterbi.cu", []),
    ("cfe.cu", []),
    ("pchannel.cu", []),
    ("rtchannel.cu", []),
    ("cchannel.cu", []),
    ("reassembly.cu", []),
    ("channelizer.cu", []),                  # restates no reference arithmetic: FMA contraction is allowed
    ("prefilter.cu", ["-fmad=false"]),
    ("burst.cu", ["-fmad=false"]),
    ("demod_kernels.cu", ["-fmad=false"]),
]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    objdir = os.path.join(HERE, "_obj")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".cu", ".cpp"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "jaero_b200.h"))
    objs = []
    for src, extra in UNITS:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        if force or _stale(obj, hdrs):
            cmd = [NVCC] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError("nvcc failed for " + src)
    if force or _stale(OUT, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", OUT] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
