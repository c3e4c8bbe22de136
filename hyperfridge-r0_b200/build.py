"""In-tree build of libhfb200.so for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libhfb200.so")
SOURCES = ["hfb200.cu"]
DEPS = ["hfb200.cu", "prover.cuh", "ntt.cuh", "ntt_tma.cuh", "ntt_mid.cuh", "transcript.cuh", "poseidon2.cuh", "poseidon2_consts.inc", "circuit.cuh", "deep.cuh", "dev.cuh", "blind.cuh", "field.cuh", "probe.cuh", "jit.cuh", "verify.cuh", "hal.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-ldl"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build_cuda(force=False, verbose=False):
    deps = [os.path.join(CSRC, d) for d in DEPS] + [os.path.join(ROOT, "include", "hfb200.h")]
    if not force and not is_stale(OUT, deps):
        return OUT
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return OUT


def build_emu(force=False):
    """Host emulator of the same kernel sources (tests/emu only; never loaded by the product)."""
    out = os.path.join(ROOT, "tests", "emu", "libhfb200_emu.so")
    deps = [os.path.join(CSRC, d) for d in DEPS] + [os.path.join(ROOT, "include", "hfb200.h")]
    if not force and not is_stale(out, deps):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-x", "c++", "-DHFB200_EMU", "-O2", "-std=c++17", "-fPIC", "-fopenmp", "-Wno-unknown-pragmas",
           "-I/usr/local/cuda/include", "-shared", "-o", out, os.path.join(CSRC, "hfb200.cu")]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    print(build_cuda(force=True, verbose=True))
