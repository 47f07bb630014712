"""In-tree build of libh263cu.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m h263_rs_b200.build [--force] [--verbose]

Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   B200 only, no other targets, no PTX fallback
  -fmad=false                               the IDCT must not contract a*b+c (SURVEY.md T1)
  -lineinfo                                 so ncu's source page maps SASS to these files
The CUDA runtime is linked statically (nvcc default), so the library has no load-time
dependency on libcudart/libcuda and can be dlopen'ed on a machine without a GPU.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libh263cu.so")
SOURCES = ["kernels.cu", "recon_tile.cu", "deblock_tile.cu", "resample.cu", "resample_filter.cu", "parse_mb.cu", "context.cu", "frontend.cpp",
           "flv.cpp"]
# the synthetic stream generator is its own library (g++ only): test / benchmark tooling, not part of the decode path
SYNTH_OUT = os.path.join(HERE, "libh263synth.so")
SYNTH_DEPS = ["synth.cpp", "bitio.hpp", "vlc_codes.inc", os.path.join("..", "..", "include", "h263synth.h")]
DEPS = SOURCES + ["kernels.cuh", "parse_mb.h", "recon_common.cuh", "device_math.cuh", "bitio.hpp", "vlc_codes.inc", os.path.join("..", "..", "include", "h263cu.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def nvcc_cmd(extra=(), out=None):
    return [
        NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
        "-Xcompiler", "-fPIC,-O2,-pthread,-ffp-contract=off", "-shared", "-o", out or OUT,
        *[os.path.join(CSRC, s) for s in SOURCES], *extra,
    ]


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(os.path.join(CSRC, d)) <= t for d in DEPS)


def build_synth(force=False):
    if not force and os.path.exists(SYNTH_OUT) and all(
            os.path.getmtime(os.path.join(CSRC, d)) <= os.path.getmtime(SYNTH_OUT) for d in SYNTH_DEPS):
        return SYNTH_OUT
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-o", SYNTH_OUT, os.path.join(CSRC, "synth.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed: " + " ".join(cmd))
    return SYNTH_OUT


TOOL_SRC = os.path.join(HERE, "..", "tools", "single_stream_bench.cpp")
TOOL_OUT = os.path.join(HERE, "single_stream_bench.bin")


def build_tools(force=False):
    """The native single-stream driver bench.py runs for configs[1] (no interpreter in the loop)."""
    if not force and os.path.exists(TOOL_OUT) and os.path.getmtime(TOOL_OUT) >= max(os.path.getmtime(TOOL_SRC), os.path.getmtime(OUT)):
        return TOOL_OUT
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-o", TOOL_OUT, TOOL_SRC, "-L", HERE, "-lh263cu", "-Wl,-rpath," + HERE, "-ldl",
           "-pthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed: " + " ".join(cmd))
    return TOOL_OUT


def build(force=False, verbose=False):
    build_synth(force)
    out = _build_lib(force, verbose)
    build_tools(force)
    return out


def _build_lib(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    cmd = nvcc_cmd(["-Xptxas", "-v"] if verbose else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed: " + " ".join(cmd))
    return OUT


def build_variant(name, defines):
    """Side-by-side experiment builds: libh263cu_<name>.so with extra -D flags; select one at run
    time with H263CU_LIB=<path> (see _lib.py).  Not part of the product build."""
    out = os.path.join(HERE, "libh263cu_%s.so" % name)
    r = subprocess.run(nvcc_cmd(["-D" + d for d in defines], out), capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed for variant " + name)
    return out


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(OUT)
