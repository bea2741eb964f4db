"""Builds libsdr_b200/libsdrg.so (the C-ABI library, include/sdrg.h) in-tree with nvcc for sm_100a.

    python -m libsdr_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsdrg.so")
SOURCES = ["api.cu", "launch.cu", "design.cc", "iqbb_kernels.cu", "iqbb_warp_kernels.cu", "iqbb_fold_kernels.cu", "iqbb_fold_perwin.cu", "demod_kernels.cu",
           "fft_kernels.cu", "fft8k_kernels.cu", "conv8k_kernels.cu", "fft_general.cu", "fft_api.cu", "bank_kernels.cu", "bank_api.cu", "multi_gpu.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O3,-fwrapv,-fno-fast-math", "-shared", "-cudart", "static"]


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".hh"))] + \
           [os.path.join(HERE, "..", "include", "sdrg.h"), os.path.abspath(__file__)]


def _compile_flags(verbose=False):
    extra = os.environ.get("SDRG_NVCC_EXTRA", "").split()
    return [f for f in NVCC_FLAGS if f != "-shared"] + extra + (["-Xptxas", "-v"] if verbose else [])


def _stamp():
    return os.path.join(HERE, "..", "build", "obj", "flags.txt")


def needs_build():
    if not os.path.exists(OUT):
        return True
    if not os.path.exists(_stamp()) or open(_stamp()).read() != " ".join(_compile_flags()):
        return True                          # built with other flags (e.g. SDRG_NVCC_EXTRA)
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in sources() + _headers())


def build(force=False, verbose=False):
    """Every source is compiled to its own object (in parallel, and only when it or a header changed),
    then the objects are linked into libsdrg.so."""
    if not force and not needs_build():
        return OUT
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(HERE, "..", "build", "obj")
    os.makedirs(objdir, exist_ok=True)
    flags = _compile_flags(verbose)
    hdr_t = max(os.path.getmtime(h) for h in _headers())
    stamp = _stamp()
    same_flags = os.path.exists(stamp) and open(stamp).read() == " ".join(flags)

    def compile_one(src):
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        if not force and same_flags and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_t):
            return obj, None
        r = subprocess.run(["nvcc"] + flags + ["-c", src, "-o", obj], capture_output=True, text=True)
        return obj, r

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, sources()))
    for obj, r in results:
        if r is not None and r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed compiling " + obj)
        if r is not None and verbose:
            sys.stderr.write(r.stderr)
    open(stamp, "w").write(" ".join(flags))
    r = subprocess.run(["nvcc"] + NVCC_FLAGS + ["-o", OUT] + [o for o, _ in results], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libsdrg.so")
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(OUT)
