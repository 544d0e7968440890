"""Build libe2e_ctc.so (the sm_100a CUDA kernels + the C ABI of include/e2e_ctc.h) in-tree.

    python -m end2end_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so lands in end2end_b200/lib/ (git-ignored, shipped to
the GPU box by gpurun).  The CUDA runtime is linked statically, so the library has no torch or
libcudart dependency: any host language can dlopen it.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libe2e_ctc.so")
SOURCES = ["api.cu", "comm.cu", "ctc_rowstats.cu", "ctc_fused_a.cu", "ctc_fused_b.cu", "ctc_fused_c.cu",
           "ctc_wave_a.cu", "ctc_wave_b.cu", "ctc_sweep_a.cu", "ctc_sweep_b.cu", "ctc_sweep_c.cu", "ctc_sweep_d.cu",
           "ctc_grad.cu", "ctc_greedy.cu", "ctc_viterbi.cu", "ctc_noblank.cu", "ctc_beam.cu",
           "ctc_score.cu", "edit_distance.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.sep not in c or os.path.exists(c)):
            return c
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra=(), tag=None):
    """``tag``: an experiment build (own object directory, lib/libe2e_ctc_<tag>.so; load it with E2E_CTC_LIB=<path>)."""
    objdir = os.path.join(OBJDIR, tag) if tag else OBJDIR
    lib = os.path.join(LIBDIR, "libe2e_ctc_%s.so" % tag) if tag else LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "ctc_fused_impl.cuh"), os.path.join(CSRC, "ctc_sweep_impl.cuh"), os.path.join(CSRC, "ctc_wave_impl.cuh"),
               os.path.join(HERE, "..", "include", "e2e_ctc.h")]
    nvcc = _nvcc()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append([nvcc, *ARCH, *FLAGS, *extra, *os.environ.get("E2E_BUILD_EXTRA", "").split(), "-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stdout + r.stderr))
        if verbose and (r.stdout or r.stderr):
            print(r.stdout + r.stderr)

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        list(ex.map(run, jobs))
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(lib, objs):
        run([nvcc, *ARCH, "-shared", "-o", lib, *objs, "-ldl"])
    return lib


if __name__ == "__main__":
    _tag = sys.argv[sys.argv.index("--tag") + 1] if "--tag" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv,
                extra=("-Xptxas", "-v") if "--ptxas" in sys.argv else (), tag=_tag))
