"""TEST INFRASTRUCTURE ONLY -- builds the *unmodified* reference CPU engines into oracle/_ref/.

Compiles the reference's own C++ sources where they lie under /root/reference (nothing is
copied into this repository) with torch.utils.cpp_extension, following the reference's
src/CMakeLists.txt target lists:

  cpp_ctc_loss     <- src/CMakeLists.txt:16-25  (losses/ctc_loss.cpp, ctc_loss_py.cpp,
                      forward_backward.cpp + utils)
  cpp_ctc_decoder  <- src/CMakeLists.txt:41-51  (decoders/ctc_decoder.cpp, ctc_decoder_py.cpp
                      + utils + the query-only KenLM file set of
                      third_party/kenlm/compile_query_only.sh)

The stock CMake build is not used (it requires Boost and C++14, neither usable with this
image's torch 2.11); see DESIGN.md "Oracle".  Outputs go only to oracle/_ref/ (git-ignored,
shipped to the GPU box by gpurun).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may load what this script produces.
"""
import glob
import os
import sys

REF = os.environ.get("E2E_REFERENCE_ROOT", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def _kenlm_sources(k):
    srcs = []
    for pat in ("util/double-conversion/*.cc", "util/*.cc", "lm/*.cc"):
        srcs += glob.glob(os.path.join(k, pat))
    return sorted(s for s in srcs if not (s.endswith("test.cc") or s.endswith("main.cc")))


def build(which=("loss", "decoder"), verbose=False):
    if not os.path.isdir(os.path.join(REF, "src")):
        raise RuntimeError("reference sources not present at %s" % REF)
    from torch.utils.cpp_extension import load
    R = os.path.join(REF, "src")
    K = os.path.join(REF, "third_party", "kenlm")
    built = []
    if "loss" in which:
        d = os.path.join(OUT, "loss")
        os.makedirs(d, exist_ok=True)
        load(name="cpp_ctc_loss",
             sources=[R + "/losses/ctc_loss.cpp", R + "/losses/ctc_loss_py.cpp",
                      R + "/losses/forward_backward.cpp", R + "/utils/threadpool.cpp",
                      R + "/utils/math_utils.cpp"],
             extra_include_paths=[R], extra_cflags=["-O3"], build_directory=d,
             verbose=verbose, is_python_module=False)
        built.append(d)
    if "decoder" in which:
        d = os.path.join(OUT, "decoder")
        os.makedirs(d, exist_ok=True)
        load(name="cpp_ctc_decoder",
             sources=[R + "/decoders/ctc_decoder.cpp", R + "/decoders/ctc_decoder_py.cpp",
                      R + "/utils/threadpool.cpp", R + "/utils/math_utils.cpp"] + _kenlm_sources(K),
             extra_include_paths=[R, K],
             extra_cflags=["-O3", "-DKENLM_MAX_ORDER=6", "-DHAVE_ZLIB", "-DNDEBUG", "-w"],
             extra_ldflags=["-lz"], build_directory=d, verbose=verbose, is_python_module=False)
        built.append(d)
    # keep only what must travel to the GPU box
    for d in built:
        for f in os.listdir(d):
            if f.endswith(".o") or f.startswith(".ninja"):
                os.remove(os.path.join(d, f))
    return built


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
