"""In-tree build of the native libraries (nvcc, sm_100a only).

  lib/libb747_b200.so  the batched C ABI (include/b747.h)
  lib/model_simple.so  the reference's scalar boundary (include/b747_scalar.h), self-contained so
                       that it can be copied per Model instance like the reference does
  lib/model.so         the boundary of the legacy core/model_win64.dll (include/b747_scalar_legacy.h)

nvcc cross-compiles without a GPU; the .so files are git-ignored but travel with the tree.
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
# translation unit -> extra flags.  The f64 parity kernels are built without FMA contraction:
# the reference DLL is SSE2 code that rounds every product and sum separately.
UNITS = {
    "b747_kernels_f64.cu": ["-fmad=false"],
    # throughput kernels: approximate (1-2 ulp) float32 division / sqrt; float64 ops unaffected
    "b747_kernels_f32.cu": ["-prec-div=false", "-prec-sqrt=false"],
    "b747_capi.cu": [],
    "b747_state.cu": [],
    "b747_env_params.cu": [],
    "b747_scalar.cu": [],
    "b747_scalar_legacy.cu": [],
}
HEADERS = ["b747_common.cuh", "b747_kernels.h", "b747_model_f64.cuh", "b747_model_mx.cuh", "b747_poly.h", "b747_tables.h",
           "../../include/b747.h", "../../include/b747_params.h", "../../include/b747_scalar.h",
           "../../include/b747_scalar_legacy.h"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the native extension cannot be built")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_native(force=False, verbose=False):
    nvcc = _nvcc()
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs = {}
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        objs[src] = o
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + ARCH + COMMON + extra + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
    core = [objs[k] for k in ("b747_kernels_f64.cu", "b747_kernels_f32.cu", "b747_capi.cu", "b747_state.cu",
                             "b747_env_params.cu")]
    lib = os.path.join(LIBDIR, "libb747_b200.so")
    if force or _stale(lib, core):
        subprocess.run([nvcc] + ARCH + ["-shared", "-o", lib] + core + ["-Xlinker", "-Bsymbolic", "-lcudart_static", "-lpthread", "-ldl", "-lrt"],
                       check=True)
    scal = os.path.join(LIBDIR, "model_simple.so")
    if force or _stale(scal, core + [objs["b747_scalar.cu"]]):
        subprocess.run([nvcc] + ARCH + ["-shared", "-o", scal] + core + [objs["b747_scalar.cu"]] +
                       ["-Xlinker", "-Bsymbolic", "-lcudart_static", "-lpthread", "-ldl", "-lrt"], check=True)
    legacy = os.path.join(LIBDIR, "model.so")
    if force or _stale(legacy, core + [objs["b747_scalar_legacy.cu"]]):
        subprocess.run([nvcc] + ARCH + ["-shared", "-o", legacy] + core + [objs["b747_scalar_legacy.cu"]] +
                       ["-Xlinker", "-Bsymbolic", "-lcudart_static", "-lpthread", "-ldl", "-lrt"], check=True)
    return lib, scal


if __name__ == "__main__":
    print(build_native(force=False, verbose=True))
