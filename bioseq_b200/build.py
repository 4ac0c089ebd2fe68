"""In-tree build of the native pieces (no setuptools, no JIT cache):

    bioseq_b200/libbsq.so                    CUDA kernels + C ABI (include/bsq.h), sm_100a only
    bioseq_b200/cbioseq.<ext-suffix>.so      pybind11 drop-in module on top of the C ABI

``python -m bioseq_b200.build`` or ``bioseq_b200.build.build()``.  nvcc cross-compiles
without a GPU; the resulting files are git-ignored but travel with the working tree.
"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)

LIB_SOURCES = ["bsq_kernels.cu", "bsq_span.cu", "bsq_varlen.cu", "bsq_mlm.cu", "bsq_crop.cu", "bsq_seqpack.cu", "bsq_kmer.cu", "bsq_revcomp.cu", "bsq_tile.cu", "bsq_translate.cu", "bsq_consumers.cu", "bsq_host.cu", "bsq_flatfile.cu", "bsq_alphabet.cpp"]
NVCC_COMPILE = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
                "-Xcompiler", "-fPIC,-Wall"]


def lib_path():
    return os.path.join(HERE, "libbsq.so")


def module_path():
    return os.path.join(HERE, "cbioseq" + sysconfig.get_config_var("EXT_SUFFIX"))


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d if os.path.isabs(d) else os.path.join(CSRC, d)) > t for d in deps)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd, cwd=CSRC)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    hdrs = ["bsq_kernels.cuh", "bsq_internal.h", os.path.join(ROOT, "include", "bsq.h")]
    # one object per source (kept under bioseq_b200/build/, git-ignored) so that touching the
    # host code does not recompile the kernels
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, relink = [], force or not os.path.exists(lib_path())
    for src in LIB_SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            _run([nvcc] + NVCC_COMPILE + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj], verbose)
            relink = True
    if relink or _stale(lib_path(), objs):
        _run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path()] + objs + ["-lz"], verbose)
    if force or _stale(module_path(), ["cbioseq_module.cpp", os.path.join(ROOT, "include", "bsq.h"), lib_path()]):
        import pybind11
        _run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-Wall",
              "-I" + sysconfig.get_paths()["include"], "-I" + pybind11.get_include(),
              "cbioseq_module.cpp", "-o", module_path(), "-L" + HERE, "-lbsq", "-Wl,-rpath,$ORIGIN"], verbose)
    return lib_path(), module_path()


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
