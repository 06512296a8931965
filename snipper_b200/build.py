"""Build libmsda_b200.so in-tree with nvcc for sm_100a (replaces the reference's
models/ops/setup.py + make.sh torch CUDAExtension build).  No torch headers are involved:
the library is plain CUDA behind a C ABI (include/msda_b200.h).

``build_all`` also builds, with the same flags, the three companion libraries: libmsda_b200_amp.so (csrc_amp/,
include/msda_b200_amp.h), the mixed-precision layer tail used under bf16 autocast; libmsda_b200_train.so
(csrc_train/, include/msda_b200_train.h), the layer tail with dropout and its backward used in training; and
libmsda_b200_amp_train.so (csrc_amp_train/, include/msda_b200_amp_train.h), the same pair for training under bf16
autocast."""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libmsda_b200.so")
SOURCES = ["msda_capi.cu", "msda_percall.cu", "msda_snippet.cu", "msda_deterministic.cu", "msda_mask.cu", "msda_frames.cu", "msda_tail.cu", "msda_planar.cu"]
HEADERS = ["msda_common.cuh", "msda_fast.cuh", "msda_snippet_common.cuh", "msda_internal.h", os.path.join("..", "..", "include", "msda_b200.h")]
OBJ_DIR = os.path.join(PKG, "lib", "obj")
AMP_CSRC = os.path.join(PKG, "csrc_amp")
AMP_LIB_PATH = os.path.join(LIB_DIR, "libmsda_b200_amp.so")
AMP_SOURCES = ["msda_amp_tail.cu"]
AMP_HEADERS = ["msda_bf16_io.cuh", os.path.join("..", "..", "include", "msda_b200_amp.h"), os.path.join("..", "..", "include", "msda_b200.h")]
TRAIN_CSRC = os.path.join(PKG, "csrc_train")
TRAIN_LIB_PATH = os.path.join(LIB_DIR, "libmsda_b200_train.so")
TRAIN_SOURCES = ["msda_train_tail.cu"]
TRAIN_HEADERS = ["msda_train_common.cuh", os.path.join("..", "..", "include", "msda_b200_train.h"), os.path.join("..", "..", "include", "msda_b200.h")]
AMP_TRAIN_CSRC = os.path.join(PKG, "csrc_amp_train")
AMP_TRAIN_LIB_PATH = os.path.join(LIB_DIR, "libmsda_b200_amp_train.so")
AMP_TRAIN_SOURCES = ["msda_amp_train_tail.cu"]
AMP_TRAIN_HEADERS = [os.path.join("..", "csrc_train", "msda_train_common.cuh"), os.path.join("..", "csrc_amp", "msda_bf16_io.cuh"),
                     os.path.join("..", "..", "include", "msda_b200_amp_train.h"), os.path.join("..", "..", "include", "msda_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libmsda_b200.so")
    return exe


def is_stale(lib_path=LIB_PATH, csrc=CSRC, files=SOURCES + HEADERS):
    if not os.path.exists(lib_path):
        return True
    t = os.path.getmtime(lib_path)
    return any(os.path.getmtime(os.path.join(csrc, f)) > t for f in files)


def _build(lib_path, csrc, sources, headers, force, verbose, extra_flags):
    if not force and not is_stale(lib_path, csrc, sources + headers):
        return lib_path
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + os.environ.get("MSDA_NVCC_EXTRA", "").split() + (["-Xptxas=-v"] if verbose else []) + ["-c", src, "-o", obj]
        res = subprocess.run(cmd, cwd=csrc, capture_output=True, text=True)
        return src, obj, res

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=len(sources)) as pool:  # the translation units compile side by side
        results = list(pool.map(compile_one, sources))
    for src, obj, res in results:
        if verbose:
            print(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, res.stdout + res.stderr))
    link = [nvcc, "-shared", "-Xcompiler", "-fPIC", "-o", lib_path] + [obj for _, obj, _ in results]
    res = subprocess.run(link, cwd=csrc, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return lib_path


def build_library(force=False, verbose=False, extra_flags=()):
    """Compile every .cu of the package into snipper_b200/lib/libmsda_b200.so."""
    return _build(LIB_PATH, CSRC, SOURCES, HEADERS, force, verbose, extra_flags)


def build_amp_library(force=False, verbose=False, extra_flags=()):
    """Compile csrc_amp/ into snipper_b200/lib/libmsda_b200_amp.so."""
    return _build(AMP_LIB_PATH, AMP_CSRC, AMP_SOURCES, AMP_HEADERS, force, verbose, extra_flags)


def build_train_library(force=False, verbose=False, extra_flags=()):
    """Compile csrc_train/ into snipper_b200/lib/libmsda_b200_train.so."""
    return _build(TRAIN_LIB_PATH, TRAIN_CSRC, TRAIN_SOURCES, TRAIN_HEADERS, force, verbose, extra_flags)


def build_amp_train_library(force=False, verbose=False, extra_flags=()):
    """Compile csrc_amp_train/ into snipper_b200/lib/libmsda_b200_amp_train.so."""
    return _build(AMP_TRAIN_LIB_PATH, AMP_TRAIN_CSRC, AMP_TRAIN_SOURCES, AMP_TRAIN_HEADERS, force, verbose, extra_flags)


def build_all(force=False, verbose=False):
    """-> (LIB_PATH, AMP_LIB_PATH, TRAIN_LIB_PATH, AMP_TRAIN_LIB_PATH), all four built."""
    return (build_library(force, verbose), build_amp_library(force, verbose), build_train_library(force, verbose),
            build_amp_train_library(force, verbose))


if __name__ == "__main__":
    print(*build_all(force=True, verbose=True), sep="\n")
