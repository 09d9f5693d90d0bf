"""Build recipe for libmctq_sm100.so (the only native artefact of the package).

    python -m mct_quantizers_b200.build [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU.  The .so is written next to this file (in-tree, git-ignored)
so that it travels with the repository snapshot to the GPU box.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["mctq_affine.cu", "mctq_lut.cu", "mctq_lutp.cu", "mctq_fused.cu", "mctq_unpack.cu", "mctq_packed_linear.cu", "mctq_packed_gemm.cu", "mctq_packed_igemm.cu", "mctq_host.cu"]
OBJ_DIR = os.path.join(HERE, "csrc", "_obj")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libmctq_sm100.so")
PYEXT_SRC = os.path.join(CSRC, "mctq_pyext.c")


def pyext_path():
    import sysconfig
    return os.path.join(HERE, "_mctq_fast" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # never contract a*b+c: the reference's op order is mul, round, clamp, mul
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math", "-Xcompiler", "-ffp-contract=off",
]
LINK_FLAGS = ["-shared", "-cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a"]   # share the CUDA runtime (primary context, stream handles) with torch


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libmctq_sm100.so cannot be built")


def _cudart_dirs():
    """Link against the libcudart torch itself loads, so both sides share one runtime instance."""
    dirs = []
    try:
        import nvidia.cuda_runtime as cr  # type: ignore
        dirs.append(os.path.join(os.path.dirname(cr.__file__), "lib"))
    except Exception:
        pass
    dirs.append("/usr/local/cuda/lib64")
    return [d for d in dirs if os.path.isdir(d)]


def _headers_mtime():
    m = os.path.getmtime(os.path.abspath(__file__))
    for d in (INCLUDE, CSRC):
        for f in os.listdir(d):
            if f.endswith((".h", ".cuh")):
                m = max(m, os.path.getmtime(os.path.join(d, f)))
    return m


def build(force=False, verbose=False):
    """Compile each translation unit to an object (in parallel, only the stale ones) and link the shared library."""
    nvcc = find_nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_m = _headers_mtime()
    jobs, objs = [], []
    for src in SOURCES:
        src_path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        stale = force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src_path), hdr_m)
        if stale:
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-I", INCLUDE, "-c", "-o", obj, src_path]
            if verbose:
                print(" ".join(cmd))
            jobs.append((src, subprocess.Popen(cmd)))
    failed = [src for src, p in jobs if p.wait() != 0]
    if failed:
        raise RuntimeError(f"nvcc failed for {failed}")
    if jobs or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        subprocess.run([nvcc] + LINK_FLAGS + ["-o", LIB] + objs, check=True)
    build_pyext(force)
    return LIB


def build_pyext(force=False):
    """_mctq_fast: CPython wrappers (METH_FASTCALL) around the hottest entry points of libmctq_sm100.so -- plumbing that takes
    ~4 us of ctypes argument conversion out of every small call.  Optional: without a C compiler or Python headers the
    package uses ctypes for every call."""
    import sysconfig
    out = pyext_path()
    inc = sysconfig.get_paths().get("include")
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc or not inc or not os.path.exists(os.path.join(inc, "Python.h")):
        return None
    newest = max(os.path.getmtime(PYEXT_SRC), os.path.getmtime(os.path.join(INCLUDE, "mctq.h")))
    if not force and os.path.exists(out) and os.path.getmtime(out) >= newest:
        return out
    cmd = [cc, "-O2", "-shared", "-fPIC", "-I", INCLUDE, "-I", inc, PYEXT_SRC, "-o", out, "-L", HERE, "-l:libmctq_sm100.so",
           "-Wl,-rpath,$ORIGIN"]
    subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
