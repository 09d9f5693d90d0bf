"""ctypes binding of libmctq_sm100.so (C ABI: include/mctq.h).

The library is loaded lazily, on the first operator call (never at import time), so that quantizer objects
stay picklable and the package imports on machines without the toolchain.  There is NO fallback: if the
shared object is missing and cannot be built, or no CUDA device is present, the operators raise.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmctq_sm100.so")

F32, BF16, F16 = 0, 1, 2
CODES_NONE, CODES_INT8, CODES_INT4 = 0, 1, 2
PRE_RELU, PRE_RELU6, PRE_ADD, PRE_ADD_RELU = 1, 2, 3, 4
PACK_AFFINE_I8, PACK_AFFINE_I4, PACK_LUT_U8, PACK_LUT_I4 = 1, 2, 3, 4
PACK_LUT_KINDS = (PACK_LUT_U8, PACK_LUT_I4)


def integer_linear_max_k(w_signed, x_signed):
    """Largest in_features of mctq_packed_linear_i8 for the (weight, x) code signedness: the int32 sum of code products
    cannot overflow (the values of mctq_packed_linear_i8_max_k)."""
    return 131071 if (w_signed and x_signed) else 65793 if (w_signed or x_signed) else 33025


def packed_code_bytes(kind, n):
    """Bytes of the codes of n elements of packed kind `kind`: one per element, or one per two for int4 codes and 4-bit
    LUT indices."""
    return n if kind in (PACK_AFFINE_I8, PACK_LUT_U8) else (n + 1) // 2


_lock = threading.Lock()
_lib = None

c_vp, c_i64, c_i32, c_int, c_f32, c_sz, c_u64 = (ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int,
                                                  ctypes.c_float, ctypes.c_size_t, ctypes.c_uint64)


class MctqTensorDesc(ctypes.Structure):
    """Mirror of `struct MctqTensorDesc` (include/mctq.h)."""
    _fields_ = [("x", c_vp), ("y", c_vp), ("codes", c_vp), ("scale", c_vp), ("zp", c_vp),
                ("n", c_i64), ("C", c_i64), ("inner", c_i64),
                ("qmin", c_i32), ("qmax", c_i32), ("dtype", c_i32), ("code_mode", c_i32)]


class MctqLutTensorDesc(ctypes.Structure):
    """Mirror of `struct MctqLutTensorDesc` (include/mctq.h)."""
    _fields_ = [("x", c_vp), ("y", c_vp), ("prepared_dev", c_vp), ("n", c_i64), ("C", c_i64), ("inner", c_i64),
                ("dtype", c_i32), ("K", c_i32), ("lut_values_bitwidth", c_i32), ("is_signed", c_i32)]


class MctqSiteDesc(ctypes.Structure):
    """Mirror of `struct MctqSiteDesc` (include/mctq.h)."""
    _fields_ = [("x", c_vp), ("y", c_vp), ("n", c_i64), ("dtype", c_i32), ("scale", c_f32), ("zp", c_i32),
                ("qmin", c_i32), ("qmax", c_i32), ("reserved", c_i32)]


class MctqPackedDesc(ctypes.Structure):
    """Mirror of `struct MctqPackedDesc` (include/mctq.h)."""
    _fields_ = [("codes", c_vp), ("y", c_vp), ("n", c_i64), ("C", c_i64), ("inner", c_i64),
                ("kind", c_i32), ("is_signed", c_i32), ("y_dtype", c_i32), ("K", c_i32),
                ("scale", c_vp), ("zp", c_vp), ("lut_quotients", c_vp)]


class MctqConv2dGeom(ctypes.Structure):
    """Mirror of `struct MctqConv2dGeom` (include/mctq.h)."""
    _fields_ = [(f, c_i32) for f in ("N", "H", "W", "Cin", "Ho", "Wo", "kh", "kw", "sh", "sw", "dh", "dw",
                                     "pt", "pb", "pl", "pr")]


class MctqDwPlan(ctypes.Structure):
    """Mirror of `struct MctqDwPlan` (include/mctq.h)."""
    _fields_ = [(f, c_i32) for f in ("S", "TH", "TW", "IH", "IW", "smem_bytes")]


# name -> (restype, argtypes): every symbol include/mctq.h declares
SIGNATURES = {
    "mctq_abi_version": (c_int, []),
    "mctq_build_info": (ctypes.c_char_p, []),
    "mctq_fq_affine": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i32, c_i32, c_int, c_vp]),
    "mctq_fq_affine_scalar": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_f32, c_i32, c_i32, c_i32, c_int, c_vp]),
    "mctq_affine_prepared_bytes": (c_sz, [c_i64]),
    "mctq_affine_prepare": (c_int, [c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "mctq_fq_affine_prepared": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_i64, c_i64, c_i64, c_i32, c_i32, c_int, c_vp]),
    "mctq_fq_affine_scalar_pre": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_f32, c_i32, c_i32, c_i32, c_vp]),
    "mctq_dequant_affine": (c_int, [c_vp, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "mctq_unpack_plan_bytes": (c_sz, [c_vp, c_int]),
    "mctq_unpack_plan": (c_i64, [c_vp, c_int, c_vp, c_sz]),
    "mctq_unpack_multi": (c_int, [c_vp, c_vp]),
    "mctq_packed_linear": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_vp, c_vp]),
    "mctq_packed_linear_batched": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mctq_quantize_rows_i8": (c_int, [c_vp, c_int, c_i64, c_i64, c_f32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "mctq_packed_linear_i8_max_k": (c_i64, [c_int, c_int]),
    "mctq_packed_linear_i8": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_vp,
                                      c_i64, c_vp]),
    "mctq_quantize_nhwc_i8": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_i64, c_f32, c_i32, c_i32, c_i32, c_vp, c_vp,
                                      c_vp]),
    "mctq_packed_conv2d_i8": (c_int, [c_vp, c_vp, c_i64, c_vp, c_int, c_i32, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int,
                                      c_vp]),
    "mctq_packed_linear_i8_lut": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_int,
                                          c_vp, c_i64, c_vp, c_vp]),
    "mctq_packed_conv2d_i8_lut": (c_int, [c_vp, c_vp, c_i64, c_vp, c_int, c_i32, c_vp, c_vp, c_vp, c_vp, c_int, c_vp,
                                          c_int, c_vp, c_vp]),
    "mctq_packed_dwconv2d_i8": (c_int, [c_vp, c_vp, c_i64, c_vp, c_int, c_int, c_f32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp,
                                        c_vp, c_vp]),
    "mctq_packed_dwconv2d_i8_plan": (c_int, [c_vp, c_i64, c_int, c_vp]),
    "mctq_quantize_rows_i8_padded": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_f32, c_i32, c_i32, c_i32, c_vp, c_vp,
                                             c_vp]),
    "mctq_quantize_nhwc_i8_padded": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_i64, c_i64, c_f32, c_i32, c_i32, c_i32,
                                             c_vp, c_vp, c_vp]),
    "mctq_packed_linear_i8_padded": (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp,
                                             c_int, c_vp, c_i64, c_vp, c_vp]),
    "mctq_packed_conv2d_i8_padded": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_int, c_i32, c_vp, c_vp, c_vp, c_vp, c_int,
                                             c_vp, c_int, c_vp, c_vp]),
    "mctq_multi_tile_elems": (c_i64, []),
    "mctq_multi_plan": (c_i64, [c_vp, c_int, c_vp]),
    "mctq_fq_affine_multi": (c_int, [c_vp, c_vp, c_int, c_i64, c_vp]),
    "mctq_fq_affine_scalar_multi": (c_int, [c_vp, c_int, c_vp]),
    "mctq_lut_table_bytes": (c_sz, [c_int]),
    "mctq_lut_build_table": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_sz]),
    "mctq_fq_lut": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_i64, c_i64, c_i64, c_f32, c_int, c_vp]),
    "mctq_fq_lut_scalar": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_f32, c_f32, c_int, c_int, c_vp]),
    "mctq_lut_prepared_bytes": (c_sz, [c_int, c_int, c_int, c_i64]),
    "mctq_lut_prepare": (c_int, [c_vp, c_int, c_vp, c_i64, c_f32, c_int, c_f32, c_f32, c_int, c_vp, c_sz, c_vp]),
    "mctq_fq_lut_prepared": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_int, c_int, c_i64, c_i64, c_i64, c_int, c_vp]),
    "mctq_lut_multi_plan_bytes": (c_sz, [c_vp, c_int]),
    "mctq_lut_multi_plan": (c_i64, [c_vp, c_int, c_vp, c_sz]),
    "mctq_fq_lut_prepared_multi": (c_int, [c_vp, c_vp]),
    "mctq_host_staging_min_bytes": (c_sz, []),
    "mctq_host_set_deferred": (c_int, [c_int, c_int]),
    "mctq_host_wait": (c_int, [c_int]),
    "mctq_fq_affine_host": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i32, c_i32, c_vp, c_sz, c_int]),
    "mctq_fq_lut_host": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_i64, c_i64, c_f32, c_int, c_f32, c_f32,
                                 c_int, c_vp, c_sz, c_int]),
    "mctq_launch_count": (c_i64, []),
    "mctq_set_tuning": (c_int, [c_int, c_int]),
    "mctq_selftest_division": (c_int, [c_i64, c_u64, c_vp, c_vp]),
}

ERRORS = {-1: "MCTQ_E_BADARG", -2: "MCTQ_E_DTYPE", -3: "MCTQ_E_RANGE", -4: "MCTQ_E_LUT", -5: "MCTQ_E_NODEVICE"}


class MctqError(RuntimeError):
    pass


def _preload_cudart():
    """Make sure the CUDA runtime torch uses is already mapped, so the DT_NEEDED entry of our library binds
    to the same instance (shared primary context, interchangeable stream handles)."""
    try:
        import torch  # noqa: F401  (maps libcudart.so.12 from the nvidia-cuda-runtime wheel)
    except Exception:
        pass
    for cand in ("libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
        try:
            ctypes.CDLL(cand, mode=ctypes.RTLD_GLOBAL)
            return
        except OSError:
            continue
    try:
        import nvidia.cuda_runtime as cr
        ctypes.CDLL(os.path.join(os.path.dirname(cr.__file__), "lib", "libcudart.so.12"), mode=ctypes.RTLD_GLOBAL)
    except Exception:
        pass


def load(build_if_missing=True):
    """Load (once) and return the ctypes handle with argtypes set.  Raises MctqError when unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            if not build_if_missing:
                raise MctqError(f"{LIB_PATH} is missing (run `python -m mct_quantizers_b200.build`)")
            from mct_quantizers_b200 import build as _build
            try:
                _build.build()
            except Exception as e:  # no nvcc, compile error ...
                raise MctqError(f"libmctq_sm100.so is missing and could not be built: {e}; "
                                f"mct_quantizers_b200 has no CPU / eager fallback") from e
        _preload_cudart()
        try:
            handle = ctypes.CDLL(LIB_PATH)
        except OSError as e:
            raise MctqError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError here = ABI drift between header and library
            fn.restype = res
            fn.argtypes = args
        if handle.mctq_abi_version() != 1:
            raise MctqError(f"ABI version mismatch: library reports {handle.mctq_abi_version()}, binding expects 1")
        # MCTQ_TUNE="key=value,..." applies mctq_set_tuning at load time: key 3 (dependent launch), key 9 (NVTX); see include/mctq.h
        for kv in filter(None, os.environ.get("MCTQ_TUNE", "").split(",")):
            k, v = kv.split("=")
            if handle.mctq_set_tuning(int(k), int(v)) < 0:
                raise MctqError(f"MCTQ_TUNE: mctq_set_tuning({k}, {v}) rejected")
        _lib = handle
        _load_fast()
    return _lib


fast = None      # module _mctq_fast (CPython wrappers of the hottest entry points) or None: then every call goes through ctypes


def _load_fast():
    """Import the optional CPython front door after libmctq_sm100.so is mapped (its DT_NEEDED entry then binds to the same
    instance: one launch counter, one set of tuning switches).  MCTQ_NO_FASTCALL=1 keeps everything on ctypes."""
    global fast
    if os.environ.get("MCTQ_NO_FASTCALL"):
        return
    try:
        from mct_quantizers_b200 import build as _build
        path = _build.pyext_path()
        if not os.path.exists(path):
            try:
                _build.build_pyext()
            except Exception:
                return
        if os.path.exists(path):
            import importlib.util
            spec = importlib.util.spec_from_file_location("mct_quantizers_b200._mctq_fast", path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            fast = mod
    except Exception:
        fast = None


def check(rc, what):
    if rc == 0:
        return
    if rc < 0:
        raise MctqError(f"{what}: {ERRORS.get(rc, rc)}")
    raise MctqError(f"{what}: CUDA error {rc}")


def launch_count():
    return int(load().mctq_launch_count())


def build_lut_table(lut_values, lut_values_bitwidth, signed):
    """Compile a centroid list into the search-table blob (host; returns bytes)."""
    import numpy as np
    lib = load()
    lut = np.ascontiguousarray(np.asarray(lut_values, dtype=np.float32).reshape(-1))
    K = int(lut.size)
    nbytes = lib.mctq_lut_table_bytes(K)
    if nbytes == 0:
        raise MctqError(f"LUT with {K} entries is not supported (1..256)")
    buf = (ctypes.c_uint8 * nbytes)()
    check(lib.mctq_lut_build_table(lut.ctypes.data_as(c_vp), K, int(lut_values_bitwidth), int(bool(signed)),
                                   ctypes.cast(buf, c_vp), nbytes), "mctq_lut_build_table")
    return bytes(buf)
