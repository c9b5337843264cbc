"""ctypes binding of ``libb200wave.so`` (the C ABI declared in ``include/b200wave.h``).

There is no CPU path: if the library cannot be loaded the first compute call
raises ``RuntimeError`` -- it never falls back to torch ops or to the oracle.
"""
import ctypes
import os
import threading

from . import _build

_c_float_p = ctypes.POINTER(ctypes.c_float)
_c_int_p = ctypes.POINTER(ctypes.c_int)
_c_vp_p = ctypes.POINTER(ctypes.c_void_p)

# status codes of include/b200wave.h
OK = 0
ERR_BAD_MODE = -1
ERR_BAD_TAPS = -2
ERR_NULL_POINTER = -3
ERR_BAD_SHAPE = -4
ERR_REFLECT_PAD = -5
ERR_PER_TOO_SHORT = -6
ERR_LAUNCH = -7
ERR_WORKSPACE = -8
ERR_BAD_WINDOW = -9

ABI_VERSION = 1
MAX_TAPS = 64
MAX_LEVELS = 8
SSIM_MAX_WINDOW = 11

# every symbol the header declares: name -> (restype, argtypes)
_vp, _i, _i64, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t
_c_double_p = ctypes.POINTER(ctypes.c_double)
SYMBOLS = {
    "b200w_abi_version": (_i, []),
    "b200w_status_string": (ctypes.c_char_p, [_i]),
    "b200w_last_cuda_error": (_i, []),
    "b200w_dwt_coeff_len": (_i, [_i, _i, _i]),
    "b200w_idwt_len": (_i, [_i, _i, _i]),
    "b200w_afb2d_f32": (_i, [_vp, _i64, _i64, _i, _i, _i,
                             _c_float_p, _c_float_p, _i, _c_float_p, _c_float_p, _i,
                             _i, _vp, _vp, _vp]),
    "b200w_sfb2d_f32": (_i, [_vp, _i64, _i64, _vp, _i, _i, _i,
                             _c_float_p, _c_float_p, _i, _c_float_p, _c_float_p, _i,
                             _i, _vp, _i, _i, _vp]),
    "b200w_afb2d_ex_f32": (_i, [_vp, _i64, _i64, _i, _i, _i,
                                _c_float_p, _c_float_p, _i, _c_float_p, _c_float_p, _i,
                                _i, _vp, _vp, ctypes.c_float, ctypes.c_float, _vp]),
    "b200w_tv_workspace_bytes": (_sz, [_i, _i]),
    "b200w_tv_fwd_f32": (_i, [_vp, _i, _i, _i, _vp, _sz, _vp, _vp]),
    "b200w_tv_bwd_f32": (_i, [_vp, _vp, ctypes.c_float, ctypes.c_float, _i, _i, _i, _vp, _vp]),
    "b200w_afb2d_f64": (_i, [_vp, _i64, _i64, _i, _i, _i, _c_double_p, _c_double_p, _i, _c_double_p, _c_double_p, _i,
                             _i, _vp, _vp, _vp]),
    "b200w_sfb2d_f64": (_i, [_vp, _i64, _i64, _vp, _i, _i, _i, _c_double_p, _c_double_p, _i, _c_double_p, _c_double_p, _i,
                             _i, _vp, _i, _i, _vp]),
    "b200w_afb1d_f32": (_i, [_vp, _i64, _i, _i, _c_float_p, _c_float_p, _i, _i, _vp, _vp, _vp]),
    "b200w_sfb1d_f32": (_i, [_vp, _i64, _vp, _i, _i, _c_float_p, _c_float_p, _i, _i, _i, _vp, _vp]),
    "b200w_swt2d_fwd_f32": (_i, [_vp, _i, _i, _i, _c_float_p, _c_float_p, _c_float_p, _c_float_p, _i, _i, _i, _vp, _vp]),
    "b200w_swt2d_bwd_f32": (_i, [_vp, _i, _i, _i, _c_float_p, _c_float_p, _c_float_p, _c_float_p, _i, _i, _i, _vp, _vp]),
    "b200w_phase_workspace_bytes": (_sz, [_i, _i, _i]),
    "b200w_phase_sums_c64": (_i, [_vp, _vp, _i, _i, _i, ctypes.c_float, _vp, _sz, _vp, _vp]),
    "b200w_phase_grad_c64": (_i, [_vp, _vp, _i, _i, _i, ctypes.c_float, _vp, _vp, ctypes.c_float, _vp, _vp, _vp]),
    "b200w_kernel_launches": (ctypes.c_ulonglong, []),
    "b200w_kernel_log": (ctypes.c_char_p, [_i]),
    "b200w_build_hash": (ctypes.c_char_p, []),
    "b200w_dwt2_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _c_int_p]),
    "b200w_dwt2_f32": (_i, [_vp, _i64, _i64, _i, _i, _i,
                            _c_float_p, _c_float_p, _i, _c_float_p, _c_float_p, _i,
                            _i, _i, _c_int_p, _vp, _c_vp_p, _vp, _sz, _vp]),
    "b200w_idwt2_workspace_bytes": (_sz, [_i, _i, _c_int_p, _c_int_p]),
    "b200w_idwt2_f32": (_i, [_vp, _i64, _i64, _c_vp_p, _i, _c_int_p, _c_int_p,
                             _c_float_p, _c_float_p, _i, _c_float_p, _c_float_p, _i,
                             _i, _i, _c_int_p, _c_int_p, _vp, _vp, _sz, _vp]),
    "b200w_freq_mask_c64": (_i, [_vp, _i, _i, _i, ctypes.c_float, _i, _vp]),
    "b200w_abs_sign_f32": (_i, [_vp, _vp, _sz, ctypes.c_float, _vp]),
    "b200w_sign_mul_f32": (_i, [_vp, _vp, _vp, _sz, ctypes.c_float, _vp]),
    "b200w_ssim_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "b200w_ssim_fwd_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _c_float_p, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "b200w_ssim_bwd_f32": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _c_float_p, _i, _i, _vp, _vp, _vp]),
    "b200w_afb1d_f64": (_i, [_vp, _i64, _i, _i, _c_double_p, _c_double_p, _i, _i, _vp, _vp, _vp]),
    "b200w_sfb1d_f64": (_i, [_vp, _i64, _vp, _i, _i, _c_double_p, _c_double_p, _i, _i, _i, _vp, _vp]),
    "b200w_swt2d_fwd_f64": (_i, [_vp, _i, _i, _i, _c_double_p, _c_double_p, _c_double_p, _c_double_p, _i, _i, _i, _vp,
                                 _vp]),
    "b200w_swt2d_bwd_f64": (_i, [_vp, _i, _i, _i, _c_double_p, _c_double_p, _c_double_p, _c_double_p, _i, _i, _i, _vp,
                                 _vp]),
    "b200w_iswt2d_f32": (_i, [_vp, _i64, _vp, _i, _i, _i, _c_float_p, _c_float_p, _c_float_p, _c_float_p, _i, _i, _vp,
                              _vp]),
    "b200w_iswt2d_f64": (_i, [_vp, _i64, _vp, _i, _i, _i, _c_double_p, _c_double_p, _c_double_p, _c_double_p, _i, _i,
                              _vp, _vp]),
    "b200w_tv_workspace_bytes_f64": (_sz, [_i, _i]),
    "b200w_tv_fwd_f64": (_i, [_vp, _i, _i, _i, _vp, _sz, _vp, _vp]),
    "b200w_tv_bwd_f64": (_i, [_vp, _vp, ctypes.c_double, ctypes.c_double, _i, _i, _i, _vp, _vp]),
    "b200w_ssim_workspace_bytes_f64": (_sz, [_i, _i, _i, _i]),
    "b200w_ssim_fwd_f64": (_i, [_vp, _vp, _i, _i, _i, _i, _c_double_p, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "b200w_ssim_bwd_f64": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _c_double_p, _i, _i, _vp, _vp, _vp]),
    "b200w_msssim_scale_fwd_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _c_float_p, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz,
                                        _vp]),
    "b200w_msssim_scale_bwd_f32": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _c_float_p, _i, _vp, _vp, _vp, _vp,
                                        _vp]),
    "b200w_msssim_scale_fwd_f64": (_i, [_vp, _vp, _i, _i, _i, _i, _c_double_p, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz,
                                        _vp]),
    "b200w_msssim_scale_bwd_f64": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _c_double_p, _i, _vp, _vp, _vp, _vp,
                                        _vp]),
    "b200w_afb2d_ex_f64": (_i, [_vp, _i64, _i64, _i, _i, _i, _c_double_p, _c_double_p, _i, _c_double_p, _c_double_p, _i,
                                _i, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp]),
    "b200w_freq_mask_c128": (_i, [_vp, _i, _i, _i, ctypes.c_double, _i, _vp]),
    "b200w_abs_sign_f64": (_i, [_vp, _vp, _sz, ctypes.c_double, _vp]),
    "b200w_sign_mul_f64": (_i, [_vp, _vp, _vp, _sz, ctypes.c_double, _vp]),
}

_lock = threading.Lock()
_lib = None


class B200WaveError(RuntimeError):
    pass


def library_path():
    return os.environ.get("B200W_LIBRARY", _build.LIB_PATH)


def load(build_if_missing=True):
    """Load (building first if the in-tree .so is missing or stale and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if path == _build.LIB_PATH and build_if_missing and not _build.is_fresh():
            if _build.find_nvcc() is not None:
                _build.build()
            elif os.path.exists(path):
                # *.so is git-ignored but travels to the GPU boxes: never let a stale binary pass silently
                import warnings
                warnings.warn("libb200wave.so does not match the sources in this tree and nvcc is not available to "
                              "rebuild it; results come from the OLD binary (see b200wave._cabi.build_hash())",
                              RuntimeWarning, stacklevel=2)
        if not os.path.exists(path):
            raise B200WaveError(
                "libb200wave.so not found at %s and nvcc is unavailable to build it. This package has no "
                "CPU or PyTorch fallback: run `python __graft_entry__.py build` on a machine with CUDA 12.9." % path)
        lib = ctypes.CDLL(path)
        for name, (restype, argtypes) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.b200w_abi_version() != ABI_VERSION:
            raise B200WaveError("libb200wave ABI version %d != expected %d" % (lib.b200w_abi_version(), ABI_VERSION))
        _lib = lib
    return _lib


def build_hash():
    """{"library": hash the loaded binary was built from, "tree": hash of the sources here, "match": bool}."""
    lib = load()
    have = lib.b200w_build_hash().decode()
    want = _build._source_hash() if library_path() == _build.LIB_PATH else None
    return {"library": have[:16], "tree": None if want is None else want[:16], "match": want is None or have == want}


def status_string(code):
    return load().b200w_status_string(int(code)).decode()


def taps_array(values):
    vals = [float(v) for v in values]
    return (ctypes.c_float * len(vals))(*vals), len(vals)


def taps_array_f64(values):
    vals = [float(v) for v in values]
    return (ctypes.c_double * len(vals))(*vals), len(vals)


def int_array(values):
    vals = [int(v) for v in values]
    return (ctypes.c_int * len(vals))(*vals)


def ptr_array(tensors):
    """HOST array of device pointers; None entries become NULL."""
    vals = [None if t is None else t.data_ptr() for t in tensors]
    return (ctypes.c_void_p * len(vals))(*vals)


def check(code, mode_name=None):
    """Map a negative status onto the reference's exception types."""
    if code == OK:
        return
    if code == ERR_BAD_MODE:
        # pw/dwt/lowlevel.py:88,170,269,290 raise exactly this text
        raise ValueError("Unkown pad type: {}".format(mode_name))
    msg = status_string(code)
    if code == ERR_LAUNCH:
        msg += " (cudaError %d)" % load().b200w_last_cuda_error()
    raise B200WaveError("b200wave: " + msg)


def kernel_launches():
    """Kernels launched by the library in this process so far."""
    return int(load().b200w_kernel_launches())


def recent_kernels(n):
    """Names of the last ``n`` kernels launched, oldest first."""
    lib = load()
    return [lib.b200w_kernel_log(i).decode() for i in range(min(n, 64) - 1, -1, -1)]
