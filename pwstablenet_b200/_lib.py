"""ctypes binding of libpwswarp.so (include/pwswarp.h).  There is no fallback:
if the CUDA library is missing or does not load, importing the ops fails loudly."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PWS_LIB_PATH") or os.path.join(HERE, "libpwswarp.so")  # override: A/B of kernel builds

PWS_F32, PWS_F16, PWS_BF16, PWS_F64, PWS_U8, PWS_I32 = range(6)
PWS_OK, PWS_EINVAL, PWS_EUNSUPPORTED, PWS_ECUDA = 0, -1, -2, -3
ABI_VERSION = 1

EXPORTS = (
    "pws_abi_version",
    "pws_last_error",
    "pws_launch_count",
    "pws_last_kernel",
    "pws_small_problem_elems",
    "pws_warp2d_forward",
    "pws_warp2d_backward",
    "pws_warp2d_taps",
    "pws_warp2d_forward_fused",
    "pws_warp2d_backward_fused",
    "pws_compose_map",
    "pws_warp2d_stages_forward",
    "pws_warp2d_stages_backward",
)


class PwsTensor(ctypes.Structure):
    _fields_ = [
        ("data", ctypes.c_void_p),
        ("dtype", ctypes.c_int32),
        ("device", ctypes.c_int32),
        ("size", ctypes.c_int64 * 4),
        ("stride", ctypes.c_int64 * 4),
    ]


class PwsMapSpec(ctypes.Structure):
    _fields_ = [
        ("drift", ctypes.POINTER(PwsTensor)),
        ("theta", ctypes.c_void_p),
        ("base", ctypes.c_int32),
        ("base_align_corners", ctypes.c_int32),
        ("upsample", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("map_h", ctypes.c_int64),
        ("map_w", ctypes.c_int64),
        ("pre_add", ctypes.c_float),
        ("pre_mul", ctypes.c_float),
        ("post_div", ctypes.c_float),
        ("post_add", ctypes.c_float),
    ]


PWS_BASE_NONE, PWS_BASE_IDENTITY, PWS_BASE_AFFINE = 0, 1, 2
PWS_UP_NONE, PWS_UP_ALIGNED, PWS_UP_HALF_PIXEL = 0, 1, 2

_lib = None


def load() -> ctypes.CDLL:
    """Load libpwswarp.so (built by pwstablenet_b200._build.build_library / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"pwstablenet_b200: {LIB_PATH} is missing. Build it with "
            "`python -m pwstablenet_b200._build` (needs nvcc 12.9); there is no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    # pws_tensor pointers are declared void*: callers pass either byref(PwsTensor) or the hand-packed ten-word array of
    # functional._desc (same bytes, much cheaper to build)
    P = ctypes.c_void_p
    lib.pws_abi_version.restype = ctypes.c_int
    lib.pws_last_error.restype = ctypes.c_char_p
    lib.pws_launch_count.restype = ctypes.c_uint64
    lib.pws_last_kernel.restype = ctypes.c_char_p
    lib.pws_small_problem_elems.restype = ctypes.c_int64
    lib.pws_small_problem_elems.argtypes = [ctypes.c_int64]
    lib.pws_warp2d_forward.restype = ctypes.c_int
    lib.pws_warp2d_forward.argtypes = [P, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.pws_warp2d_backward.restype = ctypes.c_int
    lib.pws_warp2d_backward.argtypes = [P, P, P, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.pws_warp2d_taps.restype = ctypes.c_int
    lib.pws_warp2d_taps.argtypes = [P, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    S = ctypes.POINTER(PwsMapSpec)
    lib.pws_warp2d_forward_fused.restype = ctypes.c_int
    lib.pws_warp2d_forward_fused.argtypes = [P, S, P, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.pws_warp2d_backward_fused.restype = ctypes.c_int
    lib.pws_warp2d_backward_fused.argtypes = [P, P, S, P, P, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.pws_compose_map.restype = ctypes.c_int
    lib.pws_compose_map.argtypes = [S, ctypes.c_int64, P, ctypes.c_void_p]
    PP = ctypes.c_void_p
    lib.pws_warp2d_stages_forward.restype = ctypes.c_int
    lib.pws_warp2d_stages_forward.argtypes = [P, PP, PP, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.pws_warp2d_stages_backward.restype = ctypes.c_int
    lib.pws_warp2d_stages_backward.argtypes = [PP, P, PP, P, PP, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                               ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    got = lib.pws_abi_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"pwstablenet_b200: libpwswarp.so has ABI {got}, expected {ABI_VERSION}; rebuild it")
    _lib = lib
    return lib


def launch_count() -> int:
    """Kernels launched by libpwswarp.so so far in this process."""
    return int(load().pws_launch_count())


def last_kernel() -> str:
    """Kernel family the last forward / backward call on this thread launched (debug / tests)."""
    return load().pws_last_kernel().decode("ascii", "replace")


def small_problem_elems(elems: int = -1) -> int:
    """Query (negative argument) or set the output-element threshold below which calls take the one-wave kernels; returns
    the previous value (include/pwswarp.h)."""
    return int(load().pws_small_problem_elems(int(elems)))


def last_error() -> str:
    return load().pws_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Turn a pws_status into the exception torch would have raised."""
    if rc == PWS_OK:
        return
    msg = last_error()
    if rc == PWS_EINVAL:
        raise RuntimeError(msg)  # torch raises RuntimeError for TORCH_CHECK failures
    if rc == PWS_EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"pwswarp CUDA error: {msg}")
