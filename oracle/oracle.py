"""ctypes front-end of the CPU oracle (oracle/warp_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline leg.  The product package pwstablenet_b200/ never
imports this module.  Every function takes and returns numpy arrays; strides
are honoured (the reference hands over permuted views, SURVEY.md section 7).

Reference call sites restated (R = /root/reference):
  forward / backward   R/main_new.py:106,109,116,118,197,716 (F.grid_sample) and :214 (autograd)
  generate_maps        R/lib/utils.py:386-403
  affine_map           R/lib/networks_cascading.py:164,235 (F.affine_grid + drift)
  upsample_map         R/main_new.py:706-710, R/main.py:639-641
  upsample_map_backward, affine_theta_grad   their adjoints (warp_fused's backward, R/main_new.py:214)
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpwsoracle.so")
_lib = None

PADDING = {"zeros": 0, "border": 1}


def build(force: bool = False) -> str:
    """Compile warp_oracle.c with gcc (oracle/Makefile). Returns the .so path."""
    src = os.path.join(_HERE, "warp_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "libpwsoracle.so"])
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        assert _lib.oracle_abi_version() == 2
    return _lib


def _strides(a: np.ndarray):
    assert a.ndim == 4
    s = [st // a.itemsize for st in a.strides]
    return (ctypes.c_int64 * 4)(*s)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _check(inp, grid, dtype):
    assert inp.dtype == dtype and grid.dtype == dtype, (inp.dtype, grid.dtype)
    assert inp.ndim == 4 and grid.ndim == 4 and grid.shape[3] == 2 and inp.shape[0] == grid.shape[0]


def taps(grid: np.ndarray, H: int, W: int, padding: str = "zeros", align_corners: bool = False,
         want_weights: bool = True):
    """North-west tap (x0, y0) int32, 4-bit validity mask uint8 and the four
    weights for every output pixel of `grid` (N,Ho,Wo,2) over an HxW frame."""
    assert grid.dtype == np.float32
    N, Ho, Wo, _ = grid.shape
    x0 = np.empty((N, Ho, Wo), np.int32)
    y0 = np.empty((N, Ho, Wo), np.int32)
    mask = np.empty((N, Ho, Wo), np.uint8)
    wts = np.empty((N, Ho, Wo, 4), np.float32) if want_weights else None
    lib().oracle_warp2d_taps_f32(_ptr(grid), _strides(grid), N, Ho, Wo, H, W, PADDING[padding],
                                 int(bool(align_corners)), _ptr(x0), _ptr(y0), _ptr(mask), _ptr(wts))
    return x0, y0, mask, wts


def forward(inp: np.ndarray, grid: np.ndarray, padding: str = "zeros", align_corners: bool = False):
    dt = inp.dtype
    assert dt in (np.float32, np.float64)
    _check(inp, grid, dt)
    N, C, H, W = inp.shape
    _, Ho, Wo, _ = grid.shape
    out = np.empty((N, C, Ho, Wo), dt)
    fn = lib().oracle_warp2d_forward_f32 if dt == np.float32 else lib().oracle_warp2d_forward_f64
    fn(_ptr(inp), _strides(inp), _ptr(grid), _strides(grid), _ptr(out), _strides(out),
       N, C, H, W, Ho, Wo, PADDING[padding], int(bool(align_corners)))
    return out


def backward(gout: np.ndarray, inp: np.ndarray, grid: np.ndarray, padding: str = "zeros",
             align_corners: bool = False, want_f64_accum: bool = False):
    """Returns (grad_in, grad_grid) -- plus grad_in accumulated in float64 when
    want_f64_accum (fp32 inputs only)."""
    dt = inp.dtype
    _check(inp, grid, dt)
    assert gout.dtype == dt
    N, C, H, W = inp.shape
    _, Ho, Wo, _ = grid.shape
    assert gout.shape == (N, C, Ho, Wo)
    gin = np.zeros((N, C, H, W), dt)
    ggrid = np.empty((N, Ho, Wo, 2), dt)
    pad, al = PADDING[padding], int(bool(align_corners))
    if dt == np.float32:
        gin64 = np.zeros((N, C, H, W), np.float64) if want_f64_accum else None
        lib().oracle_warp2d_backward_f32(_ptr(gout), _strides(gout), _ptr(inp), _strides(inp), _ptr(grid),
                                         _strides(grid), _ptr(gin), _ptr(gin64), _ptr(ggrid),
                                         N, C, H, W, Ho, Wo, pad, al)
        return (gin, ggrid, gin64) if want_f64_accum else (gin, ggrid)
    assert dt == np.float64
    lib().oracle_warp2d_backward_f64(_ptr(gout), _strides(gout), _ptr(inp), _strides(inp), _ptr(grid),
                                     _strides(grid), _ptr(gin), _ptr(ggrid), N, C, H, W, Ho, Wo, pad, al)
    return gin, ggrid


def generate_maps(drift: np.ndarray):
    """drift (N,2,H,W) planar -> map (N,2,H,W) planar = drift + identity meshgrid."""
    drift = np.ascontiguousarray(drift, np.float32)
    N, two, H, W = drift.shape
    assert two == 2
    out = np.empty_like(drift)
    lib().oracle_generate_maps_f32(_ptr(drift), _ptr(out), N, H, W)
    return out


def affine_map(theta: np.ndarray, H: int, W: int, drift: np.ndarray | None = None, align_corners: bool = False):
    """theta (N,2,3) [+ planar drift (N,2,H,W)] -> interleaved map (N,H,W,2)."""
    theta = np.ascontiguousarray(theta, np.float32)
    N = theta.shape[0]
    if drift is not None:
        drift = np.ascontiguousarray(drift, np.float32)
        assert drift.shape == (N, 2, H, W)
    out = np.empty((N, H, W, 2), np.float32)
    lib().oracle_affine_map_f32(_ptr(theta), _ptr(drift), _ptr(out), N, H, W, int(bool(align_corners)))
    return out


def upsample_map(src: np.ndarray, H: int, W: int, align_corners: bool = True):
    """planar map (N,2,h,w) -> (N,2,H,W), bilinear."""
    src = np.ascontiguousarray(src, np.float32)
    N, two, h, w = src.shape
    assert two == 2
    out = np.empty((N, 2, H, W), np.float32)
    lib().oracle_upsample_map_f32(_ptr(src), _ptr(out), N, h, w, H, W, int(bool(align_corners)))
    return out


def upsample_coefs(src: int, dst: int, align_corners: bool = True):
    """(i0, ip, l0, l1) of destination indices 0..dst-1 from a source of size src: upsample_map's coefficients."""
    i0, ip = np.empty(dst, np.int32), np.empty(dst, np.int32)
    l0, l1 = np.empty(dst, np.float32), np.empty(dst, np.float32)
    lib().oracle_upsample_coefs_f32(src, dst, int(bool(align_corners)), _ptr(i0), _ptr(ip), _ptr(l0), _ptr(l1))
    return i0, ip, l0, l1


def upsample_map_backward(gmap: np.ndarray, h: int, w: int, align_corners: bool = True):
    """Adjoint of upsample_map with its fp32 coefficients: gmap planar (N,2,H,W) -> (glat, gabs, nterms), each
    (N,2,h,w): the fp64 sum of the terms h_l * w_l * g each node receives, the sum of their magnitudes, their count."""
    gmap = np.ascontiguousarray(gmap, np.float64)
    N, two, H, W = gmap.shape
    assert two == 2
    glat, gabs = np.zeros((N, 2, h, w)), np.zeros((N, 2, h, w))
    nterms = np.zeros((N, 2, h, w), np.int64)
    lib().oracle_upsample_map_backward_f64(_ptr(gmap), N, h, w, H, W, int(bool(align_corners)), _ptr(glat), _ptr(gabs),
                                           _ptr(nterms))
    return glat, gabs, nterms


def affine_theta_grad(glat: np.ndarray, align_corners: bool = False):
    """glat interleaved (N,h,w,2) -> (gtheta, gabs), each (N,2,3) fp64: sum_ij glat[n,i,j,c] * (bx_j, by_i, 1) with
    affine_map's base coordinates, and the sums of the terms' magnitudes."""
    glat = np.ascontiguousarray(glat, np.float64)
    N, h, w, two = glat.shape
    assert two == 2
    gtheta, gabs = np.zeros((N, 2, 3)), np.zeros((N, 2, 3))
    lib().oracle_affine_theta_grad_f64(_ptr(glat), N, h, w, int(bool(align_corners)), _ptr(gtheta), _ptr(gabs))
    return gtheta, gabs
