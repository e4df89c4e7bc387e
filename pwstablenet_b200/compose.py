"""Map composition fused into the sample (SURVEY.md 8(a) rows a7-a11).

The reference builds the map it hands to grid_sample with separate passes over HBM:
    netG:            map = drift.permute(0,2,3,1) + F.affine_grid(theta, size)   R/lib/networks_cascading.py:164,235
    generate_maps:   map = drift + identity meshgrid                              R/lib/utils.py:386-403
    process():       map = UpsamplingBilinear2d(size=(H,W))(map_256)              R/main_new.py:706-710
                     (stale twin: nn.Upsample(scale_factor, mode='bilinear'),      R/main.py:639-641)
    train():         frame = (x+1)*127.5 ; out = warp/127.5 - 1                    R/main_new.py:106-107
    process():       frame = uint8 HWC from cv2 ; out -> uint8                     R/main_new.py:679-684,717-721
`warp_fused` does all of it inside the sampling kernel; nothing but the raw frame, the raw
drift (and theta) is read and only the final frame is written.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from .functional import _PADDING, _stream

_BASE = {"none": _lib.PWS_BASE_NONE, "identity": _lib.PWS_BASE_IDENTITY, "affine": _lib.PWS_BASE_AFFINE}
_UP = {None: _lib.PWS_UP_NONE, "none": _lib.PWS_UP_NONE, "aligned": _lib.PWS_UP_ALIGNED, "half_pixel": _lib.PWS_UP_HALF_PIXEL}
_DT = {torch.float32: _lib.PWS_F32, torch.float16: _lib.PWS_F16, torch.bfloat16: _lib.PWS_BF16, torch.uint8: _lib.PWS_U8}
_LATTICE_DTYPES = (torch.float32, torch.float16, torch.bfloat16)


def _desc(t: torch.Tensor) -> _lib.PwsTensor:
    d = _lib.PwsTensor()
    d.data = t.data_ptr()
    d.dtype = _DT[t.dtype]
    d.device = t.device.index if t.device.index is not None else torch.cuda.current_device()
    for i in range(4):
        d.size[i] = t.size(i)
        d.stride[i] = t.stride(i)
    return d


def _spec(n, drift, base, theta, base_align_corners, upsample, map_size, pre, post, keep):
    s = _lib.PwsMapSpec()
    if drift is not None:
        if not (drift.is_cuda and drift.dtype in _LATTICE_DTYPES and drift.dim() == 4 and drift.size(3) == 2 and drift.size(0) == n):
            raise RuntimeError("warp_fused: drift must be a float32, float16 or bfloat16 CUDA tensor of sizes (N, h, w, 2) "
                               "(pass netG's planar (N,2,h,w) output as drift.permute(0,2,3,1))")
        d = _desc(drift)
        keep.append(d)
        s.drift = ctypes.pointer(d)
        map_size = (drift.size(1), drift.size(2))
    if map_size is None:
        raise RuntimeError("warp_fused: map_size is needed when there is no drift")
    s.base = _BASE[base]
    if base == "affine":
        if theta is None or theta.dtype != torch.float32 or not theta.is_cuda or tuple(theta.shape) != (n, 2, 3):
            raise RuntimeError("warp_fused: theta must be a float32 CUDA tensor of sizes (N, 2, 3)")
        theta = theta.contiguous()
        keep.append(theta)
        s.theta = theta.data_ptr()
    s.base_align_corners = int(bool(base_align_corners))
    s.upsample = _UP[upsample]
    s.map_h, s.map_w = int(map_size[0]), int(map_size[1])
    s.pre_add, s.pre_mul = float(pre[0]), float(pre[1])
    s.post_div, s.post_add = float(post[0]), float(post[1])
    return s


def compose_map(n: int, out_size: Tuple[int, int], drift: Optional[torch.Tensor] = None, base: str = "none",
                theta: Optional[torch.Tensor] = None, base_align_corners: bool = False, upsample: Optional[str] = None,
                map_size: Optional[Tuple[int, int]] = None, device=None) -> torch.Tensor:
    """The (N, Ho, Wo, 2) float32 map the fused kernel samples with (debug / parity).  A 16-bit drift is upcast exactly, so
    the map equals the one composed from drift.float()."""
    lib = _lib.load()
    keep = []
    spec = _spec(n, drift, base, theta, base_align_corners, upsample, map_size, (0.0, 1.0), (1.0, 0.0), keep)
    dev = drift.device if drift is not None else (theta.device if theta is not None else torch.device(device or "cuda"))
    out = torch.empty((n, out_size[0], out_size[1], 2), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.pws_compose_map(ctypes.byref(spec), n, ctypes.byref(_desc(out)),
                                 ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _lib.check(rc)
    return out


def warp_fused(frame: torch.Tensor, drift: Optional[torch.Tensor] = None, base: str = "none",
               theta: Optional[torch.Tensor] = None, base_align_corners: bool = False,
               upsample: Optional[str] = None, out_size: Optional[Tuple[int, int]] = None,
               map_size: Optional[Tuple[int, int]] = None, padding_mode: str = "zeros", align_corners: bool = False,
               pre: Tuple[float, float] = (0.0, 1.0), post: Tuple[float, float] = (1.0, 0.0),
               out_dtype: Optional[torch.dtype] = None, out_channels_last: bool = False) -> torch.Tensor:
    """grid_sample(pre(frame), upsample(drift + base)) -> post, in one kernel, with autograd to frame, drift and theta.

    frame:  (N,C,H,W) view, float32/16-bit float or uint8, any strides (a cv2 HWC buffer is
            `buf.permute(0,3,1,2)`).
    drift:  (N,h,w,2) view (netG's planar output permuted), or None.  float32, or the float16 / bfloat16 lattice of a
            half-precision netG: it is upcast exactly and everything after that is fp32, so the result equals the same
            call with drift.float() bit for bit.  A 16-bit lattice is coarse at 1080p: for |x| in [0.5, 1) an f16
            coordinate steps by 2**-11 (about 0.5 px at a width of 1920), a bf16 one by 2**-8 (about 3.75 px), and the
            upsample interpolates between those values (DESIGN.md section 3.8).  That coarseness is in netG's output,
            not in this call.
    theta:  (N,2,3) float32.
    base:   'none' | 'identity' (generate_maps) | 'affine' (affine_grid(theta, base_align_corners)).
    upsample: None | 'aligned' (UpsamplingBilinear2d) | 'half_pixel' (nn.Upsample bilinear); needs out_size.
    pre=(a,b): frame' = (frame+a)*b.   post=(d,e): out = acc/d + e.
    out_dtype: frame dtype by default; torch.float32 or torch.uint8 (truncating) are also offered.

    Arithmetic is fp32 for every frame dtype (uint8 and 16-bit frames are upcast exactly): (x + a) * b, the sample,
    acc / d (a true division) + e, and the result is rounded once, at the store: to a float16 / bfloat16 output by round
    to nearest, to a uint8 one by clamping to [0, 255] and truncating (NaN -> 0).  warp_stages instead rounds after every
    op on a 16-bit frame, as torch does on half-precision tensors.

    Backward: when grad mode is on, the output is float and the frame (float), drift or theta requires grad, the call
    records one autograd node whose backward is one kernel (pws_warp2d_backward_fused): the map is recomputed with the
    forward's statements and the gradient reaches the lattice through the upsample's adjoint, so neither the
    full-resolution map nor its gradient is ever written.  It is the gradient of the forward's own fp32 arithmetic:
    frame gradient summed in fp32 and rounded once to the frame dtype, drift gradient rounded once to drift's dtype,
    theta gradient in float32.  Every other call (a uint8 output in particular) takes the forward kernel alone and its
    output has no grad_fn.
    """
    if not frame.is_cuda or frame.dim() != 4 or frame.dtype not in _DT:
        raise RuntimeError("warp_fused: frame must be a 4-D CUDA tensor of dtype float32/float16/bfloat16/uint8")
    if padding_mode not in ("zeros", "border"):
        raise NotImplementedError("warp_fused: padding_mode must be 'zeros' or 'border'")
    opts = (base, base_align_corners, upsample, out_size, map_size, padding_mode, align_corners, tuple(pre), tuple(post),
            out_dtype, out_channels_last)
    final_dtype = out_dtype or (torch.float32 if frame.dtype == torch.uint8 else frame.dtype)
    wants_grad = (frame.dtype != torch.uint8 and frame.requires_grad) or (drift is not None and drift.requires_grad) or \
        (theta is not None and theta.requires_grad)
    if torch.is_grad_enabled() and final_dtype.is_floating_point and wants_grad:
        return _WarpFused.apply(frame, drift, theta, opts)
    return _fused_forward(frame, drift, theta, *opts)


def _fused_forward(frame, drift, theta, base, base_align_corners, upsample, out_size, map_size, padding_mode,
                   align_corners, pre, post, out_dtype, out_channels_last):
    lib = _lib.load()
    n, c = frame.size(0), frame.size(1)
    keep = []
    if upsample is not None and base != "none":
        # Upsampling evaluates the lattice (drift + base) at four nodes per output pixel, and a base costs IEEE
        # divisions per node.  Compose the low-resolution lattice once (what netG itself returns in the reference,
        # 0.5 MB per frame at 256 x 256) and let the sampling kernel upsample that: same arithmetic per node, so the
        # result is bit-identical, and the full-resolution map still never exists.
        if map_size is None:
            map_size = (drift.size(1), drift.size(2)) if drift is not None else None
        if map_size is None:
            raise RuntimeError("warp_fused: map_size is required when there is no drift")
        drift = compose_map(n, map_size, drift, base, theta, base_align_corners, None, map_size, device=frame.device)
        base, theta = "none", None
    if upsample is not None and drift is not None and base == "none" and not drift.is_contiguous():
        # netG hands its map over as a permuted view of planar storage (R/lib/networks_cascading.py:235-237); the
        # specialised inference kernel reads an interleaved lattice with one load per node (8 bytes, 4 for a 16-bit
        # lattice, whose dtype the repack keeps).  Repacking 0.5 MB per frame is nothing next to the frame; the values,
        # hence the result, are the same.
        drift = drift.contiguous()
    spec = _spec(n, drift, base, theta, base_align_corners, upsample, map_size, pre, post, keep)
    if out_size is None:
        out_size = (spec.map_h, spec.map_w)
    out_dtype = out_dtype or (torch.float32 if frame.dtype == torch.uint8 else frame.dtype)
    if out_channels_last:   # HWC storage, what cv2 / VideoWriter consume
        out = torch.empty((n, out_size[0], out_size[1], c), dtype=out_dtype, device=frame.device).permute(0, 3, 1, 2)
    else:
        out = torch.empty((n, c, out_size[0], out_size[1]), dtype=out_dtype, device=frame.device)
    with torch.cuda.device_of(frame):
        rc = lib.pws_warp2d_forward_fused(ctypes.byref(_desc(frame)), ctypes.byref(spec), ctypes.byref(_desc(out)),
                                          _PADDING[padding_mode], int(bool(align_corners)), _stream(frame))
    _lib.check(rc)
    return out


class _WarpFused(torch.autograd.Function):
    @staticmethod
    def forward(ctx, frame, drift, theta, opts):
        out = _fused_forward(frame, drift, theta, *opts)
        ctx.save_for_backward(frame, drift, theta)
        ctx.opts = opts
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        lib = _lib.load()
        frame, drift, theta = ctx.saved_tensors
        base, base_align_corners, upsample, out_size, map_size, padding_mode, align_corners, pre, post, _, _ = ctx.opts
        n = frame.size(0)
        # the original spec (not the forward's pre-composed lattice): the kernel recomposes the map node for node, and
        # theta's gradient needs the base
        keep = []
        spec = _spec(n, drift, base, theta, base_align_corners, upsample, map_size, pre, post, keep)
        want_frame = ctx.needs_input_grad[0] and frame.dtype != torch.uint8
        want_drift = ctx.needs_input_grad[1] and drift is not None
        want_theta = ctx.needs_input_grad[2] and base == "affine"
        # grad_input sums in fp32 for every frame type and is rounded to the frame dtype once, below
        gin = torch.empty(frame.size(), dtype=torch.float32, device=frame.device) if want_frame else None
        glat = torch.empty((n, spec.map_h, spec.map_w, 2), dtype=torch.float32, device=frame.device) \
            if (want_drift or want_theta) else None
        gtheta = torch.empty((n, 2, 3), dtype=torch.float32, device=frame.device) if want_theta else None
        with torch.cuda.device_of(frame):
            rc = lib.pws_warp2d_backward_fused(ctypes.byref(_desc(gout)), ctypes.byref(_desc(frame)), ctypes.byref(spec),
                                               ctypes.byref(_desc(gin)) if gin is not None else None,
                                               ctypes.byref(_desc(glat)) if glat is not None else None,
                                               gtheta.data_ptr() if gtheta is not None else None,
                                               _PADDING[padding_mode], int(bool(align_corners)), _stream(frame))
        _lib.check(rc)
        if gin is not None and gin.dtype != frame.dtype:
            gin = gin.to(frame.dtype)
        gdrift = glat.to(drift.dtype) if want_drift else None
        return gin, gdrift, gtheta, None


# ---- K maps, one frame, one launch: forward + backward (include/pwswarp.h, csrc/warp_stages.cu) ---------------------
_STAGE_FRAMES = (torch.float32, torch.float16, torch.bfloat16)


def _desc_ptrs(tensors, keep):
    arr = (ctypes.POINTER(_lib.PwsTensor) * len(tensors))()
    for i, t in enumerate(tensors):
        if t is None:
            arr[i] = None
        else:
            d = _desc(t)
            keep.append(d)
            arr[i] = ctypes.pointer(d)
    return arr


class _WarpStages(torch.autograd.Function):
    @staticmethod
    def forward(ctx, frame, padding, align_corners, pre_add, pre_mul, post_div, post_add, *grids):
        lib = _lib.load()
        k = len(grids)
        n, c = frame.size(0), frame.size(1)
        outs = [torch.empty((n, c, g.size(1), g.size(2)), dtype=frame.dtype, device=frame.device) for g in grids]
        keep = []
        with torch.cuda.device_of(frame):
            rc = lib.pws_warp2d_stages_forward(ctypes.byref(_desc(frame)), _desc_ptrs(grids, keep), _desc_ptrs(outs, keep), k,
                                               pre_add, pre_mul, post_div, post_add, padding, int(align_corners), _stream(frame))
        _lib.check(rc)
        ctx.save_for_backward(frame, *grids)
        ctx.args = (padding, align_corners, pre_add, pre_mul, post_div, post_add)
        return tuple(outs)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gouts):
        lib = _lib.load()
        frame, *grids = ctx.saved_tensors
        padding, align_corners, pre_add, pre_mul, post_div, post_add = ctx.args
        k = len(grids)
        gouts = [g if g is not None else torch.zeros((frame.size(0), frame.size(1), grids[i].size(1), grids[i].size(2)),
                                                     dtype=frame.dtype, device=frame.device) for i, g in enumerate(gouts)]
        from .functional import _like_layout
        # grad_input is an fp32 buffer for every frame type: 16-bit frames sum their contributions in fp32 and are rounded
        # to the frame type once, below (as functional.warp2d_backward does)
        gin = torch.empty(frame.size(), dtype=torch.float32, device=frame.device) if ctx.needs_input_grad[0] else None
        ggrids = [_like_layout(grids[i]) if ctx.needs_input_grad[7 + i] else None for i in range(k)]
        keep = []
        with torch.cuda.device_of(frame):
            rc = lib.pws_warp2d_stages_backward(_desc_ptrs(gouts, keep), ctypes.byref(_desc(frame)), _desc_ptrs(grids, keep),
                                                ctypes.byref(_desc(gin)) if gin is not None else None, _desc_ptrs(ggrids, keep), k,
                                                pre_add, pre_mul, post_div, post_add, padding, int(align_corners), _stream(frame))
        _lib.check(rc)
        if gin is not None and gin.dtype != frame.dtype:
            gin = gin.to(frame.dtype)
        return (gin, None, None, None, None, None, None, *ggrids)


def warp_stages(frame: torch.Tensor, grids, padding_mode: str = "zeros", align_corners: bool = False,
                pre: Tuple[float, float] = (0.0, 1.0), post: Tuple[float, float] = (1.0, 0.0)):
    """[grid_sample((frame + pre[0]) * pre[1], g, 'bilinear', padding_mode, align_corners) / post[0] + post[1] for g in grids]
    in ONE kernel launch that reads the frame once, with autograd to every map (and to the frame when it asks for it).

    The reference's per-stage loop R/main_new.py:103-110: `warp_stages(rgb, grid1, pre=(1, 127.5), post=(127.5, -1))`.
    Up to 4 maps, C in {1, 3}, any strides.  Values and map gradients are bit-identical to the sequence of torch calls it
    replaces, with pw.grid_sample as the sampler.

    dtypes (what a half-precision netG hands over):
        frame            maps (all one dtype)      outputs, grad_grids
        float32          float32                   float32
        float16/bfloat16 float32 or the frame's    the frame's dtype; each grad_grid in its map's dtype and layout
    With a 16-bit frame every elementwise op of that sequence rounds to the frame type, as torch does on a half-precision
    tensor (fp32 arithmetic, one rounding per op), and the kernel reproduces each rounding: the pre-scaled taps, the
    sample, `/ post[0]` and `+ post[1]`.  grad_input is summed in fp32 and rounded to the frame type once."""
    grids = list(grids)
    if not 1 <= len(grids) <= 4:
        raise ValueError("warp_stages: 1 to 4 maps")
    if padding_mode not in ("zeros", "border"):
        raise NotImplementedError("warp_stages: padding_mode must be 'zeros' or 'border'")
    if not frame.is_cuda or frame.dtype not in _STAGE_FRAMES or frame.dim() != 4:
        raise RuntimeError("warp_stages: frame must be a 4-D float32, float16 or bfloat16 CUDA tensor (no CPU fallback)")
    map_dtypes = (torch.float32,) if frame.dtype == torch.float32 else (torch.float32, frame.dtype)
    for g in grids:
        if not g.is_cuda or g.dtype not in map_dtypes or g.dim() != 4 or g.size(3) != 2 or g.size(0) != frame.size(0):
            raise RuntimeError(f"warp_stages: every map must be a CUDA tensor of sizes (N, Ho, Wo, 2) and dtype "
                               f"{' or '.join(str(d) for d in map_dtypes)} for a {frame.dtype} frame")
    if any(g.dtype != grids[0].dtype for g in grids):
        raise RuntimeError("warp_stages: all maps must have one dtype, got " + ", ".join(str(g.dtype) for g in grids))
    return _WarpStages.apply(frame, _PADDING[padding_mode], bool(align_corners), float(pre[0]), float(pre[1]),
                             float(post[0]), float(post[1]), *grids)
