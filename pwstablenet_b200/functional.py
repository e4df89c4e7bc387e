"""Drop-in for the reference's warp calls: same Python signature as
torch.nn.functional.grid_sample ($TORCH/nn/functional.py:5085-5242), executed by
the hand-written sm_100a kernels behind libpwswarp.so.

Reference call sites served (R = the PWStableNet checkout):
    R/main_new.py:106,116   functional.grid_sample((rgb + 1) * 127.5, grid1[nl])
    R/main_new.py:109,118   gray warps
    R/main_new.py:197       functional.grid_sample(fake2[nl], affine_grid(...))  (grad -> frame)
    R/main_new.py:716       functional.grid_sample(now, grid_resize)              (inference)
All of them pass (input, grid) positionally and leave the keywords at their defaults.

CUDA tensors only: a CPU tensor raises (no CPU fallback, no multi-backend dispatch).
"""
from __future__ import annotations

import ctypes
import os
import warnings
from typing import Optional

import torch

from . import _lib

_DTYPES = {
    torch.float32: _lib.PWS_F32,
    torch.float16: _lib.PWS_F16,
    torch.bfloat16: _lib.PWS_BF16,
    torch.float64: _lib.PWS_F64,
}
_INTERP = {"bilinear": 0, "nearest": 1, "bicubic": 2}
_PADDING = {"zeros": 0, "border": 1, "reflection": 2}


_I64x10 = ctypes.c_int64 * 10


def _desc(t: torch.Tensor):
    """A pws_tensor for `t`, laid out by hand: {void *data; int32 dtype; int32 device; int64 size[4]; int64 stride[4]} is ten
    little-endian 64-bit words, and ONE ctypes array construction is several times cheaper than filling a Structure field
    by field -- the per-call host cost is what the 256 x 256 training shapes are bound by."""
    dev = t.device.index
    if dev is None:
        dev = torch.cuda.current_device()
    return _I64x10(t.data_ptr(), _DTYPES[t.dtype] | (dev << 32), *t.shape, *t.stride())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(t: torch.Tensor) -> int:
    """cudaStream_t of torch's current stream on t's device (the raw getter skips building a torch.cuda.Stream: 0.3 us vs 4)."""
    if _raw_stream is not None:
        return _raw_stream(t.get_device())
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(input: torch.Tensor, grid: torch.Tensor) -> None:
    if not (input.is_cuda and grid.is_cuda):
        raise RuntimeError(
            "pwstablenet_b200.grid_sample runs on CUDA tensors only (input on "
            f"{input.device}, grid on {grid.device}); there is no CPU fallback"
        )
    if input.device != grid.device:
        raise RuntimeError(
            "grid_sampler(): expected input and grid to be on same device, but input "
            f"is on {input.device} and grid is on {grid.device}"
        )
    if input.dim() != 4 or grid.dim() != 4:
        if input.dim() == 5 and grid.dim() == 5:
            raise NotImplementedError("pwstablenet_b200.grid_sample: 5-D (volumetric) sampling is out of scope")
        raise RuntimeError(
            "grid_sampler(): expected 4D input and grid with same number of dimensions, but got "
            f"input with sizes {list(input.shape)} and grid with sizes {list(grid.shape)}"
        )
    if input.dtype not in _DTYPES:
        raise NotImplementedError(f"pwstablenet_b200.grid_sample: unsupported frame dtype {input.dtype}")
    if grid.dtype != input.dtype and not (grid.dtype == torch.float32 and input.dtype in (torch.float16, torch.bfloat16)):
        raise RuntimeError(
            f"grid_sampler(): expected input and grid to have same dtype, but input has {input.dtype} "
            f"and grid has {grid.dtype} (extension: fp32 maps are accepted with fp16/bf16 frames)"
        )


def warp2d_forward(input: torch.Tensor, grid: torch.Tensor, padding: int, align_corners: bool,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """aten::grid_sampler_2d replacement (bilinear). Returns an NCHW-contiguous tensor, as ATen does
    (or fills the caller's `out`)."""
    lib = _lib.load()
    N, C = input.size(0), input.size(1)
    if out is None:
        out = torch.empty((N, C, grid.size(1), grid.size(2)), dtype=input.dtype, device=input.device)
    # (no device context here: the library selects the tensors' device itself and restores the caller's)
    rc = lib.pws_warp2d_forward(_desc(input), _desc(grid), _desc(out), 0, padding, int(align_corners), _stream(input))
    if rc:
        _lib.check(rc)
    return out


def _like_layout(t: torch.Tensor) -> torch.Tensor:
    """Uninitialised tensor with t's sizes; keeps t's strides when they are dense (the
    reference's maps are planar-stored permuted views), otherwise contiguous."""
    expected, dense = 1, t.numel() > 0
    for st, sz in sorted(zip(t.stride(), t.size())):
        if sz != 1:
            dense = dense and st == expected
            expected *= sz
    if dense:
        return torch.empty_strided(t.size(), t.stride(), dtype=t.dtype, device=t.device)
    return torch.empty(t.size(), dtype=t.dtype, device=t.device)


def warp2d_backward(grad_output: torch.Tensor, input: torch.Tensor, grid: torch.Tensor, padding: int,
                    align_corners: bool, output_mask=(True, True), grad_input: Optional[torch.Tensor] = None,
                    grad_grid: Optional[torch.Tensor] = None):
    """aten::grid_sampler_2d_backward replacement. Returns (grad_input | None, grad_grid | None);
    caller-provided buffers are filled when given (grad_input need not be zeroed)."""
    lib = _lib.load()
    half_frames = input.dtype in (torch.float16, torch.bfloat16)     # with an fp32 map or one of the frame's type
    gin = ggrid = None
    if output_mask[0]:
        if half_frames:
            # contributions are summed in fp32 and rounded to the frame type ONCE (a bf16 atomic would round after every add)
            if grad_input is not None and grad_input.dtype != torch.float32:
                raise RuntimeError("pwstablenet_b200: with 16-bit frames a caller-provided grad_input must be the fp32 accumulation buffer")
            gin = grad_input if grad_input is not None else torch.empty(input.size(), dtype=torch.float32, device=input.device)
        else:
            gin = grad_input if grad_input is not None else torch.empty(input.size(), dtype=input.dtype, device=input.device)
    if output_mask[1]:
        ggrid = grad_grid if grad_grid is not None else _like_layout(grid)
    rc = lib.pws_warp2d_backward(_desc(grad_output), _desc(input), _desc(grid),
                                 _desc(gin) if gin is not None else None, _desc(ggrid) if ggrid is not None else None,
                                 0, padding, int(align_corners), _stream(input))
    if rc:
        _lib.check(rc)
    if half_frames and gin is not None and grad_input is None:
        gin = gin.to(input.dtype)
    return gin, ggrid


class _Warp2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, input, grid, padding, align_corners):
        ctx.save_for_backward(input, grid)
        ctx.padding = padding
        ctx.align_corners = align_corners
        return warp2d_forward(input, grid, padding, align_corners)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        input, grid = ctx.saved_tensors
        mask = (ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        gin, ggrid = warp2d_backward(grad_output, input, grid, ctx.padding, ctx.align_corners, mask)
        return gin, ggrid, None, None


_ext = None


def torch_ext():
    """The compiled twin of this module's shim (csrc/torch_binding.cpp -> _pws_torch.so: descriptors, output allocation, stream
    lookup and the autograd node in C++; it calls the same libpwswarp.so entry points).  Halves the host cost of a call at the
    256 x 256 training shapes.  False when it is not built, when PWS_TORCH_EXT=0, or when PWS_LIB_PATH selects another kernel
    library (the extension is linked to the one next to it)."""
    global _ext
    if _ext is None:
        m = False
        if os.environ.get("PWS_TORCH_EXT", "1") != "0" and not os.environ.get("PWS_LIB_PATH"):
            try:
                _lib.load()
                from . import _pws_torch as m   # noqa: F811
                if m.abi_version() != _lib.ABI_VERSION:
                    m = False
            except ImportError:
                m = False
        _ext = m
    return _ext


def grid_sample(input: torch.Tensor, grid: torch.Tensor, mode: str = "bilinear", padding_mode: str = "zeros",
                align_corners: Optional[bool] = None) -> torch.Tensor:
    """Same contract as torch.nn.functional.grid_sample for 4-D CUDA tensors,
    mode='bilinear', padding_mode in {'zeros', 'border'}."""
    if mode not in _INTERP:
        raise ValueError(
            f"nn.functional.grid_sample(): expected mode to be 'bilinear', 'nearest' or 'bicubic', but got: '{mode}'")
    if padding_mode not in _PADDING:
        raise ValueError(
            "nn.functional.grid_sample(): expected padding_mode to be 'zeros', 'border', or 'reflection', "
            f"but got: '{padding_mode}'")
    if mode != "bilinear":
        raise NotImplementedError(f"pwstablenet_b200.grid_sample: mode='{mode}' is out of scope (bilinear only)")
    if padding_mode == "reflection":
        raise NotImplementedError("pwstablenet_b200.grid_sample: padding_mode='reflection' is out of scope")
    if align_corners is None:
        warnings.warn(
            "Default grid_sample and affine_grid behavior has changed to align_corners=False since 1.3.0. "
            "Please specify align_corners=True if the old behavior is desired. "
            "See the documentation of grid_sample for details.")
        align_corners = False
    _require_cuda(input, grid)
    ext = _ext if _ext is not None else torch_ext()
    if ext:
        return ext.grid_sample(input, grid, _PADDING[padding_mode], bool(align_corners))
    return _Warp2d.apply(input, grid, _PADDING[padding_mode], bool(align_corners))


def warp_taps(grid: torch.Tensor, in_h: int, in_w: int, padding_mode: str = "zeros", align_corners: bool = False,
              want_weights: bool = True):
    """Debug/parity: north-west tap indices, validity mask and weights the forward pass uses."""
    lib = _lib.load()
    if not grid.is_cuda or grid.dtype != torch.float32 or grid.dim() != 4:
        raise RuntimeError("warp_taps: grid must be a 4-D float32 CUDA tensor")
    N, Ho, Wo, _ = grid.shape
    x0 = torch.empty((N, Ho, Wo), dtype=torch.int32, device=grid.device)
    y0 = torch.empty_like(x0)
    mask = torch.empty((N, Ho, Wo), dtype=torch.uint8, device=grid.device)
    wts = torch.empty((N, Ho, Wo, 4), dtype=torch.float32, device=grid.device) if want_weights else None
    if True:
        rc = lib.pws_warp2d_taps(_desc(grid), in_h, in_w, x0.data_ptr(), y0.data_ptr(), mask.data_ptr(),
                                 wts.data_ptr() if wts is not None else None, _PADDING[padding_mode],
                                 int(align_corners), _stream(grid))
    _lib.check(rc)
    return x0, y0, mask, wts


_torch_grid_sample = None
_aten_lib = None


def _aten_grid_sampler_2d(input, grid, interpolation_mode, padding_mode, align_corners):
    """CUDA kernel of aten::grid_sampler_2d ($TORCH/include/ATen/native/cuda/GridSampler.h:12-17) while the override is installed."""
    if interpolation_mode != 0 or padding_mode not in (0, 1):
        raise NotImplementedError("pwstablenet_b200 (aten override): bilinear with zeros / border padding only; "
                                  "uninstall() the override for nearest / bicubic / reflection")
    ext = _ext if _ext is not None else torch_ext()
    if ext:
        return ext.warp2d_forward(input, grid, int(padding_mode), bool(align_corners))
    return warp2d_forward(input, grid, int(padding_mode), bool(align_corners))


def _aten_grid_sampler_2d_backward(grad_output, input, grid, interpolation_mode, padding_mode, align_corners, output_mask):
    """CUDA kernel of aten::grid_sampler_2d_backward (GridSampler.h:19-24).  ATen returns an undefined grad_input when
    output_mask[0] is false; a Python kernel cannot, it returns an empty tensor (autograd does not look at it)."""
    if interpolation_mode != 0 or padding_mode not in (0, 1):
        raise NotImplementedError("pwstablenet_b200 (aten override): bilinear with zeros / border padding only")
    gin, ggrid = warp2d_backward(grad_output, input, grid, int(padding_mode), bool(align_corners), (bool(output_mask[0]), True))
    if gin is None:
        gin = input.new_empty(0)
    return gin, ggrid


def install(aten_override: bool = False) -> None:
    """Route torch.nn.functional.grid_sample to this implementation so the reference's
    main_new.py / main.py run unmodified (they call `functional.grid_sample(...)` /
    `F.grid_sample(...)` through the module attribute).

    aten_override=True additionally registers the two C-ABI entry points as the CUDA kernels of aten::grid_sampler_2d and
    aten::grid_sampler_2d_backward (SURVEY 8(b): the optional torch.library override), for callers that hold their own
    reference to torch's function or reach the operator some other way (torch.grid_sampler, a scripted module).  The
    operator keeps ATen's autograd formula; only the kernels underneath change.  (torch routes bilinear + zeros +
    align_corners=True through cuDNN ABOVE this operator; the functional-level patch covers that case, the override alone
    does not.)"""
    global _torch_grid_sample, _aten_lib
    import torch.nn.functional as F
    _lib.load()
    if _torch_grid_sample is None:
        _torch_grid_sample = F.grid_sample
        F.grid_sample = grid_sample
    if aten_override and _aten_lib is None:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")      # "Overriding a previously registered kernel": that is the point
            lib = torch.library.Library("aten", "IMPL")
            lib.impl("grid_sampler_2d", _aten_grid_sampler_2d, "CUDA")
            lib.impl("grid_sampler_2d_backward", _aten_grid_sampler_2d_backward, "CUDA")
        _aten_lib = lib


def uninstall() -> None:
    global _torch_grid_sample, _aten_lib
    import torch.nn.functional as F
    if _torch_grid_sample is not None:
        F.grid_sample = _torch_grid_sample
        _torch_grid_sample = None
    if _aten_lib is not None:
        _aten_lib._destroy()     # drops the two registrations: ATen's own CUDA kernels are back
        _aten_lib = None
