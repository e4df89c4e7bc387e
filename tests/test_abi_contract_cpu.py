"""The argument contract of the eight C entry points (include/pwswarp.h), one table of faults per entry point.

CPU rows: every call is rejected before the library selects a device, so the data pointers are placeholders that are never
dereferenced (acceptance is never tested with them: an accepted call would launch on them).  GPU rows use real tensors:
C = 0 backward calls must return defined gradients and an all-zero grad_grid, as torch does, and a drift on another
device than the frame must be refused."""
import ctypes
import math

import pytest
import torch

FAKE = 0x1000   # never dereferenced: validation fails first

N, C, H, W, HO, WO, MH, MW = 2, 3, 16, 24, 32, 48, 8, 12


def _tensor(_lib, sizes, dtype=0, strides=None, device=0):
    t = _lib.PwsTensor()
    t.data = FAKE
    t.dtype = dtype
    t.device = device
    if strides is None:
        strides, s = [], 1
        for sz in reversed(sizes):
            strides.insert(0, s)
            s *= sz
    for i in range(4):
        t.size[i], t.stride[i] = sizes[i], strides[i]
    return t


def _ref(t):
    return ctypes.byref(t) if t is not None else None


@pytest.fixture()
def abi():
    from pwstablenet_b200 import _lib
    return _lib, _lib.load()


def _args(_lib):
    """A valid set of descriptors for every entry point; each row below breaks one of them."""
    T = lambda sizes, **kw: _tensor(_lib, sizes, **kw)   # noqa: E731
    return dict(frame=T((N, C, H, W)), grid=T((N, HO, WO, 2)), out=T((N, C, HO, WO)), gin=T((N, C, H, W)),
                ggrid=T((N, HO, WO, 2)), drift=T((N, MH, MW, 2)), glat=T((N, MH, MW, 2)), map_out=T((N, HO, WO, 2)),
                grid1=T((N, HO, WO, 2)), out1=T((N, C, HO, WO)), ggrid1=T((N, HO, WO, 2)), spec=True)


def _spec(_lib, drift):
    s = _lib.PwsMapSpec()
    s.drift = ctypes.pointer(drift) if drift is not None else None
    s.theta = FAKE
    s.base = _lib.PWS_BASE_AFFINE
    s.upsample = _lib.PWS_UP_ALIGNED
    s.map_h, s.map_w = MH, MW
    s.pre_add, s.pre_mul, s.post_div, s.post_add = 0.0, 1.0, 1.0, 0.0
    return s


def _call(_lib, lib, entry, a):
    spec = _spec(_lib, a["drift"]) if a["spec"] else None
    P = ctypes.POINTER(_lib.PwsTensor)

    def arr(*ts):
        return (P * len(ts))(*[ctypes.pointer(t) if t is not None else None for t in ts])

    if entry == "forward":
        return lib.pws_warp2d_forward(_ref(a["frame"]), _ref(a["grid"]), _ref(a["out"]), 0, 0, 0, None)
    if entry == "backward":
        return lib.pws_warp2d_backward(_ref(a["out"]), _ref(a["frame"]), _ref(a["grid"]), _ref(a["gin"]), _ref(a["ggrid"]),
                                       0, 0, 0, None)
    if entry == "taps":
        return lib.pws_warp2d_taps(_ref(a["grid"]), H, W, FAKE, FAKE, FAKE, None, 0, 0, None)
    if entry == "forward_fused":
        return lib.pws_warp2d_forward_fused(_ref(a["frame"]), _ref(spec) if spec else None, _ref(a["out"]), 0, 0, None)
    if entry == "backward_fused":
        return lib.pws_warp2d_backward_fused(_ref(a["out"]), _ref(a["frame"]), _ref(spec) if spec else None, _ref(a["gin"]),
                                             _ref(a["glat"]), None, 0, 0, None)
    if entry == "compose_map":
        return lib.pws_compose_map(_ref(spec) if spec else None, N, _ref(a["map_out"]), None)
    if entry == "stages_forward":
        return lib.pws_warp2d_stages_forward(_ref(a["frame"]), arr(a["grid"], a["grid1"]), arr(a["out"], a["out1"]), 2,
                                             0.0, 1.0, 1.0, 0.0, 0, 0, None)
    if entry == "stages_backward":
        return lib.pws_warp2d_stages_backward(arr(a["out"], a["out1"]), _ref(a["frame"]), arr(a["grid"], a["grid1"]),
                                              _ref(a["gin"]), arr(a["ggrid"], a["ggrid1"]), 2, 0.0, 1.0, 1.0, 0.0, 0, 0, None)
    raise AssertionError(entry)


# (entry point, fault, {argument: replacement}, expected status name, substrings of pws_last_error())
# Faults: null required descriptor, wrong sizes, wrong dtype, another device, non-dense grad_input, empty spatial
# dimension, maps of different sizes (stages), drift on another device.  F16 = 1, device 1 = another device.
def _rows():
    T = _tensor   # each row builds its replacement descriptors from _lib (the lambdas' argument)
    rows = [
        # pws_warp2d_forward
        ("forward", "null input", lambda l: dict(frame=None), "EINVAL", ("not be undefined",)),
        ("forward", "null output", lambda l: dict(out=None), "EINVAL", ("null", "output")),
        ("forward", "output sizes", lambda l: dict(out=T(l, (N, C, HO, WO + 1))), "EINVAL", ("output", "expected sizes")),
        ("forward", "output dtype", lambda l: dict(out=T(l, (N, C, HO, WO), dtype=1)), "EINVAL", ("output", "dtype")),
        ("forward", "output device", lambda l: dict(out=T(l, (N, C, HO, WO), device=1)), "EINVAL", ("output", "device")),
        ("forward", "empty spatial", lambda l: dict(frame=T(l, (N, C, 0, W))), "EINVAL", ("non-empty spatial dimensions",)),
        # pws_warp2d_backward
        ("backward", "null grad_output", lambda l: dict(out=None), "EINVAL", ("null", "grad_output")),
        ("backward", "grad_output sizes", lambda l: dict(out=T(l, (N, C + 1, HO, WO))), "EINVAL",
         ("grad_output", "expected sizes")),
        ("backward", "grad_output dtype", lambda l: dict(out=T(l, (N, C, HO, WO), dtype=1)), "EINVAL", ("grad_output", "dtype")),
        ("backward", "grad_output device", lambda l: dict(out=T(l, (N, C, HO, WO), device=1)), "EINVAL",
         ("grad_output", "device")),
        ("backward", "grad_input not dense", lambda l: dict(gin=T(l, (N, C, H, W), strides=(C * H * W, 1, W * C, C))),
         "EINVAL", ("grad_input", "contiguous")),
        ("backward", "grad_input sizes", lambda l: dict(gin=T(l, (N, C, H, W + 1))), "EINVAL", ("grad_input", "expected sizes")),
        ("backward", "grad_input dtype", lambda l: dict(gin=T(l, (N, C, H, W), dtype=1)), "EINVAL", ("grad_input", "dtype")),
        ("backward", "grad_input device", lambda l: dict(gin=T(l, (N, C, H, W), device=1)), "EINVAL", ("grad_input", "device")),
        ("backward", "grad_grid sizes", lambda l: dict(ggrid=T(l, (N, HO, WO + 1, 2))), "EINVAL", ("grad_grid", "expected sizes")),
        ("backward", "grad_grid dtype", lambda l: dict(ggrid=T(l, (N, HO, WO, 2), dtype=1)), "EINVAL", ("grad_grid", "dtype")),
        ("backward", "grad_grid device", lambda l: dict(ggrid=T(l, (N, HO, WO, 2), device=1)), "EINVAL", ("grad_grid", "device")),
        ("backward", "empty spatial", lambda l: dict(frame=T(l, (N, C, H, 0)), gin=None), "EINVAL",
         ("non-empty spatial dimensions",)),
        # pws_warp2d_taps
        ("taps", "null grid", lambda l: dict(grid=None), "EINVAL", ("null",)),
        ("taps", "grid dtype", lambda l: dict(grid=T(l, (N, HO, WO, 2), dtype=1)), "EUNSUPPORTED", ("f32",)),
        # pws_warp2d_forward_fused
        ("forward_fused", "null input", lambda l: dict(frame=None), "EINVAL", ("null tensor descriptor",)),
        ("forward_fused", "null output", lambda l: dict(out=None), "EINVAL", ("null tensor descriptor",)),
        ("forward_fused", "null spec", lambda l: dict(spec=False), "EINVAL", ("map spec",)),
        ("forward_fused", "output channels", lambda l: dict(out=T(l, (N, C + 1, HO, WO))), "EINVAL", ("output", "batch/channels")),
        ("forward_fused", "output device", lambda l: dict(out=T(l, (N, C, HO, WO), device=1)), "EINVAL", ("output", "device")),
        ("forward_fused", "empty spatial", lambda l: dict(frame=T(l, (N, C, 0, W))), "EINVAL", ("non-empty spatial dimensions",)),
        ("forward_fused", "drift sizes", lambda l: dict(drift=T(l, (N, MH + 1, MW, 2))), "EINVAL", ("drift", "sizes")),
        ("forward_fused", "drift device", lambda l: dict(drift=T(l, (N, MH, MW, 2), device=1)), "EINVAL", ("drift", "device")),
        # pws_warp2d_backward_fused
        ("backward_fused", "null grad_output", lambda l: dict(out=None), "EINVAL", ("null tensor descriptor",)),
        ("backward_fused", "null input", lambda l: dict(frame=None), "EINVAL", ("null tensor descriptor",)),
        ("backward_fused", "grad_output channels", lambda l: dict(out=T(l, (N, C + 1, HO, WO))), "EINVAL",
         ("grad_output", "batch/channels")),
        ("backward_fused", "grad_output dtype", lambda l: dict(out=T(l, (N, C, HO, WO), dtype=1)), "EINVAL", ("grad_output",)),
        ("backward_fused", "grad_output device", lambda l: dict(out=T(l, (N, C, HO, WO), device=1)), "EINVAL",
         ("grad_output", "device")),
        ("backward_fused", "grad_input not dense", lambda l: dict(gin=T(l, (N, C, H, W), strides=(C * H * W, 1, W * C, C))),
         "EINVAL", ("grad_input", "contiguous")),
        ("backward_fused", "grad_input dtype", lambda l: dict(gin=T(l, (N, C, H, W), dtype=1)), "EINVAL", ("grad_input", "f32")),
        ("backward_fused", "grad_input device", lambda l: dict(gin=T(l, (N, C, H, W), device=1)), "EINVAL",
         ("grad_input", "device")),
        ("backward_fused", "glattice sizes", lambda l: dict(glat=T(l, (N, MH, MW + 1, 2))), "EINVAL", ("glattice", "expected sizes")),
        ("backward_fused", "glattice device", lambda l: dict(glat=T(l, (N, MH, MW, 2), device=1)), "EINVAL",
         ("glattice", "device")),
        ("backward_fused", "empty spatial", lambda l: dict(frame=T(l, (N, C, H, 0)), gin=None), "EINVAL",
         ("non-empty spatial dimensions",)),
        ("backward_fused", "drift device", lambda l: dict(drift=T(l, (N, MH, MW, 2), device=1)), "EINVAL", ("drift", "device")),
        # pws_compose_map
        ("compose_map", "null output", lambda l: dict(map_out=None), "EINVAL", ("null", "output")),
        ("compose_map", "null spec", lambda l: dict(spec=False), "EINVAL", ("map spec",)),
        ("compose_map", "output batch", lambda l: dict(map_out=T(l, (N + 1, HO, WO, 2))), "EINVAL", ("output",)),
        ("compose_map", "output dtype", lambda l: dict(map_out=T(l, (N, HO, WO, 2), dtype=1)), "EINVAL", ("output", "f32")),
        ("compose_map", "drift device", lambda l: dict(drift=T(l, (N, MH, MW, 2), device=1)), "EINVAL", ("drift", "device")),
        # pws_warp2d_stages_forward
        ("stages_forward", "null input", lambda l: dict(frame=None), "EINVAL", ("null",)),
        ("stages_forward", "null output", lambda l: dict(out1=None), "EINVAL", ("null", "output")),
        ("stages_forward", "output sizes", lambda l: dict(out1=T(l, (N, C, HO, WO + 1))), "EINVAL", ("output", "expected sizes")),
        ("stages_forward", "output dtype", lambda l: dict(out1=T(l, (N, C, HO, WO), dtype=1)), "EINVAL", ("output 1", "dtype")),
        ("stages_forward", "output device", lambda l: dict(out1=T(l, (N, C, HO, WO), device=1)), "EINVAL", ("output", "device")),
        ("stages_forward", "maps of different sizes", lambda l: dict(grid1=T(l, (N, HO, WO + 1, 2))), "EINVAL", ("size",)),
        ("stages_forward", "map dtype", lambda l: dict(grid1=T(l, (N, HO, WO, 2), dtype=1)), "EINVAL", ("one dtype",)),
        ("stages_forward", "map device", lambda l: dict(grid1=T(l, (N, HO, WO, 2), device=1)), "EINVAL", ("same device",)),
        ("stages_forward", "empty spatial", lambda l: dict(frame=T(l, (N, C, 0, W))), "EINVAL", ("non-empty spatial dimensions",)),
        # pws_warp2d_stages_backward
        ("stages_backward", "null input", lambda l: dict(frame=None), "EINVAL", ("null",)),
        ("stages_backward", "null grad_output", lambda l: dict(out1=None), "EINVAL", ("null", "grad_output")),
        ("stages_backward", "grad_output dtype", lambda l: dict(out1=T(l, (N, C, HO, WO), dtype=1)), "EINVAL",
         ("grad_output 1", "dtype")),
        ("stages_backward", "grad_output device", lambda l: dict(out1=T(l, (N, C, HO, WO), device=1)), "EINVAL",
         ("grad_output 1", "device")),
        ("stages_backward", "grad_grid dtype", lambda l: dict(ggrid1=T(l, (N, HO, WO, 2), dtype=1)), "EINVAL",
         ("grad_grid 1", "dtype")),
        ("stages_backward", "grad_grid device", lambda l: dict(ggrid1=T(l, (N, HO, WO, 2), device=1)), "EINVAL",
         ("grad_grid 1", "device")),
        ("stages_backward", "grad_input not dense", lambda l: dict(gin=T(l, (N, C, H, W), strides=(C * H * W, 1, W * C, C))),
         "EINVAL", ("grad_input", "contiguous")),
        ("stages_backward", "grad_input dtype", lambda l: dict(gin=T(l, (N, C, H, W), dtype=1)), "EINVAL", ("grad_input", "f32")),
        ("stages_backward", "grad_input device", lambda l: dict(gin=T(l, (N, C, H, W), device=1)), "EINVAL",
         ("grad_input", "device")),
        ("stages_backward", "maps of different sizes", lambda l: dict(grid1=T(l, (N, HO + 1, WO, 2))), "EINVAL", ("size",)),
        ("stages_backward", "empty spatial", lambda l: dict(frame=T(l, (N, C, H, 0)), gin=None), "EINVAL",
         ("non-empty spatial dimensions",)),
    ]
    return [pytest.param(*r, id=f"{r[0]}-{r[1].replace(' ', '_')}") for r in rows]


@pytest.mark.parametrize("entry,fault,change,status,words", _rows())
def test_fault_is_rejected_before_device_selection(abi, entry, fault, change, status, words):
    _lib, lib = abi
    a = _args(_lib)
    a.update(change(_lib))
    rc = _call(_lib, lib, entry, a)
    msg = _lib.last_error()
    assert rc == getattr(_lib, "PWS_" + status), (fault, rc, msg)
    for w in words:
        assert w in msg, (fault, msg)


def test_non_dense_grad_grid_with_no_channels_is_unsupported(abi):
    """C = 0 leaves nothing to scatter, so every gradient buffer is zero-filled with one memset over its span; a grad_grid
    with gaps (only a direct C caller can pass one) cannot be, and the call says so instead of leaving it unwritten."""
    _lib, lib = abi
    frame = _tensor(_lib, (N, 0, H, W), strides=(H * W, H * W, W, 1))
    gout = _tensor(_lib, (N, 0, HO, WO))
    grid = _tensor(_lib, (N, HO, WO, 2))
    gapped = _tensor(_lib, (N, HO, WO, 2), strides=(HO * WO * 4, WO * 4, 4, 1))
    rc = lib.pws_warp2d_backward(_ref(gout), _ref(frame), _ref(grid), None, _ref(gapped), 0, 0, 0, None)
    assert rc == _lib.PWS_EUNSUPPORTED and "grad_grid" in _lib.last_error(), _lib.last_error()
    P = ctypes.POINTER(_lib.PwsTensor)
    rc = lib.pws_warp2d_stages_backward((P * 1)(ctypes.pointer(gout)), _ref(frame), (P * 1)(ctypes.pointer(grid)), None,
                                        (P * 1)(ctypes.pointer(gapped)), 1, 0.0, 1.0, 1.0, 0.0, 0, 0, None)
    assert rc == _lib.PWS_EUNSUPPORTED and "grad_grid 0" in _lib.last_error(), _lib.last_error()


# ---- GPU rows: real tensors only --------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as m
    from pwstablenet_b200 import _lib
    _lib.load()
    return m


def _no_channel_inputs(n, dtype, frame_grad):
    frame = torch.empty(n, 0, 20, 28, device="cuda", dtype=dtype).requires_grad_(frame_grad)
    grid = (torch.rand(n, 2, 12, 16, device="cuda") * 2.2 - 1.1).to(dtype).permute(0, 2, 3, 1).requires_grad_(True)
    return frame, grid


def _check_no_channel_grads(frame, grid, frame_grad):
    torch.cuda.synchronize()
    assert grid.grad is not None and grid.grad.shape == grid.shape and grid.grad.dtype == grid.dtype
    assert torch.equal(grid.grad, torch.zeros_like(grid))           # what torch returns: no channel, no gradient
    if frame_grad:
        assert frame.grad is not None and frame.grad.shape == frame.shape and frame.grad.dtype == frame.dtype
    else:
        assert frame.grad is None


@pytest.mark.gpu
@pytest.mark.parametrize("shim", ["compiled", "ctypes"])
@pytest.mark.parametrize("frame_grad", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("n", [1, 2])
def test_grid_sample_with_no_channels_has_zero_gradients(pw, n, dtype, frame_grad, shim):
    from pwstablenet_b200 import functional
    if shim == "compiled" and not functional.torch_ext():
        pytest.fail("pwstablenet_b200/_pws_torch.so is not built")
    frame, grid = _no_channel_inputs(n, dtype, frame_grad)
    for _ in range(2):
        frame.grad = grid.grad = None
        torch.full_like(grid, float("nan"))   # freed at once: the caching allocator hands this block to grid.grad
        out = pw.grid_sample(frame, grid, align_corners=False) if shim == "compiled" else \
            functional._Warp2d.apply(frame, grid, 0, False)
        assert out.shape == (n, 0, 12, 16)
        out.sum().backward()
        _check_no_channel_grads(frame, grid, frame_grad)
    ref_frame = frame.detach().float().cpu().requires_grad_(frame_grad)
    ref_grid = grid.detach().float().cpu().requires_grad_(True)
    torch.nn.functional.grid_sample(ref_frame, ref_grid, align_corners=False).sum().backward()
    assert torch.equal(ref_grid.grad, grid.grad.float().cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("frame_grad", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("n", [1, 2])
def test_warp_stages_with_no_channels_has_zero_gradients(pw, n, dtype, frame_grad):
    frame, grid = _no_channel_inputs(n, dtype, frame_grad)
    grid2 = grid.detach().clone().requires_grad_(True)      # interleaved layout
    torch.full_like(grid, float("nan"))
    outs = pw.warp_stages(frame, [grid, grid2], pre=(1.0, 127.5), post=(127.5, -1.0))
    sum(o.sum() for o in outs).backward()
    _check_no_channel_grads(frame, grid, frame_grad)
    _check_no_channel_grads(frame, grid2, frame_grad)


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("with_gin", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("n", [1, 2])
def test_backward_abi_with_no_channels_overwrites_grad_grid(pw, n, dtype, with_gin, planar):
    """pws_warp2d_backward directly, with NaN-filled grad_grid buffers: dense interleaved and the planar-permuted layout
    the shims allocate for netG's maps.  Both must come back all zeros, and grad_input too."""
    from pwstablenet_b200 import _lib, functional
    lib = _lib.load()
    frame = torch.empty(n, 0, 20, 28, device="cuda", dtype=dtype)
    grid = (torch.rand(n, 12, 16, 2, device="cuda") * 2 - 1).to(dtype)
    gout = torch.empty(n, 0, 12, 16, device="cuda", dtype=dtype)
    if planar:
        ggrid = torch.full((n, 2, 12, 16), float("nan"), device="cuda", dtype=dtype).permute(0, 2, 3, 1)
    else:
        ggrid = torch.full((n, 12, 16, 2), float("nan"), device="cuda", dtype=dtype)
    gin = torch.empty(n, 0, 20, 28, device="cuda") if with_gin else None     # torch's strides: (H*W, H*W, W, 1)
    rc = lib.pws_warp2d_backward(functional._desc(gout), functional._desc(frame), functional._desc(grid),
                                 functional._desc(gin) if gin is not None else None, functional._desc(ggrid),
                                 0, 0, 0, functional._stream(frame))
    _lib.check(rc)
    torch.cuda.synchronize()
    assert not math.isnan(float(ggrid.float().sum()))
    assert torch.equal(ggrid, torch.zeros_like(ggrid))


@pytest.mark.gpu
def test_drift_on_another_device_is_refused(pw):
    from pwstablenet_b200 import _lib, compose
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    frame = torch.rand(1, 3, 16, 16, device="cuda:0")
    drift = torch.zeros(1, 16, 16, 2, device="cuda:1")
    with pytest.raises(RuntimeError, match="drift"):
        pw.warp_fused(frame, drift=drift)
    with pytest.raises(RuntimeError, match="drift"):
        pw.warp_fused(frame.requires_grad_(True), drift=drift)
    keep = []
    spec = compose._spec(1, drift, "none", None, False, None, None, (0.0, 1.0), (1.0, 0.0), keep)
    out = torch.empty(1, 16, 16, 2, device="cuda:0")
    rc = _lib.load().pws_compose_map(ctypes.byref(spec), 1, ctypes.byref(compose._desc(out)), None)
    assert rc == _lib.PWS_EINVAL and "drift" in _lib.last_error()
