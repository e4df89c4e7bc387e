"""Half-precision netG through the call-site fusions: f16 / bf16 frames and maps in `pw.warp_stages`, 16-bit lattices in
`pw.warp_fused` / `pw.compose_map`.

warp_stages contract with a 16-bit frame T (maps f32 or T, one dtype for all stages):
  * forward   == the unfused sequence `pw.grid_sample((f + a) * b, g) / d + e` evaluated by torch in T  (torch.equal);
                 with T maps also == the same sequence through aten.grid_sampler_2d                   (torch.equal)
  * grad_grid == autograd of that unfused sequence, in the map's dtype and stride                      (torch.equal)
  * grad_input: fp32 sums times b over all stages, rounded to T once: within finfo(T).eps x max of ATen's fp32 backward on
    the upcast, post-scaled grad_outputs; the raw fp32 buffer of the C entry point within 1e-4 x max.
warp_fused / compose_map with a 16-bit drift == the same call with drift.float(), bit for bit (byte for byte for uint8)."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]
PAD = {"zeros": 0, "border": 1}
PRE, POST = (1.0, 127.5), (127.5, -1.0)


@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()
    return pw


def last_kernel():
    from pwstablenet_b200 import _lib
    return _lib.last_kernel()


def cascade_maps(n, h, w, align, dtype, layout, k=3, seed=3):
    """k maps that refine each other, in `dtype`; planar = netG's storage (coordinate stride h*w), else interleaved."""
    base = synth.make_map("smooth", n, h, w, align, seed=seed)
    rng = np.random.default_rng(seed + 100)
    maps = []
    for i in range(k):
        m = torch.from_numpy((base + rng.standard_normal(base.shape).astype(np.float32) * (0.004 * i)).astype(np.float32))
        m = m.cuda().to(dtype)
        if layout == "planar":
            m = m.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
        maps.append(m)
    return maps


def frames(n, c, h, w, dtype, seed):
    return (torch.from_numpy(synth.make_frames(n, c, h, w, seed=seed)).cuda() / 127.5 - 1).to(dtype)   # [-1, 1], as trained


def aten_sampler(x, g, mode, padding_mode, align_corners):
    return torch.ops.aten.grid_sampler_2d(x, g, 0, PAD[padding_mode], align_corners)


def unfused(frame, grids, pad, align, pre, post, sampler):
    """The sequence warp_stages replaces; on a 16-bit frame torch rounds after every elementwise op."""
    return [sampler((frame + pre[0]) * pre[1], g, mode="bilinear", padding_mode=pad, align_corners=align) / post[0] + post[1]
            for g in grids]


def map_dtype_of(dtype, which):
    return torch.float32 if which == "f32" else dtype


# ---- 1. forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["planar", "interleaved"])
@pytest.mark.parametrize("shape", [(16, 3, 256, 256), (2, 1, 256, 256), (3, 3, 100, 180)])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("maps", ["f32", "same"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_half_stages_forward_is_bit_identical_to_the_16bit_sequence(pw, dtype, maps, pad, align, shape, layout):
    n, c, h, w = shape
    frame = frames(n, c, h, w, dtype, seed=5)
    grids = cascade_maps(n, h, w, align, map_dtype_of(dtype, maps), layout)
    for pre, post in ((PRE, POST), ((0.0, 1.0), (1.0, 0.0))):
        got = pw.warp_stages(frame, grids, pad, align, pre=pre, post=post)
        assert last_kernel() == "stages_fwd_16"
        want = unfused(frame, grids, pad, align, pre, post, pw.grid_sample)
        for a, b in zip(got, want):
            assert a.dtype == dtype and a.shape == b.shape
            assert torch.equal(a, b)
        if maps == "same":
            for a, b in zip(got, unfused(frame, grids, pad, align, pre, post, aten_sampler)):
                assert torch.equal(a, b)


# ---- 2. backward --------------------------------------------------------------------------------------------------------
def stage_grads(fn, frame, grids, gouts, want_frame, want_maps=None, kernels=None):
    """Gradients of fn through autograd.  `kernels` collects pws_last_kernel() as seen by the thread that ran the backward
    (autograd runs CUDA backward nodes on its own device thread, and the name is thread-local)."""
    f = frame.clone().requires_grad_(want_frame)
    gs = [g.clone().requires_grad_(True if want_maps is None else want_maps[i]) for i, g in enumerate(grids)]
    if kernels is not None:
        for g in gs:
            if g.requires_grad:
                g.register_hook(lambda grad: kernels.append(last_kernel()))
    outs = fn(f, gs)
    torch.autograd.backward(list(outs), gouts)
    return [g.grad for g in gs], f.grad


def gin_reference(frame, grids, gouts, pad, align):
    """ATen's fp32 backward on the upcast inputs: post-scaled grad_outputs (rounded to T, as the sequence's autograd hands
    them to the sampler), pre-scaled frame, summed over stages, times b."""
    fpre = ((frame + PRE[0]) * PRE[1]).float()
    acc = torch.zeros(frame.shape, dtype=torch.float32, device=frame.device)
    for g, go in zip(grids, gouts):
        gi, _ = torch.ops.aten.grid_sampler_2d_backward((go / POST[0]).float(), fpre, g.float(), 0, PAD[pad], align, (True, False))
        acc += gi
    return acc * PRE[1]


@pytest.mark.parametrize("layout", ["planar", "interleaved"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("maps", ["f32", "same"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_half_stages_backward_matches_autograd_of_the_16bit_sequence(pw, dtype, maps, pad, align, layout):
    n, c, h, w = 4, 3, 128, 192
    frame = frames(n, c, h, w, dtype, seed=6)
    grids = cascade_maps(n, h, w, align, map_dtype_of(dtype, maps), layout, seed=8)
    gouts = [torch.from_numpy(synth.make_gout(n, c, h, w, seed=20 + k)).cuda().to(dtype) for k in range(3)]
    fused = lambda f, gs: pw.warp_stages(f, gs, pad, align, pre=PRE, post=POST)
    ours = lambda f, gs: unfused(f, gs, pad, align, PRE, POST, pw.grid_sample)

    gg_f, gin_none = stage_grads(fused, frame, grids, gouts, False)
    gg_o, _ = stage_grads(ours, frame, grids, gouts, False)
    assert gin_none is None
    for a, b, g in zip(gg_f, gg_o, grids):
        assert a.dtype == g.dtype and a.stride() == g.stride() == b.stride()
        assert torch.equal(a, b)

    # grad_input too: the map gradients do not change, grad_input is fp32 sums rounded once
    seen = []
    gg_f2, gin = stage_grads(fused, frame, grids, gouts, True, kernels=seen)
    assert seen == ["stages_bwd_16"] * 3
    for a, b in zip(gg_f2, gg_f):
        assert torch.equal(a, b)
    ref = gin_reference(frame, grids, gouts, pad, align)
    assert gin.dtype == dtype
    assert float((gin.float() - ref).abs().max()) <= torch.finfo(dtype).eps * float(ref.abs().max())

    # output masks: only the middle map asks
    gg_m, gin_m = stage_grads(fused, frame, grids, gouts, False, want_maps=[False, True, False])
    assert gg_m[0] is None and gg_m[2] is None and gin_m is None
    assert torch.equal(gg_m[1], gg_f[1])


def test_half_stages_raw_fp32_grad_input_buffer(pw):
    """The C entry point leaves the fp32 sums in the caller's f32 buffer: within 1e-4 x max of ATen's fp32 kernel."""
    from pwstablenet_b200 import _lib, compose
    lib = _lib.load()
    n, c, h, w = 4, 3, 128, 192
    for dtype in DTYPES:
        for maps in ("f32", "same"):
            frame = frames(n, c, h, w, dtype, seed=7)
            grids = cascade_maps(n, h, w, False, map_dtype_of(dtype, maps), "planar", seed=9)
            gouts = [torch.from_numpy(synth.make_gout(n, c, h, w, seed=30 + k)).cuda().to(dtype) for k in range(3)]
            gin = torch.full(frame.shape, float("nan"), dtype=torch.float32, device="cuda")   # need not arrive zeroed
            keep = []
            rc = lib.pws_warp2d_stages_backward(compose._desc_ptrs(gouts, keep), ctypes.byref(compose._desc(frame)),
                                                compose._desc_ptrs(grids, keep), ctypes.byref(compose._desc(gin)),
                                                compose._desc_ptrs([None] * 3, keep), 3, PRE[0], PRE[1], POST[0], POST[1],
                                                0, 0, compose._stream(frame))
            _lib.check(rc)
            assert last_kernel() == "stages_bwd_16"
            ref = gin_reference(frame, grids, gouts, "zeros", False)
            assert float((gin - ref).abs().max()) <= 1e-4 * float(ref.abs().max()), (dtype, maps)


# ---- 3. a half-precision map network trained through warp_stages ------------------------------------------------------
class MapNet(torch.nn.Module):
    """netG in miniature: one trunk, three cascade maps = identity + a small tanh drift, stored planar.  One head emits all
    six map channels, so the gradient into the trunk is assembled from disjoint slices (exact in any order)."""

    def __init__(self):
        super().__init__()
        self.trunk = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.head = torch.nn.Conv2d(8, 6, 3, padding=1)

    def forward(self, x, base):
        d = 0.05 * torch.tanh(self.head(torch.tanh(self.trunk(x))))
        return [(base + d[:, 2 * k:2 * k + 2]).permute(0, 2, 3, 1) for k in range(3)]


@pytest.mark.parametrize("dtype", DTYPES)
def test_half_precision_map_net_trains_through_warp_stages(pw, dtype):
    n, c, h, w = 4, 3, 64, 96
    torch.manual_seed(0)
    net = MapNet().cuda().to(dtype)
    twin = copy.deepcopy(net)
    x = frames(n, c, h, w, dtype, seed=40)
    target = torch.from_numpy(synth.make_frames(n, c, h, w, seed=41)).cuda() / 127.5 - 1
    base = torch.from_numpy(synth.identity_map(n, h, w, False)).cuda().permute(0, 3, 1, 2).to(dtype)
    prev = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        outs = pw.warp_stages(x, net(x, base), "zeros", False, pre=PRE, post=POST)
        sum(((o.float() - target) ** 2).mean() for o in outs).backward()
        outs2 = unfused(x, twin(x, base), "zeros", False, PRE, POST, pw.grid_sample)
        sum(((o.float() - target) ** 2).mean() for o in outs2).backward()
    finally:
        torch.backends.cudnn.deterministic = prev
    for a, b in zip(outs, outs2):
        assert torch.equal(a, b)
    for (name, p), q in zip(net.named_parameters(), twin.parameters()):
        assert p.grad is not None and p.grad.dtype == dtype
        assert torch.equal(p.grad, q.grad), name


# ---- 4. errors ----------------------------------------------------------------------------------------------------------
def test_half_stages_errors(pw):
    from pwstablenet_b200 import _lib, compose
    lib = _lib.load()
    f16 = torch.zeros(1, 3, 8, 8, device="cuda", dtype=torch.float16)
    g32 = torch.zeros(1, 8, 8, 2, device="cuda")
    g16 = g32.half()
    with pytest.raises(RuntimeError, match="one dtype"):
        pw.warp_stages(f16, [g32, g16])                                       # mixed map dtypes
    with pytest.raises(RuntimeError):
        pw.warp_stages(f16.float(), [g16])                                    # f32 frame, 16-bit map
    with pytest.raises(RuntimeError):
        pw.warp_stages(f16, [g16.bfloat16()])                                 # another 16-bit type
    with pytest.raises(RuntimeError):
        pw.warp_stages(torch.zeros(1, 2, 8, 8, device="cuda", dtype=torch.float16), [g16])    # C must be 1 or 3
    with pytest.raises(RuntimeError):
        pw.warp_stages(f16.double(), [g32.double()])

    # the C entry points check the same without the Python shim in front
    keep = []
    outs = [torch.empty(1, 3, 8, 8, device="cuda", dtype=torch.float16) for _ in range(2)]
    rc = lib.pws_warp2d_stages_forward(ctypes.byref(compose._desc(f16)), compose._desc_ptrs([g32, g16], keep),
                                       compose._desc_ptrs(outs, keep), 2, 0.0, 1.0, 1.0, 0.0, 0, 0, None)
    assert rc == _lib.PWS_EINVAL and "one dtype" in _lib.last_error()
    rc = lib.pws_warp2d_stages_forward(ctypes.byref(compose._desc(f16.float())), compose._desc_ptrs([g16], keep),
                                       compose._desc_ptrs([outs[0].float()], keep), 1, 0.0, 1.0, 1.0, 0.0, 0, 0, None)
    assert rc == _lib.PWS_EINVAL

    def backward(gouts, gin, ggrids, frame=f16, grids=(g16,)):
        return lib.pws_warp2d_stages_backward(compose._desc_ptrs(gouts, keep), ctypes.byref(compose._desc(frame)),
                                              compose._desc_ptrs(list(grids), keep),
                                              ctypes.byref(gin) if gin is not None else None,
                                              compose._desc_ptrs(ggrids, keep), len(grids), 0.0, 1.0, 1.0, 0.0, 0, 0, None)

    go = torch.zeros(1, 3, 8, 8, device="cuda", dtype=torch.float16)
    gin32 = torch.empty(1, 3, 8, 8, device="cuda")
    assert backward([go], compose._desc(gin32), [torch.empty_like(g16)]) == _lib.PWS_OK
    torch.cuda.synchronize()
    # a 16-bit grad_input buffer: 16-bit frames accumulate in fp32
    assert backward([go], compose._desc(gin32.half()), [None]) == _lib.PWS_EINVAL
    assert "f32" in _lib.last_error()
    # a grad_grid of another dtype than its map
    assert backward([go], None, [torch.empty_like(g32)]) == _lib.PWS_EINVAL


def _on_other_device(desc):
    desc.device = desc.device + 1
    return desc


def test_half_stages_backward_checks_every_device(pw):
    """Every gout, ggrid and gin must be on the input's device.  Run on two devices when there are two; the descriptors
    of the other check carry another ordinal (validation runs before any launch, so nothing touches that memory)."""
    from pwstablenet_b200 import _lib, compose
    lib = _lib.load()
    f = torch.zeros(1, 3, 8, 8, device="cuda", dtype=torch.float16)
    g = torch.zeros(1, 8, 8, 2, device="cuda", dtype=torch.float16)
    go = torch.zeros(1, 3, 8, 8, device="cuda", dtype=torch.float16)
    gin = torch.empty(1, 3, 8, 8, device="cuda")
    gg = torch.empty_like(g)
    two = torch.cuda.device_count() >= 2

    def moved(t):
        if two:
            return compose._desc(t.to("cuda:1"))
        return _on_other_device(compose._desc(t))

    def call(go_d, gin_d, gg_d):
        arr_go = (ctypes.POINTER(_lib.PwsTensor) * 1)(ctypes.pointer(go_d))
        arr_gg = (ctypes.POINTER(_lib.PwsTensor) * 1)(ctypes.pointer(gg_d) if gg_d is not None else None)
        keep = []
        return lib.pws_warp2d_stages_backward(arr_go, ctypes.byref(compose._desc(f)), compose._desc_ptrs([g], keep),
                                              ctypes.byref(gin_d) if gin_d is not None else None, arr_gg, 1,
                                              0.0, 1.0, 1.0, 0.0, 0, 0, None)

    assert call(compose._desc(go), compose._desc(gin), compose._desc(gg)) == _lib.PWS_OK
    torch.cuda.synchronize()
    assert call(moved(go), None, None) == _lib.PWS_EINVAL and "grad_output" in _lib.last_error()
    assert call(compose._desc(go), None, moved(gg)) == _lib.PWS_EINVAL and "grad_grid" in _lib.last_error()
    assert call(compose._desc(go), moved(gin), None) == _lib.PWS_EINVAL and "grad_input" in _lib.last_error()


# ---- 5. 16-bit lattices in warp_fused / compose_map ---------------------------------------------------------------------
FUSED_CASES = [
    dict(base="identity", upsample=None),
    dict(base="affine", upsample=None),
    dict(base="affine", upsample="aligned"),
    dict(base="identity", upsample="half_pixel"),
    dict(base="none", upsample="aligned"),
]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", FUSED_CASES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
def test_fused_with_16bit_drift_equals_the_upcast_drift(pw, dtype, case, pad, align):
    n, C, H, W = 2, 3, 90, 144
    h, w = (H, W) if case["upsample"] is None else (24, 40)
    frm = dev(synth.make_frames(n, C, H, W, seed=8)) / 127.5 - 1
    rng = np.random.default_rng(9)
    drift = (np.tanh(rng.standard_normal((n, 2, h, w))) * 0.035).astype(np.float32)
    if case["base"] == "none":
        drift = np.ascontiguousarray(synth.make_map("smooth", n, h, w, True, seed=9).transpose(0, 3, 1, 2))
    theta = dev(np.array([[[1.01, 0.02, 0.0], [-0.02, 0.99, 0.01]]] * n, np.float32))
    d16 = dev(drift).to(dtype).permute(0, 2, 3, 1)                       # netG's planar output, permuted
    for d in (d16, d16.contiguous()):                                    # ... and an interleaved lattice (pair loads)
        kw = dict(base=case["base"], theta=theta if case["base"] == "affine" else None, upsample=case["upsample"])
        assert torch.equal(pw.compose_map(n, (H, W), drift=d, **kw), pw.compose_map(n, (H, W), drift=d.float(), **kw))
        for extra in (dict(), dict(pre=(1.0, 127.5), post=(127.5, -1.0))):
            a = pw.warp_fused(frm, drift=d, out_size=(H, W), padding_mode=pad, align_corners=align, **kw, **extra)
            b = pw.warp_fused(frm, drift=d.float(), out_size=(H, W), padding_mode=pad, align_corners=align, **kw, **extra)
            assert torch.equal(a, b)
        f16 = frm.to(dtype)
        a = pw.warp_fused(f16, drift=d, out_size=(H, W), padding_mode=pad, align_corners=align, **kw)
        assert a.dtype == dtype
        assert torch.equal(a, pw.warp_fused(f16, drift=d.float(), out_size=(H, W), padding_mode=pad, align_corners=align, **kw))


@pytest.mark.parametrize("dtype", DTYPES)
def test_inference_site_with_a_16bit_lattice_is_byte_exact(pw, dtype):
    """R/main_new.py:697-721 with a half-precision netG: its composed 256^2 lattice arrives in 16 bits.  The specialised
    uint8 kernel reads it node by node (one 4-byte load) and matches torch's CUDA pipeline on the upcast lattice byte for
    byte, at 270p and 1080p."""
    for (H, W, hh, ww, seed) in ((270, 480, 64, 64, 21), (1080, 1920, 256, 256, 22)):
        rng = np.random.default_rng(seed)
        hwc = torch.from_numpy(rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)).cuda()
        lattice = dev(synth.make_map("smooth", 1, hh, ww, False, seed=seed).transpose(0, 3, 1, 2)).to(dtype)   # planar
        up = torch.nn.UpsamplingBilinear2d(size=(H, W))(lattice.float()).permute(0, 2, 3, 1)
        want = F.grid_sample(hwc.float().permute(0, 3, 1, 2), up, align_corners=False)[0].permute(1, 2, 0).cpu().numpy().astype(np.uint8)
        for d in (lattice.permute(0, 2, 3, 1), lattice.permute(0, 2, 3, 1).contiguous()):
            out = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=d, upsample="aligned", out_size=(H, W),
                                out_dtype=torch.uint8, out_channels_last=True)
            assert last_kernel() == "fwd_fused_u8"
            got = out[0].permute(1, 2, 0).contiguous().cpu().numpy()
            assert np.array_equal(got, want), (H, W, int((got != want).sum()))
            same = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=d.float(), upsample="aligned", out_size=(H, W),
                                 out_dtype=torch.uint8, out_channels_last=True)
            assert torch.equal(out, same)


def test_fused_rejects_other_drift_dtypes(pw):
    f = torch.zeros(1, 3, 8, 8, device="cuda")
    with pytest.raises(RuntimeError, match="drift"):
        pw.warp_fused(f, drift=torch.zeros(1, 4, 4, 2, device="cuda", dtype=torch.float64), upsample="aligned", out_size=(8, 8))
