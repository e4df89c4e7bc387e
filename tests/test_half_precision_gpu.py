"""GPU parity of the 16-bit backward: f16 / bf16 frames with maps of the same 16-bit type (the lean kernels with 16-bit map
loads, and the marching kernel `bwd_march_16` for every other layout), and 16-bit frames with fp32 maps in the layouts the
lean and TMA kernels cannot take (C not in {1, 3}, channels-last frames, channel slices, cropped windows).

Semantics of every 16-bit kernel of this library: taps and map upcast to fp32, ATen's fp32 operation order, one rounding.
  * forward   == aten.grid_sampler_2d(f.float(), g.float()).to(f.dtype)                    (torch.equal)
  * grad_grid == this library's fp32 backward on the upcast inputs, rounded to g.dtype      (torch.equal)
  * grad_input is summed in an fp32 buffer (<= 1e-4 x max against ATen's fp32 kernel on the upcast inputs: atomic order)
    and rounded to the frame type once (within one ulp of the dtype x max)."""
import pytest
import torch

import synth

pytestmark = pytest.mark.gpu
PAD = {"zeros": 0, "border": 1}
DTYPES = [torch.float16, torch.bfloat16]


@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()
    prev = _lib.small_problem_elems(-1)
    yield pw
    _lib.small_problem_elems(prev)


def last_kernel():
    from pwstablenet_b200 import _lib
    return _lib.last_kernel()


def small_problem_elems(n):
    from pwstablenet_b200 import _lib
    return _lib.small_problem_elems(n)


def layout(g, how):
    """g: contiguous (N,Ho,Wo,2).  planar: netG's storage (coordinate stride Ho*Wo); strided: every other pixel of a
    twice-as-wide interleaved map that starts one element into its buffer (not dense, pairs not aligned to their size)."""
    if how == "planar":
        return g.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
    if how == "strided":
        N, Ho, Wo, _ = g.shape
        wide = torch.zeros(N * Ho * 2 * Wo * 2 + 1, dtype=g.dtype, device=g.device)[1:].view(N, Ho, 2 * Wo, 2)
        wide[:, :, ::2] = g
        return wide[:, :, ::2]
    return g


def make(kind, N, C, H, W, Ho, Wo, align, how, dtype, map_dtype, seed=11):
    g = torch.from_numpy(synth.make_map(kind, N, Ho, Wo, align, seed=seed)).cuda().to(map_dtype)
    f = torch.from_numpy(synth.make_frames(N, C, H, W, seed=seed + 1)).cuda().to(dtype)
    go = torch.from_numpy(synth.make_gout(N, C, Ho, Wo, seed=seed + 2)).cuda().to(dtype)
    return f, layout(g, how), go


def rel(a, b):
    return float((a.float() - b.float()).abs().max()) / max(float(b.float().abs().max()), 1e-30)


def check_call(pw, f, g, go, pad, align, mask=(True, True)):
    """One forward and one backward of `pw` against the upcast oracles; returns the kernel family of the backward."""
    out = pw.warp2d_forward(f, g, PAD[pad], align)
    assert out.dtype == f.dtype
    assert torch.equal(out, torch.ops.aten.grid_sampler_2d(f.float(), g.float(), 0, PAD[pad], align).to(f.dtype))
    gin, gg = pw.warp2d_backward(go, f, g, PAD[pad], align, mask)
    kernel = last_kernel()
    rin, rg = pw.warp2d_backward(go.float(), f.float(), g.float(), PAD[pad], align, (True, True))
    ain, _ = torch.ops.aten.grid_sampler_2d_backward(go.float(), f.float(), g.float(), 0, PAD[pad], align, (True, False))
    if mask[1]:
        assert gg.dtype == g.dtype and gg.shape == g.shape
        if g.is_contiguous() or g.permute(0, 3, 1, 2).is_contiguous():
            assert gg.stride() == g.stride()      # returned in the map's own layout
        assert torch.equal(gg, rg.to(g.dtype))
    else:
        assert gg is None
    if mask[0]:
        assert gin.dtype == f.dtype
        assert rel(gin, ain) <= torch.finfo(f.dtype).eps
        # the fp32 accumulation buffer itself, arriving filled with garbage
        acc = torch.full(f.shape, 7.0, dtype=torch.float32, device="cuda")
        pw.warp2d_backward(go, f, g, PAD[pad], align, (True, False), grad_input=acc)
        assert rel(acc, ain) <= 1e-4
    else:
        assert gin is None
    return kernel


# (N, C, H, W, Ho, Wo): C in {1..5}, partial tiles in both directions, output size != frame size
SHAPES = [
    (2, 1, 40, 72, 40, 72),
    (2, 2, 33, 40, 29, 47),
    (2, 3, 37, 53, 30, 61),
    (1, 4, 64, 64, 70, 66),
    (2, 5, 24, 96, 24, 96),
]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_same_dtype_maps(pw, dtype, pad):
    for shape in SHAPES:
        N, C, H, W, Ho, Wo = shape
        for kind in ("smooth", "noisy", "random", "centre"):
            for align in (False, True):
                for how in ("planar", "interleaved", "strided"):
                    f, g, go = make(kind, N, C, H, W, Ho, Wo, align, how, dtype, dtype, seed=13 + C)
                    kernel = check_call(pw, f, g, go, pad, align)
                    lean = C in (1, 3) and how != "strided"
                    assert kernel == ("bwd_lean_16" if lean else "bwd_march_16"), (shape, how, kernel)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mask", [(True, False), (False, True)])
def test_same_dtype_maps_output_masks(pw, dtype, mask):
    for shape in (SHAPES[2], SHAPES[4]):
        N, C, H, W, Ho, Wo = shape
        for how in ("planar", "interleaved", "strided"):
            f, g, go = make("noisy", N, C, H, W, Ho, Wo, False, how, dtype, dtype, seed=17)
            check_call(pw, f, g, go, "zeros", False, mask)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_training_shape_same_dtype_maps(pw, dtype, pad):
    # the reference's training shape (16 x 3 x 256 x 256) with netG run in half precision: one-wave lean kernels
    for align in (False, True):
        for how in ("planar", "interleaved"):
            f, g, go = make("smooth", 16, 3, 256, 256, 256, 256, align, how, dtype, dtype, seed=23)
            pw.warp2d_forward(f, g, PAD[pad], align)
            assert last_kernel() == "fwd_lean"
            assert check_call(pw, f, g, go, pad, align) == "bwd_lean_16"
            _, gg = pw.warp2d_backward(go, f, g, PAD[pad], align, (False, True))
            assert last_kernel() == "bwd_lean_16"


def odd_layouts(dtype, N, H, W, seed):
    """16-bit frames the lean and TMA backward kernels do not take, each with its fp32 map and grad_output."""
    g = torch.from_numpy(synth.make_map("smooth", N, H, W, False, seed=seed)).cuda()
    cases = {}
    for C in (2, 4, 5):
        cases[f"C={C}"] = torch.from_numpy(synth.make_frames(N, C, H, W, seed=seed + C)).cuda().to(dtype)
    rgb = torch.from_numpy(synth.make_frames(N, 3, H, W, seed=seed + 7)).cuda().to(dtype)
    cases["channels-last"] = rgb.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    wide = torch.from_numpy(synth.make_frames(N, 37, H, W, seed=seed + 8)).cuda().to(dtype)
    cases["channel slice of 37"] = wide[:, 3:8]
    big = torch.from_numpy(synth.make_frames(N, 3, H + 9, W + 24, seed=seed + 9)).cuda().to(dtype)
    cases["crop"] = big[:, :, 5:5 + H, 7:7 + W]
    out = []
    for name, f in cases.items():
        go = torch.from_numpy(synth.make_gout(N, f.shape[1], H, W, seed=seed + 10)).cuda().to(dtype)
        out.append((name, f, g, go))
    return out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_16bit_frames_fp32_maps_any_layout(pw, dtype, pad):
    # refused with NotImplementedError before: now the marching kernel, fp32 grad_grid equal to the fp32 path on the upcast
    # inputs, fp32-accumulated grad_input; below and above the small-problem threshold
    for threshold in (-1, 0):
        prev = small_problem_elems(threshold)
        try:
            for name, f, g, go in odd_layouts(dtype, 2, 72, 136, seed=31):
                for align in (False, True):
                    kernel = check_call(pw, f, g, go, pad, align)
                    # at threshold 0 the persistent TMA kernel is tried first and may take an RGB layout it can describe
                    assert kernel == "bwd_march_16" or (threshold == 0 and f.shape[1] == 3 and kernel == "bwd_tma_16"), (name, kernel)
                    _, gg = pw.warp2d_backward(go, f, g, PAD[pad], align, (False, True))
                    assert gg.dtype == torch.float32
        finally:
            small_problem_elems(prev)


@pytest.mark.parametrize("dtype", DTYPES)
def test_16bit_frames_fp32_maps_any_layout_large(pw, dtype):
    # above the default small-problem threshold (2 x 5 x 720 x 640 output elements > 4 Mi)
    for name, f, g, go in odd_layouts(dtype, 2, 720, 640, seed=37):
        kernel = check_call(pw, f, g, go, "zeros", False)
        assert kernel == "bwd_march_16" or (f.shape[1] == 3 and kernel == "bwd_tma_16"), (name, kernel)


@pytest.mark.parametrize("dtype", DTYPES)
def test_config5_keeps_the_tma_backward(pw, dtype):
    # bf16 / f16 RGB frames with an fp32 map above the threshold: unchanged, the persistent TMA kernel
    f, g, go = make("smooth", 2, 3, 720, 1280, 720, 1280, False, "planar", dtype, torch.float32, seed=41)
    assert check_call(pw, f, g, go, "zeros", False) == "bwd_tma_16"


@pytest.mark.parametrize("dtype", DTYPES)
def test_grid_sample_autograd(pw, dtype):
    for C, how in ((3, "planar"), (5, "interleaved"), (1, "strided")):
        f, g, go = make("noisy", 2, C, 48, 80, 48, 80, True, how, dtype, dtype, seed=43)
        fa, ga = f.clone().requires_grad_(True), g.clone().requires_grad_(True)
        out = pw.grid_sample(fa, ga, "bilinear", "border", True)
        assert torch.equal(out, pw.warp2d_forward(f, g, 1, True))
        out.backward(go)
        gin, gg = pw.warp2d_backward(go, f, g, 1, True, (True, True))
        assert fa.grad.dtype == dtype and ga.grad.dtype == dtype
        assert torch.equal(ga.grad, gg)
        assert rel(fa.grad, gin) <= torch.finfo(dtype).eps


class _MapNet(torch.nn.Module):
    """A small conv net that predicts a per-pixel map from a frame, as netG does."""

    def __init__(self, C):
        super().__init__()
        self.c1 = torch.nn.Conv2d(C, 8, 3, padding=1)
        self.c2 = torch.nn.Conv2d(8, 2, 3, padding=1)

    def forward(self, x):
        N, _, H, W = x.shape
        theta = torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], device=x.device).expand(N, 2, 3)
        base = torch.nn.functional.affine_grid(theta, (N, 1, H, W), align_corners=False).to(x.dtype)
        drift = 0.05 * torch.tanh(self.c2(torch.relu(self.c1(x))))
        return base + drift.permute(0, 2, 3, 1)


def _net_step(net, x, target, upcast=False):
    import torch.nn.functional as F
    g = net(x)
    if upcast:   # the warp in fp32 on the upcast inputs, its result rounded once: this library's 16-bit semantics
        y = F.grid_sample(x.float(), g.float(), mode="bilinear", padding_mode="zeros", align_corners=False).to(x.dtype)
    else:
        y = F.grid_sample(x, g, mode="bilinear", padding_mode="zeros", align_corners=False)
    loss = (y.float() - target).abs().mean()
    net.zero_grad()
    loss.backward()
    return [p.grad.detach().clone() for p in net.parameters()]


@pytest.mark.parametrize("dtype", DTYPES)
def test_install_half_precision_net(pw, dtype):
    # a user who runs the map network in half precision with pw.install(): parameter gradients of the input dtype, equal
    # (within 2 ulps of the dtype x the largest gradient; measured: identical) to stock torch running the warp in fp32 on
    # the upcast inputs.  Stock torch's native 16-bit warp is far from both (measured 1.4x / 2.6x the largest gradient for
    # f16 / bf16): its 16-bit grad_grid is not the fp32 result rounded (test_aten_native_16bit_against_upcast_oracle).
    torch.manual_seed(5)
    net = _MapNet(3).cuda().to(dtype)
    x = torch.from_numpy(synth.make_frames(4, 3, 64, 96, seed=47)).cuda().to(dtype)
    target = torch.from_numpy(synth.make_frames(4, 3, 64, 96, seed=48)).cuda()
    ref = _net_step(net, x, target, upcast=True)
    native = _net_step(net, x, target)
    pw.install()
    try:
        got = _net_step(net, x, target)
    finally:
        pw.uninstall()
    scale = max(float(r.float().abs().max()) for r in ref)
    err = max(float((a.float() - b.float()).abs().max()) for a, b in zip(got, ref))
    far = max(float((a.float() - b.float()).abs().max()) for a, b in zip(got, native))
    print(f"measured {dtype}: parameter gradients, |ours - torch with the warp upcast| = {err / scale:.3g}, "
          f"|ours - torch native 16-bit| = {far / scale:.3g} x the largest gradient")
    for a in got:
        assert a.dtype == dtype
    assert err <= 2 * torch.finfo(dtype).eps * scale


@pytest.mark.parametrize("dtype", DTYPES)
def test_aten_override_half_precision(pw, dtype):
    f, g, go = make("noisy", 2, 3, 40, 64, 40, 64, False, "interleaved", dtype, dtype, seed=53)
    pw.install(aten_override=True)
    try:
        fa, ga = f.clone().requires_grad_(True), g.clone().requires_grad_(True)
        out = torch.grid_sampler(fa, ga, 0, 1, False)
        out.backward(go)
    finally:
        pw.uninstall()
    assert torch.equal(out, pw.warp2d_forward(f, g, 1, False))
    gin, gg = pw.warp2d_backward(go, f, g, 1, False, (True, True))
    assert fa.grad.dtype == dtype and ga.grad.dtype == dtype
    assert torch.equal(ga.grad, gg)
    assert rel(fa.grad, gin) <= torch.finfo(dtype).eps


@pytest.mark.parametrize("dtype", DTYPES)
def test_aten_native_16bit_against_upcast_oracle(pw, dtype):
    # ATen's own 16-bit kernels, measured (DESIGN §3.8): the forward IS the upcast-sample-round oracle, grad_grid is NOT the
    # fp32 result rounded once (it differs in ~90 % of the elements, by up to 1.2-1.7x the largest value); this library
    # returns the oracle for both
    for kind in ("smooth", "noisy"):
        for align in (False, True):
            f, g, go = make(kind, 2, 3, 128, 192, 128, 192, align, "interleaved", dtype, dtype, seed=59)
            native = torch.ops.aten.grid_sampler_2d(f, g, 0, 0, align)
            oracle = torch.ops.aten.grid_sampler_2d(f.float(), g.float(), 0, 0, align).to(dtype)
            _, ngg = torch.ops.aten.grid_sampler_2d_backward(go, f, g, 0, 0, align, (True, True))
            _, rg = pw.warp2d_backward(go.float(), f.float(), g.float(), 0, align, (True, True))
            print(f"measured {dtype} {kind} align={align}: native grad_grid differs in "
                  f"{float((ngg != rg.to(dtype)).float().mean()):.1%} of the elements, max {rel(ngg, rg):.3g} x max")
            assert torch.equal(native, oracle)
            assert not torch.equal(ngg, rg.to(dtype))
            assert torch.equal(pw.warp2d_forward(f, g, 0, align), oracle)
            _, gg = pw.warp2d_backward(go, f, g, 0, align, (False, True))
            assert torch.equal(gg, rg.to(dtype))
