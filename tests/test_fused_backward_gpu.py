"""Backward of warp_fused (pws_warp2d_backward_fused) on the GPU.

The gradient is that of the fused forward's own arithmetic (fp32 throughout, 16-bit and uint8 inputs upcast exactly):
  - without upsample, d loss / d lattice is the plain backward's grad_grid of the composed map, bit for bit;
  - with upsample it is that grad_grid through upsample_bilinear2d's adjoint;
  - against autograd of the unfused torch sequence (affine_grid / meshgrid, interpolate, grid_sample, the scales) in fp64
    on the CPU every gradient is within 1e-4 x max|ref|, BASELINE's gradient tolerance."""
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()
    return pw


def rel_err(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / max(float(ref.abs().max()), 1e-30))


def make_inputs(n, C, H, W, h, w, base, seed, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    frame = torch.rand(n, C, H, W, generator=g) * 2 - 1                      # the reference's [-1, 1] frames
    if base == "none":   # drift is the whole map: a smooth warp of the identity plus noise, slightly past the borders
        ys, xs = torch.meshgrid(torch.linspace(-1.05, 1.05, h), torch.linspace(-1.05, 1.05, w), indexing="ij")
        drift = torch.stack((xs, ys), -1)[None].repeat(n, 1, 1, 1) + torch.randn(n, h, w, 2, generator=g) * 0.03
    else:
        drift = torch.tanh(torch.randn(n, h, w, 2, generator=g)) * 0.05
    theta = torch.tensor([[1.02, 0.03, 0.01], [-0.04, 0.97, -0.02]])[None].repeat(n, 1, 1) + \
        torch.randn(n, 2, 3, generator=g) * 0.02
    return frame.to(device), drift.to(device), theta.to(device)


def lattice_chain(drift, theta, base, base_align, upsample, out_size):
    """drift + base, upsampled: R/lib/networks_cascading.py:164,235, R/lib/utils.py:386-403, R/main_new.py:706-710."""
    n, h, w = drift.size(0), drift.size(1), drift.size(2)
    lat = drift
    if base == "identity":
        xs = torch.arange(w, dtype=drift.dtype, device=drift.device) * 2 / (w - 1) - 1
        ys = torch.arange(h, dtype=drift.dtype, device=drift.device) * 2 / (h - 1) - 1
        lat = lat + torch.stack(torch.meshgrid(ys, xs, indexing="ij")[::-1], -1)[None]
    elif base == "affine":
        lat = lat + F.affine_grid(theta, (n, 1, h, w), align_corners=base_align)
    if upsample is not None:
        lat = F.interpolate(lat.permute(0, 3, 1, 2), size=out_size, mode="bilinear",
                            align_corners=upsample == "aligned").permute(0, 2, 3, 1)
    return lat


def pinned(m, map32):
    """m's value replaced by the fused kernel's fp32 map, m's gradient path kept.  A coordinate within rounding of an
    integer would otherwise fall into the neighbouring cell, whose gradient differs by O(1)."""
    return m + (map32.to(m) - m).detach()


def sample64(src, m, x0, y0, pad, align):
    """fp64 bilinear sample of src (N,C,H,W) at map m (N,Ho,Wo,2), grid_sample's formulas, in the cells (x0, y0) the
    kernel chose (pws_warp2d_taps) so that fp32 and fp64 rounding cannot pick different cells."""
    n, C, H, W = src.shape

    def index(c, size):
        i = ((c + 1) / 2 * (size - 1)) if align else (((c + 1) * size - 1) / 2)
        if pad == "border":
            # clip where the kernel's fp32 index clips (ATen's backward: no gradient at or past the border); the fp32
            # index is reproduced exactly: t = c + 1 in fp32, fma(t, size, -1) is exact in fp64 and rounds once to fp32
            t = (c.detach().float() + 1)
            i32 = (t * 0.5) * (size - 1) if align else (t.double() * size - 1).float() * 0.5
            i = torch.where(i32 <= 0, torch.zeros_like(i), torch.where(i32 >= size - 1, torch.full_like(i, size - 1), i))
        return i
    ix, iy = index(m[..., 0], W), index(m[..., 1], H)
    x0, y0 = x0.long(), y0.long()
    fx, fy = ix - x0, iy - y0
    flat = src.reshape(n, C, H * W)
    out = 0
    for dx, dy, wt in ((0, 0, (1 - fx) * (1 - fy)), (1, 0, fx * (1 - fy)), (0, 1, (1 - fx) * fy), (1, 1, fx * fy)):
        xx, yy = x0 + dx, y0 + dy
        ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H)
        idx = (yy.clamp(0, H - 1) * W + xx.clamp(0, W - 1)).reshape(n, 1, -1).expand(n, C, -1)
        v = torch.gather(flat, 2, idx).reshape(n, C, *x0.shape[1:])
        out = out + v * (wt * ok)[:, None]
    return out


def unfused(frame, drift, theta, base, base_align, upsample, out_size, pad, align, pre, post, map32=None):
    """The reference's sequence of torch calls (R/lib/networks_cascading.py:164,235, R/lib/utils.py:386-403,
    R/main_new.py:106-107,706-710); with map32, sampling at the fused kernel's map (pinned)."""
    lat = lattice_chain(drift, theta, base, base_align, upsample, out_size)
    if map32 is not None:
        lat = pinned(lat, map32)
    out = F.grid_sample((frame + pre[0]) * pre[1], lat, "bilinear", pad, align)
    return out / post[0] + post[1]


def fused_grads(pw, frame, drift, theta, gout, want=(True, True, True), **kw):
    f = frame.detach().clone().requires_grad_(want[0] and frame.is_floating_point())
    d = drift.detach().clone().requires_grad_(want[1])
    t = theta.detach().clone().requires_grad_(want[2]) if theta is not None else None
    out = pw.warp_fused(f, drift=d, theta=t, **kw)
    out.backward(gout)
    return out, f.grad, d.grad, (t.grad if t is not None else None)


def ref_grads(pw, frame, drift, theta, gout, dtype, device, base, base_align, upsample, out_size, pad, align, pre, post):
    """Autograd of the unfused sequence, sampling at the fused kernel's map: in fp64 on the CPU (frame, drift, theta
    upcast), or in fp32 with torch's CUDA kernels (F.grid_sample included)."""
    n = frame.size(0)
    map32 = pw.compose_map(n, out_size, drift=drift, base=base, theta=theta if base == "affine" else None,
                           base_align_corners=base_align, upsample=upsample)
    f = frame.detach().to(device, dtype).requires_grad_(True)
    d = drift.detach().to(device, dtype).requires_grad_(True)
    t = theta.detach().to(device, dtype).requires_grad_(True)
    m = pinned(lattice_chain(d, t, base, base_align, upsample, out_size), map32)
    src = (f + pre[0]) * pre[1]
    if dtype == torch.float64:
        x0, y0, _, _ = pw.warp_taps(map32, frame.size(2), frame.size(3), pad, align, want_weights=False)
        out = sample64(src, m, x0.to(device), y0.to(device), pad, align)
    else:
        out = F.grid_sample(src, m, "bilinear", pad, align)
    out = out / post[0] + post[1]
    out.backward(gout.detach().to(device, dtype))
    return out, f.grad, d.grad, t.grad


# ---- 1. bit-exact anchor -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("C", [1, 3, 5])
def test_no_upsample_glattice_is_the_plain_grad_grid_bit_for_bit(pw, planar, pad, align, C):
    n, H, W, h, w = 2, 29, 43, 31, 37
    frame, drift, _ = make_inputs(n, C, H, W, h, w, "none", seed=C + 10 * planar)
    gout = torch.randn(n, C, h, w, device="cuda")
    src = drift.permute(0, 3, 1, 2).contiguous() if planar else drift.clone()
    src.requires_grad_(True)
    d = src.permute(0, 2, 3, 1) if planar else src
    f = frame.clone().requires_grad_(True)
    out = pw.warp_fused(f, drift=d, padding_mode=pad, align_corners=align)
    out.backward(gout)
    gin, ggrid = pw.warp2d_backward(gout, frame, drift, 1 if pad == "border" else 0, align)
    glat = src.grad.permute(0, 2, 3, 1) if planar else src.grad
    assert torch.equal(glat, ggrid)
    assert rel_err(f.grad, gin) <= 1e-4


# ---- 2. against autograd of the unfused sequence ------------------------------------------------------------------
MATRIX = [(b, u) for b in ("none", "identity", "affine") for u in (None, "aligned", "half_pixel")]


@pytest.mark.parametrize("base,upsample", MATRIX)
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("scales", [False, True])
@pytest.mark.parametrize("C", [1, 3])
def test_against_unfused_autograd(pw, base, upsample, pad, align, scales, C):
    n, H, W, Ho, Wo = 2, 41, 47, 37, 53
    h, w = (Ho, Wo) if upsample is None else (9, 13)
    frame, drift, theta = make_inputs(n, C, H, W, h, w, base, seed=zlib.crc32(repr((base, upsample, pad, align, scales, C)).encode()) % 1000)
    gout = torch.randn(n, C, Ho, Wo, device="cuda")
    pre, post = ((1.0, 127.5), (127.5, -1.0)) if scales else ((0.0, 1.0), (1.0, 0.0))
    kw = dict(base=base, base_align=align, upsample=upsample, out_size=(Ho, Wo), pad=pad, align=align, pre=pre, post=post)
    th = theta if base == "affine" else None
    _, gf, gd, gt = fused_grads(pw, frame, drift, th, gout, base=base, base_align_corners=align, upsample=upsample,
                                out_size=(Ho, Wo), padding_mode=pad, align_corners=align, pre=pre, post=post)
    for dtype, device in ((torch.float64, "cpu"), (torch.float32, "cuda")):
        _, rf, rd, rt = ref_grads(pw, frame, drift, theta, gout, dtype, device, **kw)
        assert rel_err(gf, rf) <= 1e-4, (dtype, "frame", rel_err(gf, rf))
        assert rel_err(gd, rd) <= 1e-4, (dtype, "drift", rel_err(gd, rd))
        if base == "affine":
            assert rel_err(gt, rt) <= 1e-4, (dtype, "theta", rel_err(gt, rt))
        else:
            assert gt is None


@pytest.mark.parametrize("upsample", ["aligned", "half_pixel"])
@pytest.mark.parametrize("base", ["none", "affine"])
def test_lattice_finer_than_the_output(pw, upsample, base):
    # a downsample: every output pixel has its own lattice nodes (runs of one lane in the reduction)
    n, C, H, W, Ho, Wo, h, w = 2, 3, 40, 52, 23, 29, 41, 61
    frame, drift, theta = make_inputs(n, C, H, W, h, w, base, seed=77)
    gout = torch.randn(n, C, Ho, Wo, device="cuda")
    th = theta if base == "affine" else None
    _, gf, gd, gt = fused_grads(pw, frame, drift, th, gout, base=base, upsample=upsample, out_size=(Ho, Wo))
    _, rf, rd, rt = ref_grads(pw, frame, drift, theta, gout, torch.float64, "cpu", base=base, base_align=False,
                              upsample=upsample, out_size=(Ho, Wo), pad="zeros", align=False, pre=(0.0, 1.0), post=(1.0, 0.0))
    assert rel_err(gf, rf) <= 1e-4 and rel_err(gd, rd) <= 1e-4
    if base == "affine":
        assert rel_err(gt, rt) <= 1e-4


# ---- 3. the upsample's adjoint in isolation -------------------------------------------------------------------------
@pytest.mark.parametrize("upsample", ["aligned", "half_pixel"])
@pytest.mark.parametrize("size", [((9, 13), (37, 53)), ((64, 64), (270, 480)), ((41, 61), (23, 29))])
def test_upsample_adjoint_matches_torch(pw, upsample, size):
    (h, w), (Ho, Wo) = size
    n, C, H, W = 2, 3, 60, 90
    frame, drift, _ = make_inputs(n, C, H, W, h, w, "none", seed=h)
    gout = torch.randn(n, C, Ho, Wo, device="cuda")
    _, _, gd, _ = fused_grads(pw, frame, drift, None, gout, want=(False, True, False), upsample=upsample, out_size=(Ho, Wo))
    m = pw.compose_map(n, (Ho, Wo), drift=drift, upsample=upsample)
    _, ggrid = pw.warp2d_backward(gout, frame, m, 0, False, (False, True))
    lat = drift.clone().requires_grad_(True)
    up = F.interpolate(lat.permute(0, 3, 1, 2), size=(Ho, Wo), mode="bilinear", align_corners=upsample == "aligned")
    up.permute(0, 2, 3, 1).backward(ggrid)
    assert rel_err(gd, lat.grad) <= 1e-5


# ---- 4. dtypes ------------------------------------------------------------------------------------------------------
def eps(dt):
    return float(torch.finfo(dt).eps)


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("upsample", [None, "aligned"])
def test_16bit_frames_match_the_upcast_call(pw, dt, upsample):
    n, C, H, W, Ho, Wo = 2, 3, 50, 70, 45, 61
    h, w = (Ho, Wo) if upsample is None else (12, 17)
    frame, drift, theta = make_inputs(n, C, H, W, h, w, "affine", seed=5)
    frame16 = frame.to(dt)
    gout16 = torch.randn(n, C, Ho, Wo, device="cuda").to(dt)
    kw = dict(base="affine", upsample=upsample, out_size=(Ho, Wo), pre=(1.0, 127.5), post=(127.5, -1.0))
    _, gf, gd, gt = fused_grads(pw, frame16, drift, theta, gout16, **kw)
    _, rf, rd, rt = fused_grads(pw, frame16.float(), drift, theta, gout16.float(), **kw)
    assert gf.dtype == dt and gd.dtype == torch.float32
    assert float((gf.float() - rf.to(dt).float()).abs().max()) <= eps(dt) * float(rf.abs().max())
    assert rel_err(gd, rd) <= 1e-6 and rel_err(gt, rt) <= 1e-6


@pytest.mark.parametrize("upsample", [None, "aligned"])
def test_uint8_frame_with_float_output(pw, upsample):
    n, C, H, W, Ho, Wo = 2, 3, 50, 70, 45, 61
    h, w = (Ho, Wo) if upsample is None else (12, 17)
    _, drift, theta = make_inputs(n, C, H, W, h, w, "affine", seed=6)
    hwc = torch.randint(0, 256, (n, H, W, C), dtype=torch.uint8, device="cuda")
    frame = hwc.permute(0, 3, 1, 2)                                          # cv2 HWC buffer
    gout = torch.randn(n, C, Ho, Wo, device="cuda")
    kw = dict(base="affine", upsample=upsample, out_size=(Ho, Wo), post=(127.5, -1.0))
    out, gf, gd, gt = fused_grads(pw, frame, drift, theta, gout, **kw)
    assert out.dtype == torch.float32 and gf is None
    _, _, rd, rt = fused_grads(pw, frame.float(), drift, theta, gout, want=(False, True, True), **kw)
    if upsample is None:
        assert torch.equal(gd, rd) and torch.equal(gt, rt)
    assert rel_err(gd, rd) <= 1e-6 and rel_err(gt, rt) <= 1e-6
    # a uint8 output is not differentiable: the forward kernel alone, no grad_fn
    d = drift.clone().requires_grad_(True)
    o8 = pw.warp_fused(frame, drift=d, base="affine", theta=theta, upsample=upsample, out_size=(Ho, Wo), out_dtype=torch.uint8)
    assert o8.grad_fn is None


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("upsample", [None, "half_pixel"])
def test_16bit_lattice_matches_the_upcast_call(pw, dt, upsample):
    n, C, H, W, Ho, Wo = 2, 3, 50, 70, 45, 61
    h, w = (Ho, Wo) if upsample is None else (12, 17)
    frame, drift, theta = make_inputs(n, C, H, W, h, w, "identity", seed=7)
    drift16 = drift.to(dt)
    gout = torch.randn(n, C, Ho, Wo, device="cuda")
    kw = dict(base="identity", upsample=upsample, out_size=(Ho, Wo))
    _, gf, gd, _ = fused_grads(pw, frame, drift16, None, gout, **kw)
    _, rf, rd, _ = fused_grads(pw, frame, drift16.float(), None, gout, **kw)
    assert gd.dtype == dt and gd.shape == drift16.shape
    assert float((gd.float() - rd.to(dt).float()).abs().max()) <= eps(dt) * float(rd.abs().max())
    assert rel_err(gf, rf) <= 1e-6


# ---- 5. forward unchanged -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["small_identity", "1080p_affine_aligned"])
def test_grad_call_forward_equals_the_no_grad_call(pw, case):
    if case == "small_identity":
        n, C, H, W, Ho, Wo, h, w, base, up = 2, 3, 40, 56, 40, 56, 40, 56, "identity", None
    else:
        n, C, H, W, Ho, Wo, h, w, base, up = 2, 3, 1080, 1920, 1080, 1920, 256, 256, "affine", "aligned"
    frame, drift, theta = make_inputs(n, C, H, W, h, w, base, seed=8)
    planar = drift.permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    kw = dict(base=base, theta=theta if base == "affine" else None, upsample=up, out_size=(Ho, Wo),
              pre=(1.0, 127.5), post=(127.5, -1.0))
    out = pw.warp_fused(frame, drift=planar.permute(0, 2, 3, 1), **kw)
    assert out.grad_fn is not None
    with torch.no_grad():
        ref = pw.warp_fused(frame, drift=planar.permute(0, 2, 3, 1), **kw)
    assert torch.equal(out, ref)
    nograd = pw.warp_fused(frame, drift=planar.detach().permute(0, 2, 3, 1), **kw)
    assert nograd.grad_fn is None and torch.equal(out, nograd)


# ---- 6. 1080p geometry ----------------------------------------------------------------------------------------------
def test_1080p_sums(pw):
    n, C, H, W, h, w = 2, 3, 1080, 1920, 256, 256
    frame, drift, _ = make_inputs(n, C, H, W, h, w, "none", seed=9)
    gout = torch.randn(n, C, H, W, device="cuda")
    pre, post = (1.0, 127.5), (127.5, -1.0)
    _, gf, gd, _ = fused_grads(pw, frame, drift, None, gout, upsample="aligned", out_size=(H, W), pre=pre, post=post)
    m = pw.compose_map(n, (H, W), drift=drift, upsample="aligned")
    go = (gout / post[0]).contiguous()
    _, ggrid = pw.warp2d_backward(go, (frame + pre[0]) * pre[1], m, 0, False, (False, True))
    # the upsample weights of a pixel sum to 1: the adjoint preserves the total
    s_ref = ggrid.double().sum((0, 1, 2))
    assert float((gd.double().sum((0, 1, 2)) - s_ref).abs().max()) <= 1e-4 * float(ggrid.double().abs().sum())
    # sum of grad_input: every output pixel hands go * pre_mul times its valid tap weights to the frame
    valid = pw.grid_sample(torch.ones(n, 1, H, W, device="cuda"), m, "bilinear", "zeros", False)
    s_gin = float((go.double().sum(1, keepdim=True) * valid.double()).sum() * pre[1])
    assert abs(float(gf.double().sum()) - s_gin) <= 1e-4 * float((go.double().abs().sum(1, keepdim=True) * valid.double()).sum() * pre[1])


# ---- 7. training steps ----------------------------------------------------------------------------------------------
class MapNet(torch.nn.Module):
    """A small netG stand-in: a planar drift lattice and an affine theta from the frame."""

    def __init__(self, lattice):
        super().__init__()
        self.lattice = lattice
        self.conv = torch.nn.Conv2d(3, 2, 3, padding=1)
        self.fc = torch.nn.Linear(3, 6)
        torch.nn.init.normal_(self.fc.weight, std=0.02)
        torch.nn.init.zeros_(self.fc.bias)

    def forward(self, x):
        small = F.adaptive_avg_pool2d(x, self.lattice)
        drift = torch.tanh(self.conv(small)) * 0.05                              # (N, 2, h, w), planar as netG stores it
        eye = torch.tensor([1.0, 0, 0, 0, 1.0, 0], device=x.device)
        theta = (eye + self.fc(small.mean((2, 3)))).view(-1, 2, 3)
        return drift.permute(0, 2, 3, 1), theta


def test_training_steps_match_the_unfused_sequence(pw):
    torch.manual_seed(0)
    n, C, H, W = 2, 3, 135, 240
    net = MapNet((32, 32)).cuda()
    opt = torch.optim.SGD(net.parameters(), lr=0.05)
    x = torch.rand(n, C, H, W, device="cuda") * 2 - 1
    target = torch.roll(x, shifts=(2, 3), dims=(2, 3))
    for _ in range(3):
        grads = []
        for fused in (True, False):
            net.zero_grad()
            drift, theta = net(x)
            if fused:
                out = pw.warp_fused(x, drift=drift, base="affine", theta=theta, upsample="aligned", out_size=(H, W))
            else:
                map32 = pw.compose_map(n, (H, W), drift.detach(), "affine", theta.detach(), False, "aligned")
                out = unfused(x, drift, theta, "affine", False, "aligned", (H, W), "zeros", False, (0.0, 1.0), (1.0, 0.0),
                              map32)
            F.mse_loss(out, target).backward()
            grads.append([p.grad.clone() for p in net.parameters()])
        for a, b in zip(*grads):
            assert rel_err(a, b) <= 1e-4
        for p, g in zip(net.parameters(), grads[0]):
            p.grad = g
        opt.step()


def test_chained_affine_warp_reaches_the_frame(pw):
    # R/main_new.py:194-197: grid_sample(x, affine_grid(H)) written as warp_fused(x, base="affine", theta=H)
    n, C, H, W = 2, 3, 64, 96
    frame, _, theta = make_inputs(n, C, H, W, 4, 4, "affine", seed=12)
    gout = torch.randn(n, C, H, W, device="cuda")
    x, th = frame.clone().requires_grad_(True), theta.clone().requires_grad_(True)
    pw.warp_fused(x, base="affine", theta=th, map_size=(H, W)).backward(gout)
    xr, thr = frame.clone().requires_grad_(True), theta.clone().requires_grad_(True)
    map32 = pw.compose_map(n, (H, W), base="affine", theta=theta, map_size=(H, W))
    grid = pinned(F.affine_grid(thr, (n, C, H, W), align_corners=False), map32)
    F.grid_sample(xr, grid, align_corners=False).backward(gout)
    assert rel_err(x.grad, xr.grad) <= 1e-4 and rel_err(th.grad, thr.grad) <= 1e-4
