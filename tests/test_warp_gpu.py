"""GPU parity of the CUDA warp (through the C ABI) against the CPU oracle, the
committed golden vectors and torch's own CUDA grid_sample -- the implementation the
reference's call sites (R/main_new.py:106,116,197,716) actually execute.

Tolerances (BASELINE.json): taps and masks bit-exact; forward <= 1e-5 abs fp32 on
unit-range frames (asserted here as BIT-EXACT, also on 0..255 frames); gradients
<= 1e-4 relative (atomic ordering)."""
import hashlib
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import oracle

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()  # fail loudly if the CUDA library is absent
    return pw


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


PAD = {"zeros": 0, "border": 1}
SHAPES = [(2, 3, 37, 53, 37, 53), (1, 1, 64, 200, 64, 200), (3, 3, 96, 160, 50, 70), (2, 4, 33, 65, 33, 65),
          (1, 2, 17, 300, 40, 129), (2, 5, 20, 24, 20, 24)]
KINDS = ["smooth", "random", "centre", "noisy"]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_forward_bit_exact_vs_oracle_and_torch(pw, shape, pad, align, kind):
    N, C, H, W, Ho, Wo = shape
    frames = synth.make_frames(N, C, H, W, seed=1)
    grid = synth.make_map(kind, N, Ho, Wo, align, seed=2)
    ref = oracle.forward(frames, grid, pad, align)
    got = pw.grid_sample(dev(frames), dev(grid), "bilinear", pad, align)
    # ATen's own CUDA kernel (F.grid_sample detours to cuDNN for zeros + align_corners=True)
    torch_out = torch.ops.aten.grid_sampler_2d(dev(frames), dev(grid), 0, PAD[pad], align)
    assert got.is_contiguous() and got.shape == torch_out.shape
    np.testing.assert_array_equal(got.cpu().numpy(), ref)
    assert torch.equal(got, torch_out)
    # whatever F.grid_sample dispatches to (cuDNN included): BASELINE's 1e-5 abs on unit-range frames
    f_out = F.grid_sample(dev(frames), dev(grid), mode="bilinear", padding_mode=pad, align_corners=align)
    assert float((got - f_out).abs().max()) <= 1e-5 * 255.0


@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
def test_taps_and_masks_bit_exact(pw, pad, align):
    H, W = 45, 77
    for kind in KINDS:
        grid = synth.make_map(kind, 2, 31, 59, align, seed=5)
        x0, y0, mask, wts = oracle.taps(grid, H, W, pad, align)
        gx0, gy0, gmask, gw = pw.warp_taps(dev(grid), H, W, pad, align)
        np.testing.assert_array_equal(gx0.cpu().numpy(), x0)
        np.testing.assert_array_equal(gy0.cpu().numpy(), y0)
        np.testing.assert_array_equal(gmask.cpu().numpy(), mask)
        np.testing.assert_array_equal(gw.cpu().numpy(), wts)


def test_taps_integer_crossings_wide_frames(pw):
    # coordinates sitting on / next to integers at the widths of the BASELINE configs
    rng = np.random.default_rng(9)
    for W in (256, 1280, 1920, 3840):
        for align in (False, True):
            k = rng.integers(0, W, size=4096)
            base = (2 * k / (W - 1) - 1) if align else ((2 * k + 1) / W - 1)
            x = base.astype(np.float32)
            x = np.concatenate([x, np.nextafter(x, np.float32(2)), np.nextafter(x, np.float32(-2))])
            grid = np.zeros((1, 1, x.size, 2), np.float32)
            grid[0, 0, :, 0] = x
            ox0, oy0, om, ow = oracle.taps(grid, 4, W, "zeros", align)
            gx0, gy0, gm, gw = pw.warp_taps(dev(grid), 4, W, "zeros", align)
            np.testing.assert_array_equal(gx0.cpu().numpy(), ox0)
            np.testing.assert_array_equal(gm.cpu().numpy(), om)
            np.testing.assert_array_equal(gw.cpu().numpy(), ow)


def _rel(a, b):
    return float(np.abs(a - b).max() / max(1e-30, np.abs(b).max()))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_backward_vs_oracle_and_torch(pw, shape, pad, align, kind):
    N, C, H, W, Ho, Wo = shape
    frames = synth.make_frames(N, C, H, W, seed=3)
    grid = synth.make_map(kind, N, Ho, Wo, align, seed=4)
    gout = synth.make_gout(N, C, Ho, Wo, seed=5)
    o_gin, o_ggrid, o_gin64 = oracle.backward(gout, frames, grid, pad, align, want_f64_accum=True)

    fi = dev(frames).requires_grad_(True)
    gi = dev(grid).requires_grad_(True)
    pw.grid_sample(fi, gi, "bilinear", pad, align).backward(dev(gout))
    t_gin, t_ggrid = torch.ops.aten.grid_sampler_2d_backward(dev(gout), dev(frames), dev(grid), 0, PAD[pad], align,
                                                             [True, True])

    gin = fi.grad.cpu().numpy()
    ggrid = gi.grad.cpu().numpy()
    assert _rel(gin, o_gin64) <= 1e-4                      # vs order-free fp64 accumulation
    assert _rel(gin, t_gin.cpu().numpy()) <= 1e-4          # vs ATen CUDA (its own atomic order)
    np.testing.assert_array_equal(ggrid, o_ggrid)          # deterministic: bit-exact vs oracle
    assert _rel(ggrid, t_ggrid.cpu().numpy()) <= 1e-6      # and ATen CUDA


def test_output_mask_variants_and_grad_routing(pw):
    # R/main_new.py:106/116: map needs grad, frame does not; :197: frame needs grad, map does not
    N, C, H, W = 2, 3, 40, 72
    frames, gout = synth.make_frames(N, C, H, W), synth.make_gout(N, C, H, W)
    grid = synth.make_map("smooth", N, H, W, False)
    o_gin, o_ggrid, o_gin64 = oracle.backward(gout, frames, grid, "zeros", False, want_f64_accum=True)
    fi, gi = dev(frames), dev(grid).requires_grad_(True)
    pw.grid_sample(fi, gi, align_corners=False).backward(dev(gout))
    assert fi.grad is None
    np.testing.assert_array_equal(gi.grad.cpu().numpy(), o_ggrid)
    fi, gi = dev(frames).requires_grad_(True), dev(grid)
    pw.grid_sample(fi, gi, align_corners=False).backward(dev(gout))
    assert gi.grad is None
    assert _rel(fi.grad.cpu().numpy(), o_gin64) <= 1e-4


def test_reference_layouts_planar_map_channels_last_and_sliced_frames(pw):
    N, C, H, W = 2, 3, 48, 80
    frames, gout = synth.make_frames(N, C, H, W), synth.make_gout(N, C, H, W)
    grid = synth.make_map("smooth", N, H, W, False)
    ref = oracle.forward(frames, grid, "zeros", False)
    o_gin, o_ggrid, o_gin64 = oracle.backward(gout, frames, grid, "zeros", False, want_f64_accum=True)
    # planar-stored map: (N,2,H,W) storage viewed as (N,H,W,2), strides (2HW, W, 1, HW) -- what netG returns
    planar = dev(np.ascontiguousarray(grid.transpose(0, 3, 1, 2))).permute(0, 2, 3, 1)
    assert planar.stride() == (2 * H * W, W, 1, H * W)
    # channels-last frame view (R/main_new.py:679-684) and a channel slice of a 37-channel tensor (R/main.py:106)
    cl = dev(np.ascontiguousarray(frames.transpose(0, 2, 3, 1))).permute(0, 3, 1, 2)
    big = torch.zeros(N, 37, H, W, device="cuda")
    big[:, 31:34] = dev(frames)
    for f in (dev(frames), cl, big[:, 31:34]):
        fi = f.detach().clone(memory_format=torch.preserve_format) if f.is_contiguous() else f.detach()
        fi.requires_grad_(True)
        gi = planar.detach().requires_grad_(True)
        out = pw.grid_sample(fi, gi, align_corners=False)
        np.testing.assert_array_equal(out.detach().cpu().numpy(), ref)
        out.backward(dev(gout))
        assert gi.grad.shape == gi.shape
        np.testing.assert_array_equal(gi.grad.cpu().numpy(), o_ggrid)
        assert _rel(fi.grad.cpu().numpy(), o_gin64) <= 1e-4


def test_golden_config1_reference_netg_maps_on_gpu(pw):
    z = np.load(os.path.join(GOLD, "config1_netg.npz"))
    rng = np.random.default_rng(123)
    frame = (rng.random((1, 3, 256, 256), dtype=np.float32) * 255).astype(np.float32)
    gout = rng.random((1, 3, 256, 256), dtype=np.float32)
    assert sha(frame) == str(z["frame_sha"])
    m0, m1, m2 = synth.config1_netg_maps(z)
    cases = [("m0", m0, False), ("m1", m1, False), ("m2", m2, False)]
    gm = oracle.generate_maps(z["drift3_planar"])[0]
    cases += [("gm_f", gm, False), ("gm_t", gm, True)]
    for name, planar, align in cases:
        go = gout[:, :, ::gout.shape[2] // planar.shape[1]]       # the map's rows (every 8th: m0, m1)
        for pad in ("zeros", "border"):
            gi = dev(planar[None]).permute(0, 2, 3, 1).requires_grad_(True)
            fi = dev(frame).requires_grad_(True)
            out = pw.grid_sample(fi, gi, "bilinear", pad, align)
            key = f"{name}_{pad}"
            assert sha(out.detach().cpu().numpy()) == str(z[key + "_out_sha"]), key
            out.backward(dev(go))
            ref_gin = z[key + "_gin_sub"]
            assert np.abs(fi.grad.cpu().numpy()[:, :, ::8, ::8] - ref_gin).max() <= 1e-4 * max(1.0, np.abs(ref_gin).max()), key
            ref_gg = z[key + "_ggrid_sub"]
            assert np.abs(gi.grad.cpu().numpy()[:, ::8, ::8, :] - ref_gg).max() <= 1e-4 * np.abs(ref_gg).max(), key


def test_small_kats_on_gpu(pw):
    z = np.load(os.path.join(GOLD, "kat_small.npz"))
    for i in range(int(z["count"])):
        k = f"k{i}"
        pad = "border" if int(z[k + "_meta"][6]) else "zeros"
        align = bool(int(z[k + "_meta"][7]))
        fi = dev(z[k + "_in"]).requires_grad_(True)
        gi = dev(z[k + "_grid"]).requires_grad_(True)
        out = pw.grid_sample(fi, gi, "bilinear", pad, align)
        np.testing.assert_array_equal(out.detach().cpu().numpy(), z[k + "_out"], err_msg=k)
        out.backward(dev(z[k + "_gout"]))
        np.testing.assert_allclose(fi.grad.cpu().numpy(), z[k + "_gin"], rtol=1e-4, atol=1e-5, err_msg=k)
        s = max(1e-6, float(np.abs(z[k + "_ggrid"]).max()))
        assert np.abs(gi.grad.cpu().numpy() - z[k + "_ggrid"]).max() <= 1e-4 * s, k


def test_fp64_gradcheck(pw):
    torch.manual_seed(0)
    for pad in ("zeros", "border"):
        for align in (False, True):
            f = torch.rand(2, 3, 7, 9, dtype=torch.float64, device="cuda", requires_grad=True)
            g = (torch.rand(2, 5, 6, 2, dtype=torch.float64, device="cuda") * 2.2 - 1.1).requires_grad_(True)
            assert torch.autograd.gradcheck(lambda a, b: pw.grid_sample(a, b, "bilinear", pad, align), (f, g),
                                            eps=1e-6, atol=1e-5, nondet_tol=1e-9)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_16bit_frames_with_fp32_maps(pw, dtype):
    # BASELINE config 5: 16-bit frames, fp32 maps; oracle = upcast, sample in fp32, round once
    N, C, H, W = 2, 3, 64, 96
    frames = synth.make_frames(N, C, H, W)
    f16 = torch.from_numpy(frames).to(dtype)
    up = f16.float().numpy()
    for pad in ("zeros", "border"):
        for align in (False, True):
            grid = synth.make_map("smooth", N, H, W, align)
            ref = torch.from_numpy(oracle.forward(up, grid, pad, align)).to(dtype)
            got = pw.grid_sample(f16.cuda(), dev(grid), "bilinear", pad, align)
            assert got.dtype == dtype
            assert torch.equal(got.cpu(), ref)


def test_nonfinite_coordinates(pw):
    inp = np.arange(12, dtype=np.float32).reshape(1, 1, 3, 4) + 1
    grid = np.array([[[[np.nan, 0.0], [np.inf, 0.0], [-np.inf, np.nan], [3e38, -3e38]]]], np.float32)
    for pad in ("zeros", "border"):
        for align in (False, True):
            got = pw.grid_sample(dev(inp), dev(grid), "bilinear", pad, align)
            np.testing.assert_array_equal(got.cpu().numpy(), oracle.forward(inp, grid, pad, align))
            assert torch.equal(got, torch.ops.aten.grid_sampler_2d(dev(inp), dev(grid), 0, PAD[pad], align))


def test_error_behaviour_matches_torch(pw):
    f = torch.zeros(2, 3, 4, 4, device="cuda")
    g = torch.zeros(2, 4, 4, 2, device="cuda")
    with pytest.raises(ValueError):
        pw.grid_sample(f, g, mode="cubic")
    with pytest.raises(ValueError):
        pw.grid_sample(f, g, padding_mode="wrap")
    with pytest.raises(NotImplementedError):
        pw.grid_sample(f, g, mode="nearest", align_corners=False)
    with pytest.raises(RuntimeError, match="same batch size"):
        pw.grid_sample(f, g[:1], align_corners=False)
    with pytest.raises(RuntimeError, match="size 2 in last dimension"):
        pw.grid_sample(f, torch.zeros(2, 4, 4, 3, device="cuda"), align_corners=False)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        pw.grid_sample(f.cpu(), g.cpu(), align_corners=False)
    with pytest.warns(UserWarning, match="align_corners=False"):
        pw.grid_sample(f, g)
    # empty outputs are fine
    assert pw.grid_sample(f, torch.zeros(2, 0, 4, 2, device="cuda"), align_corners=False).shape == (2, 3, 0, 4)
    assert pw.grid_sample(f[:0], g[:0], align_corners=False).shape == (0, 3, 4, 4)


def test_install_routes_functional_grid_sample(pw):
    f = dev(synth.make_frames(1, 3, 16, 16))
    g = dev(synth.make_map("smooth", 1, 16, 16, False))
    want = F.grid_sample(f, g, align_corners=False)
    pw.install()
    try:
        import torch.nn.functional as functional  # the reference's import name (R/main_new.py:4)
        assert functional.grid_sample is pw.grid_sample
        assert torch.equal(functional.grid_sample(f, g, align_corners=False), want)
    finally:
        pw.uninstall()
    assert F.grid_sample is not pw.grid_sample


@pytest.mark.parametrize("H,W,N", [(720, 1280, 4), (1080, 1920, 3)])
def test_full_size_against_torch_cuda_and_conservation(pw, H, W, N):
    # BASELINE configs 2 and 4 geometry: bit-exact forward vs torch CUDA, gradient within
    # tolerance, and the size-independent checksum sum(grad_in) == sum(gout * valid tap weights)
    C = 3
    torch.manual_seed(0)
    frames = torch.rand(N, C, H, W, device="cuda") * 255
    grid = dev(synth.make_map("smooth", N, H, W, False, seed=11))
    gout = torch.rand(N, C, H, W, device="cuda")
    fi, gi = frames.clone().requires_grad_(True), grid.clone().requires_grad_(True)
    out = pw.grid_sample(fi, gi, align_corners=False)
    ti, tg = frames.clone().requires_grad_(True), grid.clone().requires_grad_(True)
    tout = F.grid_sample(ti, tg, align_corners=False)
    assert torch.equal(out, tout)
    out.backward(gout)
    tout.backward(gout)
    scale = float(ti.grad.abs().max())
    assert float((fi.grad - ti.grad).abs().max()) <= 1e-4 * scale
    assert float((gi.grad - tg.grad).abs().max()) <= 1e-6 * float(tg.grad.abs().max())
    x0, y0, mask, w = pw.warp_taps(grid, H, W, "zeros", False)
    valid_w = sum(w[..., k].double() * ((mask >> k) & 1).double() for k in range(4))
    want = float((gout.double().sum(1) * valid_w).sum())
    got = float(fi.grad.double().sum())
    assert abs(got - want) <= 1e-6 * abs(want)


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_frame_sharded_clip_equals_unsharded(pw, world):
    # BASELINE config 4 in miniature: a clip cut into contiguous frame ranges, one per rank; the
    # concatenation must be BIT-identical to the unsharded run (no reduction crosses ranks)
    from pwstablenet_b200 import sharding
    frames_n, C, H, W = 19, 3, 72, 128
    frames = dev(synth.make_frames(frames_n, C, H, W, seed=21))
    grid = dev(synth.make_map("smooth", frames_n, H, W, False, seed=22))
    gout = dev(synth.make_gout(frames_n, C, H, W, seed=23))
    full = pw.warp2d_forward(frames, grid, 0, False)
    full_gin, full_gg = pw.warp2d_backward(gout, frames, grid, 0, False, (True, True))
    outs, ggs = [], []
    for r in range(world):
        sh = sharding.shard_frames(frames_n, world, r)
        if sh.count == 0:
            continue
        sl = slice(sh.begin, sh.end)
        outs.append(pw.warp2d_forward(frames[sl], grid[sl], 0, False))
        _, gg = pw.warp2d_backward(gout[sl], frames[sl], grid[sl], 0, False, (False, True))
        ggs.append(gg)
    assert torch.equal(torch.cat(outs), full)
    assert torch.equal(torch.cat(ggs), full_gg)


def test_host_pipeline_matches_device_path(pw):
    # HostWarpPipeline is plumbing: results must equal the device-resident calls (forward and
    # grad_grid bit for bit; grad_input within the atomic-order tolerance)
    n, C, H, W = 7, 3, 120, 200
    frames = torch.from_numpy(synth.make_frames(n, C, H, W, seed=31)).pin_memory()
    maps = torch.from_numpy(np.ascontiguousarray(synth.make_map("smooth", n, H, W, False, seed=32).transpose(0, 3, 1, 2))).pin_memory()
    gout = torch.from_numpy(synth.make_gout(n, C, H, W, seed=33)).pin_memory()
    out, gf, gm = pw.warp_host(frames, maps, gout, chunk=2)
    grid = maps.cuda().permute(0, 2, 3, 1)
    want = pw.warp2d_forward(frames.cuda(), grid, 0, False)
    w_gin, w_gg = pw.warp2d_backward(gout.cuda(), frames.cuda(), grid, 0, False, (True, True))
    assert torch.equal(out, want.cpu())
    assert torch.equal(gm, w_gg.permute(0, 3, 1, 2).contiguous().cpu())
    assert float((gf - w_gin.cpu()).abs().max()) <= 1e-4 * float(w_gin.abs().max())
    out2, gf2, gm2 = pw.warp_host(frames, maps, None, chunk=3)
    assert gf2 is None and torch.equal(out2, out)


def test_training_shapes_take_the_one_wave_kernels(pw):
    # 16 x 3 x 256 x 256 (R/main_new.py:103-119): the working set sits in L2, the call is launch-bound -> no tensor maps, no
    # counter slots, no persistent CTAs (pws_small_problem_elems); same bits as ATen either way
    from pwstablenet_b200 import _lib
    assert _lib.small_problem_elems() == 4 << 20
    g = torch.from_numpy(synth.make_map("smooth", 16, 256, 256, False, seed=3)).cuda()
    g = g.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
    fr = torch.from_numpy(synth.make_frames(16, 3, 256, 256, seed=4)).cuda()
    go = torch.from_numpy(synth.make_gout(16, 3, 256, 256, seed=5)).cuda()
    out = pw.warp2d_forward(fr, g, 0, False)
    assert _lib.last_kernel() == "fwd_lean"
    assert torch.equal(out, torch.ops.aten.grid_sampler_2d(fr, g, 0, 0, False))
    gin, gg = pw.warp2d_backward(go, fr, g, 0, False, (True, True))
    assert _lib.last_kernel() == "bwd_lean"
    rin, rg = torch.ops.aten.grid_sampler_2d_backward(go, fr, g, 0, 0, False, (True, True))
    assert float((gg - rg).abs().max()) <= 1e-5 * float(rg.abs().max())
    assert float((gin - rin).abs().max()) <= 1e-4 * float(rin.abs().max())
    prev = _lib.small_problem_elems(0)
    try:
        assert torch.equal(pw.warp2d_forward(fr, g, 0, False), out) and _lib.last_kernel() == "fwd_tma"
        gin2, gg2 = pw.warp2d_backward(go, fr, g, 0, False, (True, True))
        assert _lib.last_kernel() == "bwd_tma" and torch.equal(gg2, gg)
    finally:
        _lib.small_problem_elems(prev)
