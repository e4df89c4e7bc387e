"""Fused map composition (SURVEY.md 8(a) rows a7-a11) on the GPU.

Contract (SURVEY section 7 "fused composition vs. the 1e-5 contract"):
  (i)   the emitted map equals the oracle's composition bit for bit and the torch-composed
        map within a couple of ulp (generate_maps: bit-exact, also against the sha256 of the
        REFERENCE's own generate_maps output in tests/golden);
  (ii)  the fused sample is bit-identical to the plain sample of the emitted map;
  (iii) end to end against the unfused torch pipeline: reported within BASELINE tolerance."""
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
    _lib.load()
    return pw


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def planar_drift(n, h, w, seed=0, amp=0.035):
    rng = np.random.default_rng(seed)
    return (np.tanh(rng.standard_normal((n, 2, h, w))) * amp).astype(np.float32)


def test_generate_maps_base_is_bit_exact_against_the_reference(pw):
    z = np.load(os.path.join(GOLD, "config1_netg.npz"))
    drift = z["drift3_planar"]                                   # (1,2,256,256): netG's stage-3 drift
    d = dev(drift).permute(0, 2, 3, 1)
    m = pw.compose_map(1, (256, 256), drift=d, base="identity")
    planar = m.permute(0, 3, 1, 2).contiguous().cpu().numpy()
    assert hashlib.sha256(planar.tobytes()).hexdigest() == str(z["genmaps_sha"])   # R/lib/utils.py:386-403 output
    np.testing.assert_array_equal(planar, oracle.generate_maps(drift))


@pytest.mark.parametrize("align", [False, True])
def test_affine_base_plus_drift(pw, align):
    n, h, w = 3, 40, 56
    rng = np.random.default_rng(3)
    theta = (np.array([[1, 0, 0], [0, 1, 0]], np.float32)[None] + rng.standard_normal((n, 2, 3)).astype(np.float32) * 0.05)
    drift = planar_drift(n, h, w, 4)
    m = pw.compose_map(n, (h, w), drift=dev(drift).permute(0, 2, 3, 1), base="affine", theta=dev(theta), base_align_corners=align)
    np.testing.assert_array_equal(m.cpu().numpy(), oracle.affine_map(theta, h, w, drift, align))
    # R/lib/networks_cascading.py:164,235: x.permute(0,2,3,1) + F.affine_grid(theta, size)
    ref = dev(drift).permute(0, 2, 3, 1) + F.affine_grid(dev(theta), (n, 3, h, w), align_corners=align)
    assert float((m - ref).abs().max()) <= 3 * np.spacing(np.float32(1.0))


@pytest.mark.parametrize("mode,align", [("aligned", True), ("half_pixel", False)])
def test_map_upsample(pw, mode, align):
    n, h, w, H, W = 2, 32, 48, 135, 240
    drift = planar_drift(n, h, w, 5, amp=1.0)
    m = pw.compose_map(n, (H, W), drift=dev(drift).permute(0, 2, 3, 1), upsample=mode)
    got = m.permute(0, 3, 1, 2).contiguous()
    np.testing.assert_array_equal(got.cpu().numpy(), oracle.upsample_map(drift, H, W, align))
    # R/main_new.py:708 UpsamplingBilinear2d (align_corners=True); R/main.py:639 nn.Upsample (False)
    # The kernel follows ATen's sm_100 SASS of upsample_bilinear2d_out_frame<float> operation for operation (source index
    # h2 * rheight resp. fma(h2 + 0.5, rheight, -0.5) clamped at 0, truncation, lambda1 = src - i, lambda0 = 1 - lambda1,
    # fma(h0, fma(w0, v00, w1 * v01), h1 * fma(w0, v10, w1 * v11))): bit-identical to torch's CUDA result
    ref = F.interpolate(dev(drift), size=(H, W), mode="bilinear", align_corners=align)
    assert torch.equal(got, ref)
    ref2 = (torch.nn.UpsamplingBilinear2d(size=(H, W)) if align else torch.nn.Upsample(size=(H, W), mode="bilinear"))(dev(drift))
    assert torch.equal(got, ref2)


def test_map_upsample_scale_factor_form(pw):
    # R/main.py:639-641: nn.Upsample(scale_factor=(H/256, W/256), mode='bilinear'): torch then derives the source scale from
    # 1/scale_factor (a double, rounded to float) instead of in/out; with H, W multiples of the lattice they coincide
    n, h, w, H, W = 1, 32, 48, 128, 240
    drift = planar_drift(n, h, w, 6, amp=1.0)
    m = pw.compose_map(n, (H, W), drift=dev(drift).permute(0, 2, 3, 1), upsample="half_pixel")
    ref = torch.nn.Upsample(scale_factor=(H / h, W / w), mode="bilinear")(dev(drift))
    assert torch.equal(m.permute(0, 3, 1, 2).contiguous(), ref)


CASES = [
    dict(base="identity", upsample=None),
    dict(base="affine", upsample=None),
    dict(base="affine", upsample="aligned"),
    dict(base="identity", upsample="half_pixel"),
    dict(base="none", upsample="aligned"),
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
def test_fused_sample_equals_plain_sample_of_the_emitted_map(pw, case, pad, align):
    n, C, H, W = 2, 3, 90, 144
    h, w = (H, W) if case["upsample"] is None else (24, 40)
    frames = dev(synth.make_frames(n, C, H, W, seed=8)) / 127.5 - 1           # the reference's [-1,1] frames
    drift = planar_drift(n, h, w, 9)
    if case["base"] == "none":   # drift is the whole map
        drift = np.ascontiguousarray(synth.make_map("smooth", n, h, w, True, seed=9).transpose(0, 3, 1, 2))
    theta = dev(np.array([[[1.01, 0.02, 0.0], [-0.02, 0.99, 0.01]]] * n, np.float32))
    kw = dict(drift=dev(drift).permute(0, 2, 3, 1), base=case["base"], theta=theta if case["base"] == "affine" else None,
              upsample=case["upsample"])
    emitted = pw.compose_map(n, (H, W), **kw)
    fused = pw.warp_fused(frames, out_size=(H, W), padding_mode=pad, align_corners=align, **kw)
    plain = pw.grid_sample(frames, emitted, "bilinear", pad, align)
    assert torch.equal(fused, plain)
    # R/main_new.py:106-107: warp((x+1)*127.5) / 127.5 - 1 folded into the same kernel.  torch's CUDA
    # `tensor / scalar` multiplies by the rounded reciprocal, the kernel divides: allow 2 ulp of the result scale
    fused2 = pw.warp_fused(frames, out_size=(H, W), padding_mode=pad, align_corners=align, pre=(1.0, 127.5), post=(127.5, -1.0), **kw)
    scaled = pw.grid_sample((frames + 1) * 127.5, emitted, "bilinear", pad, align)
    assert float((fused2 - (scaled / 127.5 - 1)).abs().max()) <= 2.5e-7
    assert torch.equal(fused2, torch.from_numpy(scaled.cpu().numpy() / np.float32(127.5) - np.float32(1)).cuda())  # true division


def test_inference_site_uint8_hwc_in_and_out(pw):
    # R/main_new.py:679-684,697-721: cv2 uint8 HWC frame, 256^2 netG map (drift + affine), UpsamplingBilinear2d
    # to the frame size, grid_sample, .astype(uint8)
    H, W = 270, 480
    rng = np.random.default_rng(11)
    hwc = torch.from_numpy(rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)).cuda()
    drift = dev(planar_drift(1, 64, 64, 12, amp=0.02))
    theta = dev(np.array([[[1.0, 0.01, 0.0], [-0.01, 1.0, 0.0]]], np.float32))
    # unfused torch pipeline, as the reference runs it
    now = hwc.float().permute(0, 3, 1, 2)
    grid = drift.permute(0, 2, 3, 1) + F.affine_grid(theta, (1, 3, 64, 64), align_corners=False)
    grid_resize = torch.nn.UpsamplingBilinear2d(size=(H, W))(grid.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
    fake = torch.ops.aten.grid_sampler_2d(now, grid_resize, 0, 0, False)
    want_u8 = fake[0].permute(1, 2, 0).cpu().numpy().astype(np.uint8)
    # fused: uint8 HWC in, uint8 HWC out, map composed and upsampled in the kernel
    out = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=drift.permute(0, 2, 3, 1), base="affine", theta=theta,
                        upsample="aligned", out_size=(H, W), out_dtype=torch.uint8, out_channels_last=True)
    got_u8 = out[0].permute(1, 2, 0).contiguous().cpu().numpy()
    assert out.permute(0, 2, 3, 1).is_contiguous()
    diff = np.abs(got_u8.astype(np.int32) - want_u8.astype(np.int32))
    print("u8 mismatch fraction", (diff != 0).mean(), "max", diff.max())
    # the map differs from torch's by a few ulp (bmm / upsample contraction): a truncation may flip on an integer boundary
    assert diff.max() <= 1 and (diff != 0).mean() < 1e-3
    # fp32 output of the same call is within BASELINE's 1e-5 of full scale of the unfused pipeline
    out_f = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=drift.permute(0, 2, 3, 1), base="affine", theta=theta,
                          upsample="aligned", out_size=(H, W), out_dtype=torch.float32)
    # reported, not gated by BASELINE (SURVEY section 7): a map that differs by k ulp moves the sample point by
    # k*ulp(1)*W/2 pixels; on white-noise frames (|gradient| up to 255 per pixel) 4 ulp is 0.03 grey levels
    bound = 255.0 * 4 * float(np.spacing(np.float32(1.0))) * W / 2
    assert float((out_f - fake).abs().max()) <= bound


def test_inference_site_is_byte_exact_against_the_torch_cuda_pipeline(pw):
    # R/main_new.py:697-721 exactly as written: netG hands over the COMPOSED 256^2 map (drift + affine were added inside
    # netG), process() upsamples it with UpsamplingBilinear2d(size=(H,W)), samples the float frame and truncates to uint8.
    # The fused kernel takes that lattice as it is: upsample (bit-exact, test_map_upsample) + sample (bit-exact) + the same
    # truncation -> every byte equal to torch's CUDA pipeline, at 1080p too
    for (H, W, hh, ww, seed) in ((270, 480, 64, 64, 21), (1080, 1920, 256, 256, 22)):
        rng = np.random.default_rng(seed)
        hwc = torch.from_numpy(rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)).cuda()
        lattice = dev(np.ascontiguousarray(synth.make_map("smooth", 1, hh, ww, False, seed=seed).transpose(0, 3, 1, 2)))  # planar, as netG stores it
        now = hwc.float().permute(0, 3, 1, 2)
        grid_resize = torch.nn.UpsamplingBilinear2d(size=(H, W))(lattice).permute(0, 2, 3, 1)
        fake = F.grid_sample(now, grid_resize, align_corners=False)
        want = fake[0].permute(1, 2, 0).cpu().numpy().astype(np.uint8)
        out = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=lattice.permute(0, 2, 3, 1), upsample="aligned", out_size=(H, W),
                            out_dtype=torch.uint8, out_channels_last=True)
        from pwstablenet_b200 import _lib
        assert _lib.last_kernel() == "fwd_fused_u8"       # netG's planar map view is repacked for the specialised kernel
        got = out[0].permute(1, 2, 0).contiguous().cpu().numpy()
        assert np.array_equal(got, want), (H, W, int((got != want).sum()))


def test_fused_errors(pw):
    f = torch.zeros(1, 3, 8, 8, device="cuda")
    d = torch.zeros(1, 4, 4, 2, device="cuda")
    with pytest.raises(RuntimeError, match="no upsample was requested"):
        pw.warp_fused(f, drift=d, out_size=(8, 8))
    with pytest.raises(RuntimeError, match="theta"):
        pw.warp_fused(f, drift=d, base="affine", upsample="aligned", out_size=(8, 8))
    with pytest.raises(NotImplementedError):
        pw.warp_fused(f, drift=d, padding_mode="reflection", upsample="aligned", out_size=(8, 8))


@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("upsample", ["aligned", "half_pixel"])
def test_inference_site_specialised_uint8_kernel_equals_the_generic_one(pw, pad, align, upsample):
    # dense uint8 HWC in/out + dense lattice take fwd_fused_u8_kernel; the same call with an NCHW-stored frame takes
    # the generic kernel: identical bytes out, for every padding / align_corners / upsample mode, partial tiles
    # included; and the truncated fp32 plain sample of the emitted map gives the same bytes again
    from pwstablenet_b200 import _lib
    N, H, W = 2, 137, 204
    rng = np.random.default_rng(5)
    hwc = torch.from_numpy(rng.integers(0, 256, (N, H, W, 3), dtype=np.uint8)).cuda()
    drift = dev(planar_drift(N, 48, 64, 3, amp=0.05)).permute(0, 2, 3, 1)
    theta = dev(np.tile(np.array([[[1.02, 0.03, 0.01], [-0.03, 0.98, -0.02]]], np.float32), (N, 1, 1)))
    kw = dict(drift=drift, base="affine", theta=theta, upsample=upsample, out_size=(H, W), padding_mode=pad,
              align_corners=align, out_dtype=torch.uint8)
    fast = pw.warp_fused(hwc.permute(0, 3, 1, 2), out_channels_last=True, **kw)
    assert _lib.last_kernel() == "fwd_fused_u8"
    nchw = hwc.permute(0, 3, 1, 2).contiguous()
    generic = pw.warp_fused(nchw, out_channels_last=False, **kw)
    assert _lib.last_kernel() == "fwd_fused"
    assert torch.equal(fast.contiguous(), generic)
    emitted = pw.compose_map(N, (H, W), drift, "affine", theta, False, upsample)
    plain = pw.grid_sample(nchw.float(), emitted, "bilinear", pad, align)
    assert torch.equal(generic, plain.clamp(0, 255).to(torch.uint8))


def test_inference_site_golden_uint8_through_the_fused_kernel(pw):
    # tests/golden/inference_site.npz (the reference flow replayed on CPU, make_golden.py): the specialised uint8 kernel
    # fed with the same frame and netG's stored stage-3 map.  The golden bytes come from torch's CPU kernels, whose
    # upsample differs from torch's own CUDA upsample by an ulp of the map here and there (different contraction), so a
    # truncation may flip on an integer boundary: <= 1 grey level in < 1e-3 of the bytes against the CPU golden, and
    # EXACTLY the bytes of torch's CUDA pipeline on the same inputs (the "netg" case, where the lattice is taken as is)
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    site = np.load(os.path.join(gold, "inference_site.npz"))
    cfg = np.load(os.path.join(gold, "config1_netg.npz"))
    ih, iw = 144, 256
    hwc = torch.from_numpy(np.random.default_rng(716).integers(0, 256, (1, ih, iw, 3), dtype=np.uint8)).cuda()
    m2 = dev(synth.config1_netg_maps(cfg)[2][None])            # (1,2,256,256) planar, as netG stores it
    theta = dev(np.array([[[1, 0, 0], [0, 1, 0]]], np.float32))
    for name, kw in (("netg", dict(base="none")), ("netg_plus_identity", dict(base="affine", theta=theta))):
        out = pw.warp_fused(hwc.permute(0, 3, 1, 2), drift=m2.permute(0, 2, 3, 1), upsample="aligned", out_size=(ih, iw),
                            out_dtype=torch.uint8, out_channels_last=True, **kw)
        got = out[0].permute(1, 2, 0).contiguous().cpu().numpy()
        diff = np.abs(got.astype(np.int32) - site[name + "_out_u8"].astype(np.int32))
        assert diff.max() <= 1 and (diff != 0).mean() < 1e-3, (name, int(diff.max()), float((diff != 0).mean()))
        if name == "netg":
            grid_resize = torch.nn.UpsamplingBilinear2d(size=(ih, iw))(m2).permute(0, 2, 3, 1)
            fake = F.grid_sample(hwc.float().permute(0, 3, 1, 2), grid_resize, align_corners=False)
            assert np.array_equal(got, fake[0].permute(1, 2, 0).cpu().numpy().astype(np.uint8))
