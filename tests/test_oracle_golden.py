"""Pins the CPU oracle (oracle/warp_oracle.c) to vectors produced by the
reference itself (tests/golden/make_golden.py: reference netG + torch CPU
grid_sample called as R/main_new.py:106,116,716 call it)."""
import hashlib
import os

import numpy as np
import pytest

import synth
from oracle import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def cfg1():
    z = np.load(os.path.join(GOLD, "config1_netg.npz"))
    rng = np.random.default_rng(123)
    frame = (rng.random((1, 3, 256, 256), dtype=np.float32) * 255).astype(np.float32)
    gout = rng.random((1, 3, 256, 256), dtype=np.float32)
    assert sha(frame) == str(z["frame_sha"])
    return z, frame, gout


def _planar_view(planar):  # (2,H,W) storage -> (1,H,W,2) view with strides (2HW, W, 1, HW)
    return np.transpose(planar[None], (0, 2, 3, 1))


CASES = [("m0", 0, False), ("m1", 1, False), ("m2", 2, False), ("gm_f", None, False), ("gm_t", None, True)]


@pytest.mark.parametrize("name,stage,align", CASES)
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_config1_reference_netg_maps(cfg1, name, stage, align, pad):
    z, frame, gout = cfg1
    if stage is None:
        planar = oracle.generate_maps(z["drift3_planar"])[0]
        assert sha(planar[None]) == str(z["genmaps_sha"])  # generate_maps restated bit-exactly
    else:
        planar = synth.config1_netg_maps(z)[stage]
    grid = _planar_view(planar)
    assert grid.strides[3] > grid.strides[2]  # the non-contiguous view the reference passes
    gout = np.ascontiguousarray(gout[:, :, ::gout.shape[2] // planar.shape[1]])  # the map's rows (every 8th: m0, m1)
    key = f"{name}_{pad}"
    out = oracle.forward(frame, grid, pad, align)
    # forward: bit-exact against torch CPU (same fma chain)
    assert sha(out) == str(z[key + "_out_sha"])
    np.testing.assert_array_equal(out[:, :, ::8, ::8], z[key + "_out_sub"])
    gin, ggrid, gin64 = oracle.backward(gout, frame, grid, pad, align, want_f64_accum=True)
    ref_gin = z[key + "_gin_sub"]
    scale = max(1.0, float(np.abs(ref_gin).max()))
    assert np.abs(gin[:, :, ::8, ::8] - ref_gin).max() <= 1e-4 * scale
    assert np.abs(gin64[:, :, ::8, ::8] - ref_gin).max() <= 1e-4 * scale
    assert abs(gin64.sum() - float(z[key + "_gin_sum"])) <= 1e-4 * max(1.0, abs(float(z[key + "_gin_sum"])))
    ref_gg = z[key + "_ggrid_sub"]
    gscale = float(np.abs(ref_gg).max())
    assert np.abs(ggrid[:, ::8, ::8, :] - ref_gg).max() <= 1e-4 * gscale
    tot = float(z[key + "_ggrid_abssum"])
    assert abs(np.abs(ggrid.astype(np.float64)).sum() - tot) <= 1e-5 * tot


def test_small_kats_full():
    z = np.load(os.path.join(GOLD, "kat_small.npz"))
    for i in range(int(z["count"])):
        k = f"k{i}"
        N, C, H, W, Ho, Wo, pad, align = [int(v) for v in z[k + "_meta"]]
        pad = "border" if pad else "zeros"
        inp, grid, gout = z[k + "_in"], z[k + "_grid"], z[k + "_gout"]
        out = oracle.forward(inp, grid, pad, bool(align))
        np.testing.assert_array_equal(out, z[k + "_out"], err_msg=k)
        gin, ggrid = oracle.backward(gout, inp, grid, pad, bool(align))
        np.testing.assert_allclose(gin, z[k + "_gin"], rtol=1e-4, atol=1e-5, err_msg=k)
        s = max(1e-6, float(np.abs(z[k + "_ggrid"]).max()))
        assert np.abs(ggrid - z[k + "_ggrid"]).max() <= 1e-4 * s, k
        # fp64 twin agrees with the fp32 path to fp32 accuracy
        o64 = oracle.forward(inp.astype(np.float64), grid.astype(np.float64), pad, bool(align))
        # coordinates landing within 1 ulp of an integer may pick another tap in fp64; compare loosely
        assert np.median(np.abs(o64 - out)) <= 1e-4


def test_taps_match_forward_and_mask_semantics():
    rng = np.random.default_rng(7)
    H, W = 9, 14
    grid = (rng.random((2, 6, 5, 2), dtype=np.float32) * 3 - 1.5).astype(np.float32)
    inp = rng.random((2, 2, H, W), dtype=np.float32)
    for pad in ("zeros", "border"):
        for align in (False, True):
            x0, y0, mask, w = oracle.taps(grid, H, W, pad, align)
            out = oracle.forward(inp, grid, pad, align)
            # rebuild the forward from the taps: same fma chain
            for n in range(2):
                for c in range(2):
                    acc = np.zeros((6, 5), np.float32)
                    for k, (dy, dx) in enumerate([(0, 0), (0, 1), (1, 0), (1, 1)]):
                        yy, xx = y0[n] + dy, x0[n] + dx
                        valid = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
                        np.testing.assert_array_equal(valid, (mask[n] >> k) & 1 == 1)
                        v = np.where(valid, inp[n, c][np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)], 0).astype(np.float32)
                        acc = (v.astype(np.float64) * w[n, :, :, k].astype(np.float64) + acc.astype(np.float64)).astype(np.float32)
                    np.testing.assert_array_equal(acc, out[n, c])
            if pad == "border":
                # clipped before floor: x0 in [0, W-1], east tap at x0 = W-1 is masked with weight 0
                assert x0.min() >= 0 and x0.max() <= W - 1
                edge = x0 == W - 1
                assert np.all(w[..., 1][edge] == 0) and np.all((mask[edge] & 2) == 0)


def test_composition_helpers_against_torch_outputs():
    z = np.load(os.path.join(GOLD, "composition.npz"))
    for align in (0, 1):
        got = oracle.affine_map(z["theta"], 16, 24, None, bool(align))
        ref = z[f"affine_{align}"]
        assert np.abs(got - ref).max() <= 2 * np.spacing(np.float32(np.abs(ref).max()))
        up = oracle.upsample_map(z["up_src"], 54, 96, bool(align))
        assert np.abs(up - z[f"up_{align}"]).max() <= 4 * np.spacing(np.float32(1.0))


def test_nonfinite_coordinates_follow_cuda_semantics():
    # zeros: non-finite -> -100 -> no taps; border: forward clips NaN to pixel 0
    # (fmaxf drops the NaN), GridSampler.cuh:53-57,138-147
    inp = np.arange(12, dtype=np.float32).reshape(1, 1, 3, 4) + 1
    grid = np.array([[[[np.nan, 0.0], [np.inf, 0.0], [-np.inf, np.nan], [3e38, -3e38]]]], np.float32)
    out_z = oracle.forward(inp, grid, "zeros", False)
    assert np.all(out_z == 0)
    x0, y0, mask, _ = oracle.taps(grid, 3, 4, "zeros", False)
    assert np.all(mask == 0) and x0[0, 0, 0] == -100
    out_b = oracle.forward(inp, grid, "border", True)
    assert np.all(np.isfinite(out_b))
    assert out_b[0, 0, 0, 2] == inp[0, 0, 0, 0]  # (-inf, NaN) -> (0, 0)


def test_inference_site_golden_from_the_reference_flow():
    # tests/golden/inference_site.npz: R/main_new.py:679-684,697-721 replayed on CPU by make_golden.py -- uint8 HWC frame,
    # netG's 256x256 stage-3 map, UpsamplingBilinear2d to the frame size, grid_sample, astype(uint8).  The oracle's
    # upsample differs from torch's by a few ulp of the map, which may flip a truncation on an integer boundary.
    site = np.load(os.path.join(GOLD, "inference_site.npz"))
    cfg = np.load(os.path.join(GOLD, "config1_netg.npz"))
    ih, iw = 144, 256
    hwc = np.random.default_rng(716).integers(0, 256, (ih, iw, 3), dtype=np.uint8)
    assert hashlib.sha256(np.ascontiguousarray(hwc).tobytes()).hexdigest() == str(site["frame_sha"])
    frame = np.ascontiguousarray(hwc.astype(np.float32).transpose(2, 0, 1)[None])
    m2 = synth.config1_netg_maps(cfg)[2][None]                        # (1,2,256,256), as netG stores it
    ident = oracle.affine_map(np.array([[[1, 0, 0], [0, 1, 0]]], np.float32), 256, 256, None, False).transpose(0, 3, 1, 2)
    for name, lattice in (("netg", m2), ("netg_plus_identity", m2 + ident)):
        up = oracle.upsample_map(lattice, ih, iw, align_corners=True)             # (1,2,H,W)
        out = oracle.forward(frame, np.ascontiguousarray(up.transpose(0, 2, 3, 1)), "zeros", False)
        want_f = site[name + "_out_f32_sub"]
        assert np.abs(out[:, :, ::4, ::4] - want_f).max() <= 1e-3, name   # measured: 0 (a map off by k ulp would move the tap by k*ulp*W/2 px)
        got = out[0].transpose(1, 2, 0).astype(np.uint8)
        diff = np.abs(got.astype(np.int32) - site[name + "_out_u8"].astype(np.int32))
        assert diff.max() <= 1 and (diff != 0).mean() < 1e-3, (name, diff.max(), (diff != 0).mean())
