"""Edge cases of the two call-site fusions, held to a CPU reference: `pw.warp_stages` (csrc/warp_stages.cu: K maps on one
frame, pre / post scale folded in, forward and backward) and `pw.warp_fused` / `pw.compose_map` (csrc/warp_fused.cu: the map
composed and upsampled inside the sampling kernel).

Both fusions have coordinate code of their own (warp_stages: src_index_f / src_index_b, the tap cache shared by the K
stages, the grad_input scatter; warp_fused: the lattice bases, the upsample coefficients, the uint8 store), so the plain
warp's tests do not reach it.  Here it runs on rough maps (random, centre-heavy, noisy, entirely off the frame), on the
probe maps of test_tile_boundaries_gpu (coordinates on every tap edge, beyond +-2^30 / +-2^31, NaN, +-inf), on 1-pixel
frames and outputs, odd sizes, every frame dtype and every switch of the scales.

The reference composes the C oracle (oracle/oracle.py) with numpy float32 elementwise ops, which round once per op as the
kernels' __fadd_rn / __fmul_rn do; 16-bit roundings go through torch CPU tensors.  No ATen CUDA op takes part in it, so the
guard probes, on which ATen's CUDA sampler has faulted, only ever meet this library's kernels and the CPU.
  warp_stages (include/pwswarp.h, pws_warp2d_stages_forward):
    tap = T((T(x + a)) * b), s = T(sample(tap, g_k)), out = T(T(s * f32(1/d)) + e)      T = rounding to the frame type
    grad_grid_k = G(oracle grad_grid of go'_k = T(gout_k * f32(1/d)))                      bit for bit
    grad_input  = b * sum_k oracle grad_input(go'_k)  (fp64)                               1e-4 of its maximum, and
                  sum(grad_input) == b * sum_k sum go'_k * (valid tap weights)             1e-6
  warp_fused (pws_warp2d_forward_fused):
    map = oracle upsample / affine / generate_maps composition                             bit for bit
    out = store(sample((x + a) * b, map) / d + e), all fp32, one rounding at the store     bit for bit
    store: the frame's 16-bit type (round to nearest), or uint8 (clamp to [0, 255], truncate, NaN -> 0)

`PYTHONPATH=.:tests python tests/test_fusion_edges_gpu.py` prints the coverage table (no GPU needed)."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import oracle
from test_tile_boundaries_gpu import PROBE_H, PROBE_W, probe_map

gpu = pytest.mark.gpu
F32 = np.float32
PAD = {"zeros": 0, "border": 1}
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16, "u8": torch.uint8}
OFF_PRE, OFF_POST = (0.0, 1.0), (1.0, 0.0)
PRE, POST = (1.0, 127.5), (127.5, -1.0)          # the reference's (x + 1) * 127.5 ... / 127.5 - 1
PAD_ALIGN = [("zeros", False), ("border", True)]


# ---------------------------------------------------------------------------------------------------------------------
# CPU reference
# ---------------------------------------------------------------------------------------------------------------------
def round_to(a, dtype):
    """float32 values rounded to `dtype` (round to nearest even, torch CPU) and read back as float32."""
    a = np.ascontiguousarray(a, F32)
    if dtype == torch.float32:
        return a
    return torch.from_numpy(a).to(dtype).float().numpy()


def scales(pre, post):
    """(has_pre, a, b, has_post, 1/d as fp32, d, e): a scale is off when it is (0, 1) resp. (1, 0), as the C ABI decides."""
    a, b, d, e = F32(pre[0]), F32(pre[1]), F32(post[0]), F32(post[1])
    return not (a == 0 and b == 1), a, b, not (d == 1 and e == 0), F32(1) / d, d, e


def tap_weight_sums(grid, H, W, pad, align):
    """Sum of the valid tap weights of every output pixel (N, Ho, Wo), float64, as the backward scatters them."""
    _, _, mask, w = oracle.taps(np.ascontiguousarray(grid), H, W, pad, align)
    valid = ((mask[..., None] >> np.arange(4)) & 1).astype(np.float64)
    wsum = (w.astype(np.float64) * valid).sum(-1)
    if pad == "border":     # the forward's clip turns a NaN coordinate into 0, the backward's keeps it (-> no tap)
        wsum[np.isnan(grid).any(-1)] = 0.0
    return wsum


def stages_taps(x, dtype, pre):
    """The pre-scaled frame warp_stages samples: T(T(x + a) * b) per element, or x when the pre scale is off."""
    has_pre, a, b, _, _, _, _ = scales(pre, OFF_POST)
    if not has_pre:
        return np.ascontiguousarray(x, F32)
    with np.errstate(all="ignore"):
        return round_to(round_to(x + a, dtype) * b, dtype)


def stages_forward_ref(x, grids, dtype, pad, align, pre=OFF_PRE, post=OFF_POST):
    """x: the frame as float32 (a 16-bit frame upcast), grids: float32 maps (upcast).  One output per map, float32
    holding values of `dtype`."""
    _, _, _, has_post, m, _, e = scales(pre, post)
    tap = stages_taps(x, dtype, pre)
    outs = []
    for g in grids:
        s = round_to(oracle.forward(tap, np.ascontiguousarray(g, F32), pad, align), dtype)
        if has_post:
            with np.errstate(all="ignore"):
                s = round_to(round_to(s * m, dtype) + e, dtype)
        outs.append(s)
    return outs


class StagesBackwardRef:
    """grad_grid of every stage (float32 holding values of the map dtype), grad_input in fp64 and its checksum, for the
    grad_outputs `gouts` (None: a stage without a grad_output, i.e. zeros)."""

    def __init__(self, x, grids, gouts, dtype, map_dtype, pad, align, pre=OFF_PRE, post=OFF_POST):
        has_pre, _, b, has_post, m, _, _ = scales(pre, post)
        N, C, H, W = x.shape
        tap = stages_taps(x, dtype, pre)
        self.gg, self.gin64 = [], np.zeros((N, C, H, W), np.float64)
        self.checksum = self.checksum_scale = 0.0
        for g, go in zip(grids, gouts):
            g = np.ascontiguousarray(g, F32)
            go = np.zeros((N, C) + g.shape[1:3], F32) if go is None else np.ascontiguousarray(go, F32)
            if has_post:            # autograd of `s / d`: grad * (1/d), a tensor of the frame's type
                go = round_to(go * m, dtype)
            _, gg, gin64 = oracle.backward(go, tap, g, pad, align, want_f64_accum=True)
            self.gg.append(round_to(gg, map_dtype))
            self.gin64 += gin64
            wsum = tap_weight_sums(g, H, W, pad, align)
            self.checksum += float((go.astype(np.float64) * wsum[:, None]).sum())
            self.checksum_scale += float((np.abs(go.astype(np.float64)) * wsum[:, None]).sum())
        if has_pre:                 # d((x + a) * b) / dx = b
            self.gin64 *= float(b)
            self.checksum *= float(b)
            self.checksum_scale *= abs(float(b))


def lattice_ref(drift, base, theta, base_align):
    """drift + base on the lattice, planar (N, 2, h, w) float32 (drift: planar)."""
    drift = np.ascontiguousarray(drift, F32)
    if base == "none":
        return drift
    if base == "identity":
        return oracle.generate_maps(drift)
    N, _, h, w = drift.shape
    return np.ascontiguousarray(oracle.affine_map(theta, h, w, drift, base_align).transpose(0, 3, 1, 2))


def fused_map_ref(drift, base, theta, base_align, upsample, Ho, Wo):
    """The map warp_fused samples with, interleaved (N, Ho, Wo, 2) float32."""
    lat = lattice_ref(drift, base, theta, base_align)
    if upsample is not None:
        lat = oracle.upsample_map(lat, Ho, Wo, upsample == "aligned")
    return np.ascontiguousarray(lat.transpose(0, 2, 3, 1))


def store(v, dtype):
    """warp_fused's store of an fp32 result: uint8 clamps to [0, 255] and truncates (NaN -> 0, fmaxf drops it), a float
    type rounds once."""
    if dtype == torch.uint8:
        return np.fmin(np.fmax(v, F32(0)), F32(255)).astype(np.uint8)
    return round_to(v, dtype)


def fused_sample_ref(x, grid, pad, align, pre, post, out_dtype):
    """x: the frame as float32 (uint8 / 16-bit upcast).  fp32 arithmetic throughout, true division by d."""
    has_pre, a, b, has_post, _, d, e = scales(pre, post)
    with np.errstate(all="ignore"):
        if has_pre:
            x = (np.asarray(x, F32) + a) * b
        s = oracle.forward(np.ascontiguousarray(x, F32), np.ascontiguousarray(grid, F32), pad, align)
        if has_post:
            s = s / d + e
    return store(s, out_dtype)


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
STAGE_KINDS = ["smooth", "random", "centre", "noisy", "offframe"]
PROBE_KINDS = ["edges", "guards"]


def make_map(kind, N, Ho, Wo, align, seed, pad="zeros"):
    """(N, Ho, Wo, 2) float32.  offframe: every coordinate outside [-1.2, 1.2]; edges / guards: the probe maps of
    test_tile_boundaries_gpu for a PROBE_H x PROBE_W frame (their own size, N = 1)."""
    if kind in PROBE_KINDS:
        return probe_map(kind, "f32", pad, align)[0]
    if kind == "offframe":
        rng = np.random.default_rng(seed)
        mag = F32(1.25) + rng.random((N, Ho, Wo, 2), dtype=F32) * F32(1.75)
        return np.where(rng.random((N, Ho, Wo, 2)) < 0.5, -mag, mag).astype(F32)
    return synth.make_map(kind, N, Ho, Wo, align, seed=seed)


def frames_pm1(N, C, H, W, seed):
    """[-1, 1] frames, as the training loop feeds them"""
    return (synth.make_frames(N, C, H, W, seed=seed) / F32(127.5) - F32(1)).astype(F32)


def dev(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda().to(dtype)


def host(t):
    """device tensor -> float32 numpy (16-bit and uint8 values upcast exactly)"""
    return t.detach().float().cpu().numpy()


def planar(g):
    return g.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)


def offset_by_one(t):
    """A dense copy of t whose storage starts one element into its buffer."""
    buf = torch.zeros(t.numel() + 1, dtype=t.dtype, device=t.device)[1:].view(t.shape)
    buf.copy_(t)
    return buf


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("align", [False, True])
def test_stages_reference_without_scales_is_the_oracle(pad, align):
    N, C, H, W, Ho, Wo = 2, 3, 9, 13, 7, 11
    x = frames_pm1(N, C, H, W, seed=1)
    grids = [make_map(k, N, Ho, Wo, align, seed=2) for k in ("random", "noisy")]
    gouts = [synth.make_gout(N, C, Ho, Wo, seed=3 + k) for k in range(2)]
    for g, out in zip(grids, stages_forward_ref(x, grids, torch.float32, pad, align)):
        np.testing.assert_array_equal(out, oracle.forward(x, g, pad, align))
    ref = StagesBackwardRef(x, grids, gouts, torch.float32, torch.float32, pad, align)
    gin64 = np.zeros(x.shape)
    for k, (g, go) in enumerate(zip(grids, gouts)):
        _, gg, gi = oracle.backward(go, x, g, pad, align, want_f64_accum=True)
        np.testing.assert_array_equal(ref.gg[k], gg)
        gin64 += gi
    np.testing.assert_array_equal(ref.gin64, gin64)
    assert abs(gin64.sum() - ref.checksum) <= 1e-9 * ref.checksum_scale


def test_stages_reference_hand_computed():
    """One output pixel halfway between two frame pixels (align_corners, a 1 x 2 frame): s = (tap0 + tap1) / 2 with the
    reference's scales, worked by hand."""
    x = np.array([[[[0.25, -0.5]]]], F32)
    g = np.array([[[[0.0, 0.0]]]], F32)                      # ix = 0.5, iy = 0: weights 0.5 / 0.5, the south row is off
    # fp32: taps 159.375, 63.75; s = 111.5625; s * f32(1/127.5) = 0.87500006 (the reciprocal is 0.007843138); - 1
    out = stages_forward_ref(x, [g], torch.float32, "zeros", True, PRE, POST)[0]
    assert out.item() == F32(-0.12499994)
    # bf16: 159.375 -> 159, 63.75 stays; s = 111.375 -> 111.5; * (1/127.5) = 0.87451 -> 0.875; - 1 = -0.125
    out = stages_forward_ref(x, [g], torch.bfloat16, "zeros", True, PRE, POST)[0]
    assert out.item() == -0.125
    # true division, one rounding: the fused contract of the same numbers
    assert fused_sample_ref(x, g, "zeros", True, PRE, POST, torch.float32).item() == F32(111.5625) / F32(127.5) - F32(1)
    # backward: go' = T(1 * (1/127.5)); grad_grid x = (W-1)/2 * (tap1 - tap0) * go'; y: (H-1)/2 = 0
    go = np.ones((1, 1, 1, 1), F32)
    ref = StagesBackwardRef(x, [g], [go], torch.float32, torch.float32, "zeros", True, PRE, POST)
    assert abs(ref.gg[0][0, 0, 0, 0] - 0.5 * (63.75 - 159.375) / 127.5) <= 1e-6 and ref.gg[0][0, 0, 0, 1] == 0
    # grad_input: b * go' * weight = 127.5 * f32(1/127.5) * 0.5 on each tap
    np.testing.assert_allclose(ref.gin64[0, 0, 0], [0.5, 0.5], rtol=1e-7)
    assert abs(ref.checksum - 1.0) <= 1e-7
    ref = StagesBackwardRef(x, [g], [go], torch.bfloat16, torch.bfloat16, "zeros", True, PRE, POST)
    # bf16(1/127.5) = 0.00787353515625; 0.5 * (63.75 - 159) * that = -0.374969..., rounded to bf16
    assert ref.gg[0][0, 0, 0, 0] == round_to(np.array([0.5 * (63.75 - 159.0) * 0.00787353515625], F32), torch.bfloat16)[0]


def test_fused_reference_uint8_store():
    v = np.array([np.nan, -np.inf, -3.7, -0.0, 0.99, 254.99, 255.0, 255.5, 1e9, np.inf], F32)
    np.testing.assert_array_equal(store(v, torch.uint8), [0, 0, 0, 0, 0, 254, 255, 255, 255, 255])


@pytest.mark.parametrize("dt", ["f16", "bf16"])
def test_fused_16bit_reference_rounds_once(dt):
    """The 16-bit contracts of the two fusions differ on ordinary inputs: warp_fused rounds once at the store, warp_stages
    after every op.  (Otherwise the comparisons below could not tell them apart.)"""
    T = DTYPES[dt]
    x = round_to(frames_pm1(1, 3, 20, 28, seed=5), T)
    g = make_map("noisy", 1, 20, 28, False, seed=6)
    once = fused_sample_ref(x, g, "zeros", False, PRE, POST, T)
    per_op = stages_forward_ref(x, [g], T, "zeros", False, PRE, POST)[0]
    assert (once != per_op).mean() > 0.05


def test_offframe_maps_are_off_the_frame():
    g = make_map("offframe", 2, 30, 40, False, seed=7)
    assert (np.abs(g) > 1.2).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()
    return pw


def last_kernel():
    from pwstablenet_b200 import _lib
    return _lib.last_kernel()


def stages_families(dtype):
    return ("stages_fwd", "stages_bwd") if dtype == torch.float32 else ("stages_fwd_16", "stages_bwd_16")


def stages_backward_raw(frame, grids, gouts, pad, align, pre, post, want_gg=None, want_gin=True):
    """pws_warp2d_stages_backward with caller-made buffers: grad_input stays the raw fp32 sums (NaN-filled first: the
    library zero-fills it), a False in want_gg passes a NULL grad_grid."""
    from pwstablenet_b200 import _lib, compose
    lib = _lib.load()
    want_gg = want_gg or [True] * len(grids)
    gin = torch.full(frame.shape, float("nan"), dtype=torch.float32, device="cuda") if want_gin else None
    ggs = [torch.full_like(g, float("nan")) if w else None for g, w in zip(grids, want_gg)]
    keep = []
    rc = lib.pws_warp2d_stages_backward(compose._desc_ptrs(gouts, keep), ctypes.byref(compose._desc(frame)),
                                        compose._desc_ptrs(grids, keep),
                                        ctypes.byref(compose._desc(gin)) if gin is not None else None,
                                        compose._desc_ptrs(ggs, keep), len(grids), pre[0], pre[1], post[0], post[1],
                                        PAD[pad], int(align), compose._stream(frame))
    _lib.check(rc)
    kernel = last_kernel()
    torch.cuda.synchronize()
    return gin, ggs, kernel


def check_gin(gin, ref, extra_tol=0.0):
    gi = gin.detach().double().cpu().numpy()
    scale = max(float(np.abs(ref.gin64).max()), 1e-30)
    assert float(np.abs(gi - ref.gin64).max()) <= (1e-4 + extra_tol) * scale
    assert abs(float(gi.sum()) - ref.checksum) <= (1e-6 + extra_tol) * ref.checksum_scale + 1e-30


def check_stages(pw, frame, grids, pad, align, pre=OFF_PRE, post=OFF_POST, gouts=None, want_gg=None):
    """Forward through pw.warp_stages and, when gouts are given, the backward through the C entry point, against the CPU
    reference; the kernel family asserted each time.  Returns the forward outputs."""
    T, G = frame.dtype, grids[0].dtype
    fam_f, fam_b = stages_families(T)
    x, gs = host(frame), [host(g) for g in grids]
    with torch.no_grad():
        outs = pw.warp_stages(frame, grids, pad, align, pre=pre, post=post)
    assert last_kernel() == fam_f
    for k, (o, want) in enumerate(zip(outs, stages_forward_ref(x, gs, T, pad, align, pre, post))):
        assert o.dtype == T and o.shape == want.shape
        np.testing.assert_array_equal(host(o), want, err_msg=f"forward, stage {k}")
    if gouts is not None:
        gin, ggs, kernel = stages_backward_raw(frame, grids, gouts, pad, align, pre, post, want_gg)
        assert kernel == fam_b
        ref = StagesBackwardRef(x, gs, [host(go) for go in gouts], T, G, pad, align, pre, post)
        for k, gg in enumerate(ggs):
            if gg is not None:
                assert gg.dtype == G
                np.testing.assert_array_equal(host(gg), ref.gg[k], err_msg=f"grad_grid, stage {k}")
        check_gin(gin, ref)
    return outs


def stage_gouts(N, C, Ho, Wo, K, dtype, seed):
    return [dev(synth.make_gout(N, C, Ho, Wo, seed=seed + k) * F32(2) - F32(1), dtype) for k in range(K)]


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: map kinds
# ---------------------------------------------------------------------------------------------------------------------
MAP_CONFIGS = [("f32", "f32"), ("f16", "f32"), ("bf16", "bf16")]      # (frame, maps): "bf16" maps are the frame's type
PROBE_CONFIGS = [("f32", "f32"), ("bf16", "f32")]                      # probes are fp32 values: a 16-bit map would move them


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("kind", STAGE_KINDS + PROBE_KINDS)
def test_stages_map_kinds(pw, kind, pad, align):
    """Three stages of one kind (unrelated seeds: the tap cache misses), or a probe map next to a smooth one."""
    if kind in PROBE_KINDS:
        probe = make_map(kind, 1, 0, 0, align, 0, pad)
        N, C, H, W, (Ho, Wo) = 1, 3, PROBE_H, PROBE_W, probe.shape[1:3]
        maps = [probe, make_map("smooth", N, Ho, Wo, align, seed=11)]
        configs = PROBE_CONFIGS
    else:
        N, C, H, W, Ho, Wo = 2, 3, 40, 72, 24, 100
        maps = [make_map(kind, N, Ho, Wo, align, seed=11 + k) for k in range(3)]
        configs = MAP_CONFIGS
    for dt, mt in configs:
        T, G = DTYPES[dt], DTYPES[mt]
        frame = dev(frames_pm1(N, C, H, W, seed=12), T)
        grids = [dev(m, G) for m in maps]
        gouts = stage_gouts(N, C, Ho, Wo, len(grids), T, seed=13)
        check_stages(pw, frame, grids, pad, align, PRE, POST, gouts)


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: stage structure (the tap cache)
# ---------------------------------------------------------------------------------------------------------------------
STRUCTURES = [("unrelated", 1), ("unrelated", 2), ("unrelated", 3), ("unrelated", 4), ("identical", 4),
              ("same_column", 3), ("cascade", 3), ("mixed_layout", 2), ("mixed_layout", 4)]


def structure_maps(structure, K, N, H, Ho, Wo, align):
    """unrelated: a different kind and seed per stage (every stage misses the tap cache); identical: one map K times
    (every stage hits); same_column: equal x, y one source row further per stage (x0 equal, y0 not); cascade: small
    refinements of one map (netG's); mixed_layout: unrelated maps, alternately planar and interleaved (and one stored one
    element into its buffer)."""
    kinds = ["random", "noisy", "centre", "smooth"]
    if structure in ("unrelated", "mixed_layout"):
        return [make_map(kinds[k], N, Ho, Wo, align, seed=21 + k) for k in range(K)]
    base = make_map("noisy", N, Ho, Wo, align, seed=21)
    if structure == "identical":
        return [base] * K
    if structure == "same_column":
        out = []
        for k in range(K):
            m = base.copy()
            m[..., 1] += F32(2.0 * k / H)
            out.append(m)
        return out
    rng = np.random.default_rng(22)
    return [(base + rng.standard_normal(base.shape).astype(F32) * F32(0.004 * k)).astype(F32) for k in range(K)]


def structure_layout(k, structure, g):
    if structure != "mixed_layout":
        return planar(g)
    return (planar, lambda t: t, offset_by_one, lambda t: t)[k](g)


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("structure,K", STRUCTURES)
def test_stages_structure(pw, structure, K, pad, align):
    N, C, H, W, Ho, Wo = 2, 3, 36, 60, 40, 70
    maps = structure_maps(structure, K, N, H, Ho, Wo, align)
    if structure == "same_column":     # the case the cache key must tell apart: same column of taps, another row
        t = [oracle.taps(m, H, W, pad, align, want_weights=False) for m in maps]
        for a, b in zip(t, t[1:]):
            assert (a[0] == b[0]).all() and (a[1] != b[1]).mean() > 0.5
    for dt, mt in (("f32", "f32"), ("bf16", "bf16")):
        T, G = DTYPES[dt], DTYPES[mt]
        frame = dev(frames_pm1(N, C, H, W, seed=23), T)
        grids = [structure_layout(k, structure, dev(m, G)) for k, m in enumerate(maps)]
        outs = check_stages(pw, frame, grids, pad, align, PRE, POST, stage_gouts(N, C, Ho, Wo, K, T, seed=24))
        if structure == "identical":
            assert all(torch.equal(o, outs[0]) for o in outs)


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: sizes
# ---------------------------------------------------------------------------------------------------------------------
STAGE_SIZES = [  # (N, C, H, W, Ho, Wo, what)
    (2, 3, 40, 72, 24, 50, "output smaller than the frame"),
    (2, 1, 30, 40, 70, 130, "output larger; Wo % 64 != 0, Ho % 16 != 0"),
    (2, 3, 1, 64, 17, 65, "1-row frame"),
    (2, 1, 48, 1, 17, 65, "1-column frame"),
    (2, 3, 1, 1, 5, 7, "1-pixel frame"),
    (3, 3, 40, 72, 1, 1, "1-pixel output"),
    (3, 1, 40, 72, 1, 97, "1-row output"),
    (2, 3, 40, 72, 33, 1, "1-column output"),
    (4, 3, 20, 30, 20, 30, "N = 4, a map per frame"),
]


@gpu
@pytest.mark.parametrize("size", STAGE_SIZES, ids=[s[-1] for s in STAGE_SIZES])
def test_stages_sizes(pw, size):
    N, C, H, W, Ho, Wo, _ = size
    maps = [make_map(k, N, Ho, Wo, False, seed=31 + i) for i, k in enumerate(("random", "noisy"))]
    for pad in ("zeros", "border"):
        for align in (False, True):
            for dt in ("f32", "bf16"):
                T = DTYPES[dt]
                frame = dev(frames_pm1(N, C, H, W, seed=32), T)
                grids = [planar(dev(maps[0], T)), dev(maps[1], T)]
                check_stages(pw, frame, grids, pad, align, PRE, POST, stage_gouts(N, C, Ho, Wo, 2, T, seed=33))


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: frame / map dtypes x scales
# ---------------------------------------------------------------------------------------------------------------------
SCALES = {
    "off": (OFF_PRE, OFF_POST),
    "pre": (PRE, OFF_POST),
    "post": (OFF_PRE, POST),
    "both": (PRE, POST),
    "div3": ((0.5, 2.0), (3.0, 0.25)),            # f32(1/3) * s differs from s / 3
    "negpre": ((1.0, -127.5), (3.0, 0.5)),
}
FRAME_MAPS = [("f32", "f32"), ("f16", "f32"), ("f16", "f16"), ("bf16", "f32"), ("bf16", "bf16")]


@gpu
@pytest.mark.parametrize("scale", list(SCALES))
@pytest.mark.parametrize("dt,mt", FRAME_MAPS)
def test_stages_dtypes_and_scales(pw, dt, mt, scale):
    pre, post = SCALES[scale]
    N, C, H, W, Ho, Wo = 2, 3, 36, 70, 30, 66
    T, G = DTYPES[dt], DTYPES[mt]
    maps = [make_map(k, N, Ho, Wo, False, seed=41 + i) for i, k in enumerate(("noisy", "random", "smooth"))]
    frame = dev(frames_pm1(N, C, H, W, seed=42), T)
    for pad, align in PAD_ALIGN:
        grids = [planar(dev(m, G)) for m in maps]
        check_stages(pw, frame, grids, pad, align, pre, post, stage_gouts(N, C, Ho, Wo, 3, T, seed=43))


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: autograd routing
# ---------------------------------------------------------------------------------------------------------------------
def autograd_run(pw, frame, grids, want_frame, want_maps, loss, pad, align):
    """pw.warp_stages under autograd.  Returns (frame grad, map grads, the grad_output each output received (None when
    the loss does not use it), the kernel the backward ran)."""
    f = frame.clone().requires_grad_(want_frame)
    gs = [g.clone().requires_grad_(w) for g, w in zip(grids, want_maps)]
    outs = pw.warp_stages(f, gs, pad, align, pre=PRE, post=POST)
    seen, kernels = [None] * len(outs), []
    for k, o in enumerate(outs):
        o.register_hook(lambda g, k=k: seen.__setitem__(k, g))
    for t in [f] + gs:          # autograd runs the node on its device thread: read the thread-local name there
        if t.requires_grad:
            t.register_hook(lambda g: kernels.append(last_kernel()))
    loss(outs).backward()
    return f.grad, [g.grad for g in gs], seen, kernels


@gpu
@pytest.mark.parametrize("dt,mt", [("f32", "f32"), ("bf16", "f32"), ("f16", "f16")])
def test_stages_autograd_routing(pw, dt, mt):
    N, C, H, W, Ho, Wo, pad, align = 2, 3, 30, 44, 26, 50, "border", False
    T, G = DTYPES[dt], DTYPES[mt]
    frame = dev(frames_pm1(N, C, H, W, seed=51), T)
    grids = [planar(dev(make_map(k, N, Ho, Wo, align, seed=52 + i), G)) for i, k in enumerate(("random", "noisy", "centre"))]
    w = [dev(synth.make_gout(N, C, Ho, Wo, seed=53 + k), T) for k in range(3)]
    w1 = [dev(synth.make_gout(N, 1, Ho, Wo, seed=56 + k)[:, 0], T) for k in range(3)]
    losses = {
        "outputs 0 and 2 only": lambda outs: (outs[0] * w[0]).sum() + (outs[2] * w[2]).sum(),
        "out.sum()": lambda outs: sum(o.sum() for o in outs),                     # grad_output strides all 0
        "out.mean(1).sum()": lambda outs: sum(o.mean(1).sum() for o in outs),
        "(out.sum(1) * w).sum()": lambda outs: sum((o.sum(1) * v).sum() for o, v in zip(outs, w1)),   # C stride 0
    }
    requests = [(True, [True, True, True]), (False, [True, False, True]), (True, [False, False, False])]
    eps = float(torch.finfo(T).eps) if T != torch.float32 else 0.0
    x, gs = host(frame), [host(g) for g in grids]
    for name, loss in losses.items():
        for want_frame, want_maps in requests:
            fgrad, ggrads, seen, kernels = autograd_run(pw, frame, grids, want_frame, want_maps, loss, pad, align)
            assert kernels and set(kernels) == {stages_families(T)[1]}, (name, kernels)
            if name == "outputs 0 and 2 only":
                assert seen[1] is None and seen[0] is not None and seen[2] is not None
            if name == "out.sum()":
                assert all(s.stride() == (0, 0, 0, 0) for s in seen)
            if name == "(out.sum(1) * w).sum()":
                assert all(s.stride(1) == 0 for s in seen)
            ref = StagesBackwardRef(x, gs, [None if s is None else host(s) for s in seen], T, G, pad, align, PRE, POST)
            for k, (gg, want) in enumerate(zip(ggrads, want_maps)):
                if not want:
                    assert gg is None
                    continue
                assert gg.dtype == G and gg.stride() == grids[k].stride()
                np.testing.assert_array_equal(host(gg), ref.gg[k], err_msg=f"{name}: grad_grid {k}")
            if want_frame:
                assert fgrad.dtype == T
                check_gin(fgrad, ref, extra_tol=eps)      # summed in fp32, rounded to the frame type once
            else:
                assert fgrad is None


# ---------------------------------------------------------------------------------------------------------------------
# warp_stages: frame and map layouts
# ---------------------------------------------------------------------------------------------------------------------
def frame_layout(x, how, T):
    """x: (N, C, H, W) float32 numpy -> a device view of it in the layout `how`."""
    N, C, H, W = x.shape
    if how == "channels_last":
        return dev(x, T).contiguous(memory_format=torch.channels_last)
    if how == "channel_slice":        # channels 1..C of a (C + 2)-channel buffer
        big = torch.zeros((N, C + 2, H, W), dtype=T, device="cuda")
        big[:, 1:1 + C] = dev(x, T)
        return big[:, 1:1 + C]
    if how == "window":               # a crop of a larger frame
        big = torch.zeros((N, C, H + 5, W + 9), dtype=T, device="cuda")
        big[:, :, 2:2 + H, 4:4 + W] = dev(x, T)
        return big[:, :, 2:2 + H, 4:4 + W]
    return dev(x, T)


@gpu
@pytest.mark.parametrize("layout", ["channels_last", "channel_slice", "window", "map_offset"])
@pytest.mark.parametrize("dt,mt", [("f32", "f32"), ("f16", "f32"), ("bf16", "bf16")])
def test_stages_layouts(pw, layout, dt, mt):
    T, G = DTYPES[dt], DTYPES[mt]
    for C in (1, 3):
        N, H, W, Ho, Wo = 2, 34, 58, 29, 67
        frame = frame_layout(frames_pm1(N, C, H, W, seed=61), layout, T)
        grids = [dev(make_map(k, N, Ho, Wo, True, seed=62 + i), G) for i, k in enumerate(("noisy", "random"))]
        grids = [offset_by_one(g) if layout == "map_offset" else planar(g) for g in grids]
        for pad, align in PAD_ALIGN:
            check_stages(pw, frame, grids, pad, align, PRE, POST, stage_gouts(N, C, Ho, Wo, 2, T, seed=63))


# ---------------------------------------------------------------------------------------------------------------------
# warp_fused / compose_map
# ---------------------------------------------------------------------------------------------------------------------
def run_fused(pw, frame, drift, out_size, base="none", theta=None, base_align=False, upsample=None, pad="zeros",
              align=False, pre=OFF_PRE, post=OFF_POST, out_dtype=None, out_cl=False, kernel="fwd_fused"):
    """warp_fused and compose_map against the CPU reference (drift: (N, h, w, 2) device view).  Returns (out, map)."""
    N = frame.size(0)
    kw = dict(drift=drift, base=base, theta=theta, base_align_corners=base_align, upsample=upsample)
    out = pw.warp_fused(frame, out_size=out_size, padding_mode=pad, align_corners=align, pre=pre, post=post,
                        out_dtype=out_dtype, out_channels_last=out_cl, **kw)
    assert last_kernel() == kernel
    emitted = pw.compose_map(N, out_size, **kw)
    assert last_kernel() == "compose_map"
    want_map = fused_map_ref(host(drift).transpose(0, 3, 1, 2), base, None if theta is None else host(theta), base_align,
                             upsample, *out_size)
    np.testing.assert_array_equal(emitted.cpu().numpy(), want_map, err_msg="emitted map")
    want = fused_sample_ref(host(frame), want_map, pad, align, pre, post, out.dtype)
    got = out.cpu().numpy() if out.dtype == torch.uint8 else host(out)
    np.testing.assert_array_equal(got, want, err_msg="fused sample")
    return out, emitted


UP_SIZES = [  # (h, w, Ho, Wo, what)
    (48, 80, 30, 50, "downsampled lattice"),
    (30, 50, 30, 50, "same size"),
    (17, 23, 40, 61, "non-integer ratio"),
    (13, 19, 1, 37, "Ho = 1"),
    (13, 19, 29, 1, "Wo = 1"),
    (1, 19, 30, 40, "1 x w lattice"),
    (13, 1, 30, 40, "h x 1 lattice"),
    (2, 2, 30, 40, "2 x 2 lattice"),
    (4, 4, 1080, 1920, "4 x 4 lattice to 1080p"),
]


@gpu
@pytest.mark.parametrize("size", UP_SIZES, ids=[s[-1] for s in UP_SIZES])
@pytest.mark.parametrize("mode", ["aligned", "half_pixel"])
def test_fused_upsample(pw, mode, size):
    h, w, Ho, Wo, _ = size
    N = 2
    rng = np.random.default_rng(71)
    lattice = (rng.random((N, 2, h, w), dtype=F32) * F32(2.2) - F32(1.1)).astype(F32)   # planar, rough
    frame = dev(frames_pm1(N, 3, 36, 52, seed=72))
    drift = dev(lattice).permute(0, 2, 3, 1)
    for pad, align in PAD_ALIGN:
        out, emitted = run_fused(pw, frame, drift, (Ho, Wo), upsample=mode, pad=pad, align=align)
        assert torch.equal(out, pw.grid_sample(frame, emitted, "bilinear", pad, align))
    # torch's CUDA upsample: a second, independent reference for the map
    ref = F.interpolate(dev(lattice), size=(Ho, Wo), mode="bilinear", align_corners=mode == "aligned")
    assert torch.equal(emitted.permute(0, 3, 1, 2), ref)


BASE_SIZES = [(1, 1), (1, 6), (6, 1), (2, 2), (2, 7), (16, 24), (37, 53)]   # 7, 16, 24, 37, 53: the two linspace halves
                                                                            # round their middle node differently


@gpu
@pytest.mark.parametrize("size", BASE_SIZES, ids=[f"{h}x{w}" for h, w in BASE_SIZES])
@pytest.mark.parametrize("base_align", [False, True])
@pytest.mark.parametrize("base", ["identity", "affine"])
def test_fused_bases(pw, base, base_align, size):
    """A lattice of size 1 makes generate_maps divide 0 by 0: the map is NaN there, in the reference as in the kernel."""
    h, w = size
    N = 2
    rng = np.random.default_rng(81)
    drift = dev((np.tanh(rng.standard_normal((N, 2, h, w))) * 0.035).astype(F32)).permute(0, 2, 3, 1)
    theta = dev((np.array([[1, 0, 0], [0, 1, 0]], F32)[None] + rng.standard_normal((N, 2, 3)).astype(F32) * F32(0.05)))
    theta = theta if base == "affine" else None
    frame = dev(frames_pm1(N, 3, 20, 28, seed=82))
    for pad, align in PAD_ALIGN:
        kw = dict(base=base, theta=theta, base_align=base_align, pad=pad, align=align)
        out, emitted = run_fused(pw, frame, drift, (h, w), **kw)
        assert torch.equal(out, pw.grid_sample(frame, emitted, "bilinear", pad, align))
        out, emitted = run_fused(pw, frame, drift, (25, 33), upsample="aligned", **kw)
        assert torch.equal(out, pw.grid_sample(frame, emitted, "bilinear", pad, align))
        run_fused(pw, frame, drift, (25, 33), upsample="half_pixel", pre=PRE, post=POST, **kw)


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("kind", ["random", "offframe"] + PROBE_KINDS)
def test_fused_rough_drifts(pw, kind, pad, align):
    """Rough lattices taken as the map (base 'none'): sampled directly and upsampled.  The probe lattices (edge and guard
    coordinates, NaN, inf) are resampled at their own size, which keeps every finite value where the probe put it."""
    if kind in PROBE_KINDS:
        lat = make_map(kind, 1, 0, 0, align, 0, pad)
        N, H, W = 1, PROBE_H, PROBE_W
        h, w = lat.shape[1:3]
        runs = [(None, (h, w)), ("half_pixel", (h, w)), ("aligned", (h, w))]
    else:
        N, H, W, h, w = 2, 40, 72, 30, 50
        lat = make_map(kind, N, h, w, align, seed=91)
        runs = [(None, (h, w)), ("aligned", (61, 97)), ("half_pixel", (23, 37))]
    frame = dev(frames_pm1(N, 3, H, W, seed=92))
    for layout in ("interleaved", "planar"):
        drift = dev(lat) if layout == "interleaved" else planar(dev(lat))
        for upsample, out_size in runs:
            out, emitted = run_fused(pw, frame, drift, out_size, upsample=upsample, pad=pad, align=align)
            assert torch.equal(out, pw.grid_sample(frame, emitted, "bilinear", pad, align))
            run_fused(pw, frame, drift, out_size, upsample=upsample, pad=pad, align=align, pre=PRE, post=POST)


FUSED_IO = [("f32", "f32"), ("u8", "f32"), ("f32", "u8"), ("u8", "u8"), ("f16", "f16"), ("bf16", "bf16")]


def fused_frame(io_in, io_out, N, C, H, W, seed):
    """float frames in [-1, 1]; for f32 -> uint8 a few NaN / +-inf pixels as well; uint8 frames random bytes."""
    if io_in == "u8":
        return torch.from_numpy(np.random.default_rng(seed).integers(0, 256, (N, C, H, W), dtype=np.uint8)).cuda()
    x = frames_pm1(N, C, H, W, seed)
    if io_out == "u8":
        x.reshape(-1)[::97] = np.nan
        x.reshape(-1)[5::89] = np.inf
        x.reshape(-1)[7::83] = -np.inf
    return dev(x, DTYPES[io_in])


FUSED_SCALES = {   # per (in, out): the scales each pair runs with, besides none
    ("f32", "f32"): [(PRE, POST)],
    ("u8", "f32"): [((-127.5, 1.0 / 127.5), OFF_POST), (OFF_PRE, (3.0, -0.5))],
    ("f32", "u8"): [((1.0, 300.0), (1.0, -50.0)), ((0.0, -1.0), (0.5, 200.0))],   # outside [0, 255] on both sides
    ("u8", "u8"): [(OFF_PRE, (0.5, -100.0))],
    ("f16", "f16"): [(PRE, POST), ((0.5, -3.0), (3.0, 0.25))],
    ("bf16", "bf16"): [(PRE, POST), ((0.5, -3.0), (3.0, 0.25))],
}


@gpu
@pytest.mark.parametrize("io", FUSED_IO, ids=[f"{a}-{b}" for a, b in FUSED_IO])
@pytest.mark.parametrize("C", [1, 2, 3, 4, 5])
def test_fused_channels_and_dtypes(pw, C, io):
    """C = 2, 4, 5 take the generic channel loop.  A 16-bit frame is computed in fp32 and rounded once at the store
    (include/pwswarp.h): the per-op rounding of warp_stages would differ."""
    N, H, W, h, w, Ho, Wo = 2, 28, 41, 19, 29, 33, 47
    frame = fused_frame(*io, N, C, H, W, seed=100 + C)
    drift = dev(make_map("noisy", N, h, w, False, seed=101))
    out_dtype = DTYPES[io[1]]
    for pad, align in PAD_ALIGN:
        for pre, post in [(OFF_PRE, OFF_POST)] + FUSED_SCALES[io]:
            out, emitted = run_fused(pw, frame, drift, (Ho, Wo), upsample="half_pixel", pad=pad, align=align, pre=pre,
                                     post=post, out_dtype=out_dtype)
            assert out.dtype == out_dtype
            if io[0] in ("f16", "bf16") and (pre, post) == (PRE, POST):
                T = out_dtype
                per_op = stages_forward_ref(host(frame), [emitted.cpu().numpy()], T, pad, align, pre, post)[0]
                assert (host(out) != per_op).any()


@gpu
@pytest.mark.parametrize("upsample", ["aligned", "half_pixel"])
def test_fused_u8_fast_path_predicate(pw, upsample):
    """The specialised uint8 kernel takes dense HWC frames and a dense, aligned interleaved lattice.  A padded batch or a
    lattice one element into its buffer falls back to the generic kernel, with the same bytes.  An expanded (N-broadcast)
    lattice is repacked by warp_fused and keeps the fast path."""
    N, H, W, h, w, Ho, Wo = 3, 45, 70, 12, 17, 37, 90
    rng = np.random.default_rng(111)
    hwc = torch.from_numpy(rng.integers(0, 256, (N, H, W, 3), dtype=np.uint8)).cuda()
    lat = dev(make_map("noisy", N, h, w, False, seed=112))
    kw = dict(upsample=upsample, out_dtype=torch.uint8, out_cl=True)
    for pad, align in PAD_ALIGN:
        fast, _ = run_fused(pw, hwc.permute(0, 3, 1, 2), lat, (Ho, Wo), pad=pad, align=align, kernel="fwd_fused_u8", **kw)
        big = torch.zeros((N, H + 3, W, 3), dtype=torch.uint8, device="cuda")
        big[:, :H] = hwc
        padded = big[:, :H].permute(0, 3, 1, 2)
        assert padded.stride(0) != 3 * H * W
        out, _ = run_fused(pw, padded, lat, (Ho, Wo), pad=pad, align=align, **kw)
        assert torch.equal(out, fast)
        off = offset_by_one(lat)
        assert off.is_contiguous() and off.storage_offset() == 1
        out, _ = run_fused(pw, hwc.permute(0, 3, 1, 2), off, (Ho, Wo), pad=pad, align=align, **kw)
        assert torch.equal(out, fast)
        one = lat[:1]
        dense, _ = run_fused(pw, hwc.permute(0, 3, 1, 2), one.repeat(N, 1, 1, 1), (Ho, Wo), pad=pad, align=align,
                             kernel="fwd_fused_u8", **kw)
        out, _ = run_fused(pw, hwc.permute(0, 3, 1, 2), one.expand(N, h, w, 2), (Ho, Wo), pad=pad, align=align,
                           kernel="fwd_fused_u8", **kw)
        assert torch.equal(out, dense)


# ---------------------------------------------------------------------------------------------------------------------
# the coverage table (host-side, no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def coverage_report():
    lines = ["| group | kernel families | maps | K | sizes and layouts |", "|" + "---|" * 5]

    def row(group, fams, maps, K, sizes):
        lines.append(f"| {group} | {fams} | {maps} | {K} | {sizes} |")

    both = "stages_fwd, stages_bwd, stages_fwd_16, stages_bwd_16"
    row("test_stages_map_kinds", both, ", ".join(STAGE_KINDS) + "; probes " + ", ".join(PROBE_KINDS) + " (fp32 maps)",
        "3 (probes: 2)", f"40x72 -> 24x100 (shorter, wider); probes {PROBE_H}x{PROBE_W} -> 48x256; "
        + "; ".join(f"{a}/{b} maps" for a, b in MAP_CONFIGS))
    row("test_stages_structure", "stages_fwd, stages_bwd, stages_fwd_16, stages_bwd_16", "random, noisy, centre, smooth",
        ", ".join(sorted({str(k) for _, k in STRUCTURES})), "; ".join(f"{s} K={k}" for s, k in STRUCTURES)
        + "; 36x60 -> 40x70")
    row("test_stages_sizes", "stages_fwd, stages_bwd, stages_fwd_16, stages_bwd_16", "random, noisy", "2",
        "; ".join(s[-1] for s in STAGE_SIZES))
    row("test_stages_dtypes_and_scales", both, "noisy, random, smooth", "3",
        "frames/maps " + ", ".join(f"{a}/{b}" for a, b in FRAME_MAPS) + "; scales " + ", ".join(SCALES))
    row("test_stages_autograd_routing", "stages_bwd, stages_bwd_16", "random, noisy, centre", "3",
        "unused outputs, NULL grad_grids, frame-only gradient, grad_output strides 0 / C stride 0")
    row("test_stages_layouts", both, "noisy, random", "2",
        "channels-last, channel slice, cropped window frames; maps one element into their buffer; C = 1, 3")
    row("test_fused_upsample", "fwd_fused, compose_map", "rough lattice, base none", "-",
        "; ".join(f"{s[-1]} ({s[0]}x{s[1]} -> {s[2]}x{s[3]})" for s in UP_SIZES) + "; aligned and half_pixel")
    row("test_fused_bases", "fwd_fused, compose_map", "identity, affine x base_align_corners", "-",
        "lattices " + ", ".join(f"{h}x{w}" for h, w in BASE_SIZES) + "; no upsample, aligned, half_pixel")
    row("test_fused_rough_drifts", "fwd_fused, compose_map", "random, offframe, probes edges, guards", "-",
        "interleaved and planar lattices; no upsample, aligned, half_pixel")
    row("test_fused_channels_and_dtypes", "fwd_fused, compose_map", "noisy", "-",
        "C = 1..5; " + ", ".join(f"{a} -> {b}" for a, b in FUSED_IO) + "; NaN / inf / out-of-range uint8 stores")
    row("test_fused_u8_fast_path_predicate", "fwd_fused_u8, fwd_fused, compose_map", "noisy", "-",
        "padded batch, lattice one element in (fall back); expanded lattice (fast path)")
    return "\n".join(lines)


if __name__ == "__main__":
    print(coverage_report())
