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
  warp_fused backward (pws_warp2d_backward_fused): FusedBackwardRef states the contract and its per-node bounds;
    backward_census restates the kernel's tile window and column runs to pick the cases that reach their edges.

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
BASE_SIZES = [(1, 1), (1, 6), (6, 1), (2, 2), (2, 7), (16, 24), (37, 53)]   # 7, 16, 24, 37, 53: the two linspace halves
                                                                            # round their middle node differently


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


U = 2.0 ** -24     # unit roundoff of fp32


class FusedBackwardRef:
    """The contract of pws_warp2d_backward_fused (include/pwswarp.h), restated on the CPU.  x: the frame as float32 (uint8
    and 16-bit frames upcast exactly), drift: planar (N, 2, h, w) float32, gout: float32 (a 16-bit grad_output upcast and
    not rounded back: the fused contract, not the stages one).
        x' = f32((x + a) * b), go' = f32(gout / d) (a true division), map = fused_map_ref
        gg, gin64 = oracle.backward(go', x', map)
    Lattice gradient (interleaved (N, h, w, 2)):
      - no upsample: glattice == gg bit for bit (tol 0), probe and NaN / inf lattices included;
      - upsample: the fp64 adjoint of the upsample (oracle.upsample_map_backward, the forward's fp32 coefficients).  Per
        node k with m_k terms t = h_l * w_l * gg: |got_k - ref_k| <= (m_k + 3) * u * sum|t|_k.  The kernel forms each
        term with two fp32 products and sums the m_k terms in some order (a shuffle scan per run of lanes, then the
        REDs); first-order fp32 summation error of m_k terms in any order is (m_k - 1) * u * sum|t|, plus one rounding
        per product and one for the RED.  A node no pixel touches is exactly 0.  Unlike a max-norm this fails when a
        run, a row of REDs or a tile's contribution goes missing from any node.
    Theta gradient: oracle.affine_theta_grad of the fp64 lattice reference, per item and entry
        |got - ref| <= sum_k |b_k| * tol_k + (ceil(nodes / 256) + 9) * u * sum_k |glat_k * b_k|
      (the kernel's glattice differs from ref by at most tol_k per node; theta_grad_kernel sums ceil(nodes / 256) fmas
      per thread, then a tree of 8 levels).
    grad_input: b * gin64, held to 1e-4 of its maximum, and its sum to b * sum go' * (valid tap weights) within 1e-6
      (check_gin); never element by element: the REDs make it order-dependent."""

    def __init__(self, x, drift, base, theta, base_align, upsample, gout, pad, align, pre=OFF_PRE, post=OFF_POST):
        has_pre, a, b, has_post, _, d, _ = scales(pre, post)
        N, C, H, W = x.shape
        Ho, Wo = gout.shape[2:]
        h, w = drift.shape[2:]
        self.upsample, self.base = upsample, base
        grid = fused_map_ref(drift, base, theta, base_align, upsample, Ho, Wo)
        with np.errstate(all="ignore"):
            xs = (np.asarray(x, F32) + a) * b if has_pre else np.ascontiguousarray(x, F32)
            go = np.asarray(gout, F32) / d if has_post else np.ascontiguousarray(gout, F32)
        _, gg, gin64 = oracle.backward(np.ascontiguousarray(go), np.ascontiguousarray(xs), grid, pad, align,
                                       want_f64_accum=True)
        if upsample is None:
            self.glat32 = gg
            self.glat64, self.tol = gg.astype(np.float64), np.zeros(gg.shape)
            self.nterms = np.ones(gg.shape, np.int64)
        else:
            g64, gabs, nterms = oracle.upsample_map_backward(gg.transpose(0, 3, 1, 2), h, w, upsample == "aligned")
            il = lambda p: np.ascontiguousarray(p.transpose(0, 2, 3, 1))   # noqa: E731  planar -> interleaved
            self.glat32 = None
            self.glat64, self.nterms = il(g64), il(nterms)
            self.tol = (self.nterms + 3) * U * il(gabs)
        if base == "affine":
            self.gtheta, gabs = oracle.affine_theta_grad(self.glat64, base_align)
            _, tol_b = oracle.affine_theta_grad(self.tol, base_align)            # sum_k |b_k| * tol_k
            self.theta_tol = tol_b + (-(-h * w // 256) + 9) * U * gabs
        self.gin64 = gin64 * float(b) if has_pre else gin64
        wsum = tap_weight_sums(grid, H, W, pad, align)
        self.checksum = float((go.astype(np.float64) * wsum[:, None]).sum()) * float(b)
        self.checksum_scale = float((np.abs(go.astype(np.float64)) * wsum[:, None]).sum()) * abs(float(b))


def half_ulp_bound(ref, dtype):
    """Half an ulp of `dtype` at |ref| (an upper bound), for a float32 result rounded once to a 16-bit type."""
    if dtype in (None, torch.float32):
        return np.zeros(np.shape(ref))
    fi = torch.finfo(dtype)
    return 0.5 * fi.eps * np.abs(ref) + float(fi.smallest_normal) * fi.eps


def check_glattice(got, ref, dtype=None, what="glattice"):
    """got: (N, h, w, 2) float32 holding the kernel's lattice gradient (rounded once to `dtype` when it is 16-bit)."""
    got = np.asarray(got, np.float64)
    if ref.upsample is None:
        want = ref.glat32 if dtype in (None, torch.float32) else round_to(ref.glat32, dtype)
        np.testing.assert_array_equal(got, want, err_msg=what)
        return
    fin = np.isfinite(ref.glat64)
    np.testing.assert_array_equal(got[~fin], ref.glat64[~fin], err_msg=what + ": non-finite nodes")
    untouched = ref.nterms == 0
    assert (got[untouched] == 0).all(), what + ": a node no pixel touches is not 0"
    tol = ref.tol + half_ulp_bound(ref.glat64, dtype)
    with np.errstate(invalid="ignore"):
        bad = fin & ~(np.abs(got - ref.glat64) <= tol)
    if bad.any():
        k = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} nodes out of bound; first {k}: got {got[k]!r}, "
                             f"ref {ref.glat64[k]!r}, bound {tol[k]!r}, terms {ref.nterms[k]}")


def check_gtheta(got, ref, what="gtheta"):
    err = np.abs(np.asarray(got, np.float64) - ref.gtheta)
    bad = ~(err <= ref.theta_tol)
    assert not bad.any(), f"{what}: entries {np.argwhere(bad).tolist()} out of bound: got {got}, ref {ref.gtheta}, " \
                          f"bound {ref.theta_tol}"


# ---------------------------------------------------------------------------------------------------------------------
# census of the fused backward's tiles: shared-memory window or per-pixel maps, and the runs of its column scan
# ---------------------------------------------------------------------------------------------------------------------
KW_TILE, KH_TILE, WIN_NODES = 64, 16, 1280      # warp_fused.cu: kTileW, kTileH, kWinNodes


def up_scale(src, dst, aligned):
    """warp_fused.cu's up_scales: (src - 1) / (dst - 1) aligned (0 for dst = 1), src / dst half_pixel, fp32 division."""
    if aligned:
        return F32(src - 1) / F32(dst - 1) if dst > 1 else F32(0)
    return F32(src) / F32(dst)


def up_coef(dst, src, scale, aligned):
    """warp_fused.cu's up_coef for an integer array dst: (i0, ip, l0, l1).  Aligned: one fp32 multiply.  half_pixel:
    fmaf(scale, dst + 0.5, -0.5) clamped at 0; the product of two fp32 values is exact in fp64 and, for a result >= 0
    (the only one the clamp keeps), so is the sum with -0.5: one rounding, as the fma."""
    d = np.asarray(dst, np.int64).astype(F32)
    if aligned:
        s = (F32(scale) * d).astype(F32)
    else:
        s = (np.float64(scale) * (d + F32(0.5)).astype(np.float64) - 0.5).astype(F32)
        s = np.where(s < 0, F32(0), s)
    i0 = s.astype(np.int64)
    ip = (i0 < src - 1).astype(np.int64)
    l1 = (s - i0.astype(F32)).astype(F32)
    return i0, ip, (F32(1) - l1).astype(F32), l1


def backward_census(mh, mw, Ho, Wo, upsample):
    """bwd_fused_kernel's structure for an upsample from an mh x mw lattice to Ho x Wo:
      nodes[ty, tx]  nr * nc of the tile's window (first / last row and column, the last clamped to Ho-1 / Wo-1);
                     <= WIN_NODES composes the window in shared memory, more evaluates the map per pixel
      runs           lengths of the runs of equal cx.i0 over the 32 lanes of each half tile row (i = 0, 1)
      split          runs that continue from lane 31 of the first half into lane 0 of the second
      ip0_runs       runs whose column has ip == 0 (two REDs into one node)
      edge_lanes     lanes past the right edge, per half (they carry zeros and join the last run)"""
    al = upsample == "aligned"
    rh, rw = up_scale(mh, Ho, al), up_scale(mw, Wo, al)
    ty, tx = -(-Ho // KH_TILE), -(-Wo // KW_TILE)
    r0 = up_coef(np.arange(ty) * KH_TILE, mh, rh, al)
    r1 = up_coef(np.minimum(np.arange(ty) * KH_TILE + KH_TILE - 1, Ho - 1), mh, rh, al)
    c0 = up_coef(np.arange(tx) * KW_TILE, mw, rw, al)
    c1 = up_coef(np.minimum(np.arange(tx) * KW_TILE + KW_TILE - 1, Wo - 1), mw, rw, al)
    nr, nc = r1[0] + r1[1] - r0[0] + 1, c1[0] + c1[1] - c0[0] + 1
    nodes = nr[:, None] * nc[None, :]
    runs, split, ip0_runs, edge = [], 0, 0, [0, 0]
    for bx in range(tx):
        w = bx * KW_TILE + np.arange(KW_TILE)
        i0, ip, _, _ = up_coef(np.minimum(w, Wo - 1), mw, rw, al)
        for half in (0, 1):
            k, p = i0[32 * half:32 * half + 32], ip[32 * half:32 * half + 32]
            starts = np.flatnonzero(np.r_[True, k[1:] != k[:-1]])
            runs += np.diff(np.r_[starts, 32]).tolist()
            ip0_runs += int((p[starts] == 0).sum())
            edge[half] += int((w[32 * half:32 * half + 32] >= Wo).sum())
        split += int(i0[31] == i0[32])
    return dict(nodes=nodes, window=int((nodes <= WIN_NODES).sum()), per_pixel=int((nodes > WIN_NODES).sum()),
                runs=np.array(runs), split=split, ip0_runs=ip0_runs, edge_lanes=tuple(edge))


def census_row(c):
    n, r = c["nodes"], c["runs"]
    return (f"nodes {', '.join(str(v) for v in sorted(set(n.ravel().tolist())))}; window {c['window']} / per-pixel "
            f"{c['per_pixel']} tiles; runs {r.min()}..{r.max()} lanes; split at 31/32: {c['split']}; ip == 0 runs: "
            f"{c['ip0_runs']}; edge lanes (first / second half): {c['edge_lanes'][0]} / {c['edge_lanes'][1]}")


# (mh, mw, Ho, Wo, upsample, what the case reaches)
BWD_CASES = [
    (8, 160, 16, 64, "aligned", "window exactly full (1280)"),
    (8, 250, 16, 100, "aligned", "full window and a clamped right tile"),
    (13, 183, 40, 64, "aligned", "window, per-pixel and window in one call (1281)"),
    (8, 251, 16, 100, "aligned", "per-pixel (1288) next to a window"),
    (20, 64, 16, 64, "half_pixel", "half_pixel window exactly full"),
    (21, 64, 16, 64, "half_pixel", "half_pixel per-pixel"),
    (4, 4, 1080, 1920, "aligned", "runs of 32 lanes, 1e5 terms per node"),
    (9, 1, 37, 90, "half_pixel", "mw = 1: ip == 0 everywhere"),
    (7, 11, 20, 65, "aligned", "Wo = 1 mod 64"),
    (7, 11, 20, 95, "half_pixel", "Wo = 31 mod 64"),
    (7, 11, 20, 97, "aligned", "Wo = 33 mod 64"),
    (7, 11, 20, 127, "half_pixel", "Wo = 63 mod 64"),
    (7, 11, 1, 70, "aligned", "Ho = 1"),
    (7, 11, 30, 1, "half_pixel", "Wo = 1"),
    (40, 9, 20, 70, "aligned", "downsample in y, upsample in x"),
    (6, 150, 50, 70, "half_pixel", "upsample in y, downsample in x: runs of one lane"),
]
BWD_IDS = [f"{c[0]}x{c[1]}-{c[2]}x{c[3]}-{c[4]}" for c in BWD_CASES]


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


ADJ_SIZES = [  # (h, w, Ho, Wo): upsample, same size, downsample, 1 x w, h x 1, 1 x 1 lattices, Ho = 1, Wo = 1
    (9, 13, 37, 53), (12, 17, 12, 17), (41, 61, 23, 29), (1, 19, 30, 40), (13, 1, 30, 40), (1, 1, 5, 7),
    (13, 19, 1, 37), (13, 19, 29, 1), (6, 150, 50, 70)]


def upsample_f64(lat, Ho, Wo, aligned):
    """fp64 bilinear resize of a planar (N, 2, h, w) array with upsample_map's fp32 coefficients: a gather, written apart
    from the oracle's scatter."""
    (yi, yp, yl0, yl1), (xi, xp, xl0, xl1) = (oracle.upsample_coefs(lat.shape[2], Ho, aligned),
                                              oracle.upsample_coefs(lat.shape[3], Wo, aligned))
    r0, r1, c0, c1 = yi, yi + yp, xi, xi + xp
    top = xl0.astype(np.float64) * lat[:, :, r0][..., c0] + xl1.astype(np.float64) * lat[:, :, r0][..., c1]
    bot = xl0.astype(np.float64) * lat[:, :, r1][..., c0] + xl1.astype(np.float64) * lat[:, :, r1][..., c1]
    return yl0.astype(np.float64)[:, None] * top + yl1.astype(np.float64)[:, None] * bot


@pytest.mark.parametrize("mode", ["aligned", "half_pixel"])
@pytest.mark.parametrize("size", ADJ_SIZES, ids=[f"{a}x{b}-{c}x{d}" for a, b, c, d in ADJ_SIZES])
def test_upsample_adjoint_identity(mode, size):
    """<U x, y> == <x, U^T y> in fp64, U the upsample with the forward's fp32 coefficients; the gather U x is the oracle's
    fp32 forward up to its own rounding.  Also the term counts: 4 per output pixel, spread over the nodes."""
    h, w, Ho, Wo = size
    al = mode == "aligned"
    rng = np.random.default_rng(h * 1000 + w)
    x = rng.standard_normal((2, 2, h, w)).astype(F32).astype(np.float64)
    y = rng.standard_normal((2, 2, Ho, Wo))
    ux = upsample_f64(x, Ho, Wo, al)
    np.testing.assert_allclose(ux, oracle.upsample_map(x.astype(F32), Ho, Wo, al), rtol=0, atol=4e-7 * np.abs(x).max())
    uty, gabs, nterms = oracle.upsample_map_backward(y, h, w, al)
    lhs, rhs = float((ux * y).sum()), float((x * uty).sum())
    assert abs(lhs - rhs) <= 1e-12 * float((np.abs(ux) * np.abs(y)).sum() + (np.abs(x) * gabs).sum())
    assert (nterms.sum(axis=(2, 3)) == 4 * Ho * Wo).all()
    assert (gabs >= np.abs(uty)).all()


@pytest.mark.parametrize("mode", ["aligned", "half_pixel"])
@pytest.mark.parametrize("size", ADJ_SIZES, ids=[f"{a}x{b}-{c}x{d}" for a, b, c, d in ADJ_SIZES])
def test_upsample_adjoint_matches_torch_interpolate(mode, size):
    """Against autograd of F.interpolate in fp64 on the CPU.  torch computes the coefficients in fp64 here, the oracle in
    fp32: a source index s < max(h, w) is off by at most 2 ulp of fp32 (scale, then fma / multiply), which moves each of
    a node's terms by at most that times |y|."""
    h, w, Ho, Wo = size
    rng = np.random.default_rng(h * 7 + w)
    y = rng.standard_normal((2, 2, Ho, Wo))
    lat = torch.zeros((2, 2, h, w), dtype=torch.float64, requires_grad=True)
    F.interpolate(lat, size=(Ho, Wo), mode="bilinear", align_corners=mode == "aligned").backward(torch.from_numpy(y))
    got, _, nterms = oracle.upsample_map_backward(y, h, w, mode == "aligned")
    tol = 4 * max(h, w) * 2.0 ** -23 * nterms * float(np.abs(y).max())
    assert (np.abs(got - lat.grad.numpy()) <= tol).all()


@pytest.mark.parametrize("base_align", [False, True])
@pytest.mark.parametrize("size", BASE_SIZES, ids=[f"{h}x{w}" for h, w in BASE_SIZES])
def test_theta_grad_matches_affine_grid_autograd(base_align, size):
    """oracle.affine_theta_grad against the fp64 CPU autograd of F.affine_grid (torch's linspace differs from the fp32
    base by its rounding); one item per N with its own theta."""
    h, w = size
    rng = np.random.default_rng(h * 31 + w)
    N = 3
    glat = rng.standard_normal((N, h, w, 2))
    theta = torch.from_numpy(rng.standard_normal((N, 2, 3))).requires_grad_(True)
    F.affine_grid(theta, (N, 1, h, w), align_corners=base_align).backward(torch.from_numpy(glat))
    got, gabs = oracle.affine_theta_grad(glat, base_align)
    assert np.abs(got - theta.grad.numpy()).max() <= 1e-6 * max(float(gabs.max()), 1.0)
    # the forward base the gradient uses is the one affine_map composes
    unit = oracle.affine_map(np.tile(np.array([[1, 0, 0], [0, 1, 0]], F32), (N, 1, 1)), h, w, None, base_align)
    ones = np.zeros((N, h, w, 2))
    ones[..., 0] = 1
    gx, _ = oracle.affine_theta_grad(ones, base_align)
    np.testing.assert_allclose(gx[:, 0, 0], unit[..., 0].astype(np.float64).sum((1, 2)), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("mode", ["aligned", "half_pixel"])
@pytest.mark.parametrize("src,dst", [(256, 1080), (256, 1920), (4, 1920), (7, 20), (20, 16), (21, 16), (183, 64),
                                     (150, 70), (1, 30), (9, 1), (13, 1), (1000, 3)])
def test_census_coefficients_are_the_oracles(mode, src, dst):
    """The census restates up_coef; it must give the C oracle's coefficients exactly (aligned: one fp32 multiply,
    half_pixel: one fma)."""
    al = mode == "aligned"
    want = oracle.upsample_coefs(src, dst, al)
    got = up_coef(np.arange(dst), src, up_scale(src, dst, al), al)
    for g, w_, name in zip(got, want, ("i0", "ip", "l0", "l1")):
        np.testing.assert_array_equal(np.asarray(g, w_.dtype), w_, err_msg=name)


def test_backward_census_cases_reach_what_they_claim():
    c = {case[-1]: backward_census(*case[:5]) for case in BWD_CASES}
    nodes = lambda what: set(c[what]["nodes"].ravel().tolist())   # noqa: E731
    assert nodes("window exactly full (1280)") == {1280}
    assert nodes("full window and a clamped right tile") == {1280, 720}
    one_call = c["window, per-pixel and window in one call (1281)"]
    assert nodes("window, per-pixel and window in one call (1281)") == {1098, 1281, 732}
    assert one_call["window"] == 2 and one_call["per_pixel"] == 1
    assert nodes("per-pixel (1288) next to a window") == {1288, 720}
    assert nodes("half_pixel window exactly full") == {1280}
    assert nodes("half_pixel per-pixel") == {1344}
    assert c["runs of 32 lanes, 1e5 terms per node"]["runs"].max() == 32
    assert c["mw = 1: ip == 0 everywhere"]["ip0_runs"] == len(c["mw = 1: ip == 0 everywhere"]["runs"])
    for what, half in (("Wo = 1 mod 64", 0), ("Wo = 31 mod 64", 0), ("Wo = 33 mod 64", 1), ("Wo = 63 mod 64", 1)):
        assert c[what]["edge_lanes"][half] > 0, what
    assert c["upsample in y, downsample in x: runs of one lane"]["runs"].min() == 1
    every = {k: sum(v[k] for v in c.values()) for k in ("split", "ip0_runs", "per_pixel")}
    assert all(every.values()), every
    lengths = set(np.concatenate([v["runs"] for v in c.values()]).tolist())
    assert {1, 32} <= lengths


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
    if out.dtype.is_floating_point:    # a differentiable call: its backward too
        check_fused_backward(frame, drift, out_size, base, theta, base_align, upsample, pad, align, pre, post)
    return out, emitted


def grad_out_dtype(frame):
    return frame.dtype if frame.dtype in (torch.float16, torch.bfloat16) else torch.float32


def fused_backward_raw(frame, drift, gout, base="none", theta=None, base_align=False, upsample=None, pad="zeros",
                       align=False, pre=OFF_PRE, post=OFF_POST, want_gin=True, map_size=None):
    """pws_warp2d_backward_fused with caller-made buffers, each NaN-filled first (the library zero-fills or stores every
    element): (rc, gin, glattice, gtheta, kernel).  gtheta is asked for with the affine base."""
    from pwstablenet_b200 import _lib, compose
    lib = _lib.load()
    N = frame.size(0)
    keep = []
    spec = compose._spec(N, drift, base, theta, base_align, upsample, map_size, pre, post, keep)
    nan = float("nan")
    gin = torch.full(frame.shape, nan, dtype=torch.float32, device="cuda") if want_gin else None
    glat = torch.full((N, spec.map_h, spec.map_w, 2), nan, dtype=torch.float32, device="cuda")
    gtheta = torch.full((N, 2, 3), nan, dtype=torch.float32, device="cuda") if base == "affine" else None
    rc = lib.pws_warp2d_backward_fused(ctypes.byref(compose._desc(gout)), ctypes.byref(compose._desc(frame)),
                                       ctypes.byref(spec), ctypes.byref(compose._desc(gin)) if gin is not None else None,
                                       ctypes.byref(compose._desc(glat)),
                                       gtheta.data_ptr() if gtheta is not None else None, PAD[pad], int(align),
                                       compose._stream(frame))
    kernel = last_kernel()
    torch.cuda.synchronize()
    return rc, gin, glat, gtheta, kernel


def check_fused_backward(frame, drift, out_size, base="none", theta=None, base_align=False, upsample=None, pad="zeros",
                         align=False, pre=OFF_PRE, post=OFF_POST, want_gin=True, seed=0):
    """The backward of a warp_fused call through the C entry point (a [-1, 1] grad_output of the frame's gradient dtype)
    against FusedBackwardRef; every buffer NaN-filled first.  Returns the reference."""
    from pwstablenet_b200 import _lib
    N, C = frame.shape[:2]
    gout = dev(synth.make_gout(N, C, *out_size, seed=seed) * F32(2) - F32(1), grad_out_dtype(frame))
    want_gin = want_gin and frame.dtype != torch.uint8
    rc, gin, glat, gtheta, kernel = fused_backward_raw(frame, drift, gout, base, theta, base_align, upsample, pad, align,
                                                       pre, post, want_gin)
    _lib.check(rc)
    assert kernel == "bwd_fused"
    ref = FusedBackwardRef(host(frame), host(drift).transpose(0, 3, 1, 2), base, None if theta is None else host(theta),
                           base_align, upsample, host(gout), pad, align, pre, post)
    check_glattice(host(glat), ref)
    if base == "affine":
        check_gtheta(host(gtheta), ref)
    if want_gin:
        check_gin(gin, ref)
    return ref


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
# warp_fused backward: window and scan boundaries, autograd layouts and routing, the C entry's edges
# ---------------------------------------------------------------------------------------------------------------------
def rough_lattice(N, h, w, seed):
    """planar (N, 2, h, w) float32 in [-1.1, 1.1]"""
    return (np.random.default_rng(seed).random((N, 2, h, w), dtype=F32) * F32(2.2) - F32(1.1)).astype(F32)


def affine_thetas(N, seed):
    """(N, 2, 3) float32, a distinct theta per item near the identity"""
    rng = np.random.default_rng(seed)
    return (np.array([[1, 0, 0], [0, 1, 0]], F32)[None] + rng.standard_normal((N, 2, 3)).astype(F32) * F32(0.08))


LATTICE_LAYOUTS = {"interleaved": lambda t: t, "planar": planar, "offset_by_one": offset_by_one}


@gpu
@pytest.mark.parametrize("case", BWD_CASES, ids=BWD_IDS)
def test_fused_backward_window_and_scan(pw, case):
    """The census cases (backward_census): shared-memory windows exactly full and one node over, both kinds of tile in
    one call, runs of 1 and 32 lanes, ip == 0 columns, lanes past the right edge in either half of a tile row.  fp32 and
    bf16 lattices, interleaved, planar (with the affine base: the window composes drift + base per node) and one element
    into its buffer (lattice_map's scalar loads); with and without a frame gradient."""
    mh, mw, Ho, Wo, upsample, _ = case
    N, C, H, W = 2, 3, 30, 44
    frame = dev(frames_pm1(N, C, H, W, seed=131))
    lat = rough_lattice(N, mh, mw, seed=132)
    theta = dev(affine_thetas(N, seed=133))
    for lt in ("f32", "bf16"):
        for layout, make in LATTICE_LAYOUTS.items():
            base = "affine" if layout == "planar" else "none"
            drift = make(dev(lat if base == "none" else lat * F32(0.05), DTYPES[lt]).permute(0, 2, 3, 1).contiguous())
            for pad, align in PAD_ALIGN:
                check_fused_backward(frame, drift, (Ho, Wo), base, theta if base == "affine" else None, align, upsample,
                                     pad, align, PRE, POST, want_gin=pad == "zeros", seed=134)


def fused_autograd_run(pw, frame, drift, theta, want, loss, **kw):
    """pw.warp_fused under autograd with requires_grad per `want` (frame, drift, theta).  Returns (grads, the grad_output
    the output received, the kernels the backward ran, read on autograd's device thread)."""
    leaves = [t.detach().requires_grad_(w and t.is_floating_point()) if t is not None else None
              for t, w in zip((frame, drift, theta), want)]
    f, d, t = leaves
    out = pw.warp_fused(f, drift=d, theta=t, **kw)
    seen, kernels = [], []
    out.register_hook(seen.append)
    for x in leaves:
        if x is not None and x.requires_grad:
            x.register_hook(lambda g: kernels.append(last_kernel()))
    loss(out).backward()
    return [x.grad if x is not None else None for x in leaves], seen[0], kernels


def check_autograd_grads(grads, want, ref, frame, drift, what):
    fg, dg, tg = grads
    if want[0] and frame.dtype != torch.uint8:
        assert fg.dtype == frame.dtype and fg.shape == frame.shape, what
        check_gin(fg, ref, extra_tol=float(torch.finfo(frame.dtype).eps) if frame.dtype != torch.float32 else 0.0)
    else:
        assert fg is None, what
    if want[1]:
        assert dg.dtype == drift.dtype and dg.shape == drift.shape, what
        check_glattice(host(dg), ref, drift.dtype, what + ": drift")
    else:
        assert dg is None, what
    if want[2]:
        check_gtheta(host(tg), ref, what + ": theta")
    else:
        assert tg is None, what


@gpu
@pytest.mark.parametrize("layout", ["channels_last", "channel_slice", "window", "out_channels_last"])
@pytest.mark.parametrize("dt,lt", [("f32", "f32"), ("bf16", "bf16"), ("f16", "f32")])
def test_fused_autograd_layouts(pw, layout, dt, lt):
    """Frame layouts, a channels-last output, and losses whose grad_output has all strides 0 (out.sum()) or a C stride of
    0, through pw.warp_fused(...).backward."""
    N, C, H, W, h, w, Ho, Wo = 2, 3, 34, 58, 11, 17, 29, 67
    T, L = DTYPES[dt], DTYPES[lt]
    frame = frame_layout(frames_pm1(N, C, H, W, seed=141), "contiguous" if layout == "out_channels_last" else layout, T)
    drift = dev(rough_lattice(N, h, w, seed=142) * F32(0.05), L).permute(0, 2, 3, 1)      # planar storage
    theta = dev(affine_thetas(N, seed=143))
    wt = dev(synth.make_gout(N, C, Ho, Wo, seed=144), T)
    w1 = dev(synth.make_gout(N, 1, Ho, Wo, seed=145)[:, 0], T)
    losses = {"(out * w).sum()": lambda o: (o * wt).sum(), "out.sum()": lambda o: o.sum(),
              "(out.sum(1) * w).sum()": lambda o: (o.sum(1) * w1).sum()}
    kw = dict(base="affine", base_align_corners=True, upsample="half_pixel", out_size=(Ho, Wo), padding_mode="border",
              align_corners=False, pre=PRE, post=POST, out_channels_last=layout == "out_channels_last")
    for name, loss in losses.items():
        grads, seen, kernels = fused_autograd_run(pw, frame, drift, theta, (True, True, True), loss, **kw)
        assert kernels and set(kernels) == {"bwd_fused"}, (name, kernels)
        if name == "out.sum()":
            assert seen.stride() == (0, 0, 0, 0)
        if name == "(out.sum(1) * w).sum()":
            assert seen.stride(1) == 0
        ref = FusedBackwardRef(host(frame), host(drift).transpose(0, 3, 1, 2), "affine", host(theta), True, "half_pixel",
                               host(seen), "border", False, PRE, POST)
        check_autograd_grads(grads, (True, True, True), ref, frame, drift, f"{layout}, {name}")


@gpu
@pytest.mark.parametrize("case", ["f32_n3", "u8_pre", "broadcast_drift"])
@pytest.mark.parametrize("upsample", [None, "aligned"])
def test_fused_autograd_routing(pw, case, upsample):
    """Each combination of frame, drift and theta requiring grad (theta alone: glattice is internal and drift.grad None),
    N = 3 with a distinct theta per item, checked per item; a uint8 frame with a pre scale; an N-broadcast drift, whose
    gradient autograd sums over the N items."""
    N, C, H, W, h, w = 3, 3, 26, 40, 9, 14
    Ho, Wo = (h, w) if upsample is None else (23, 37)
    lat = dev(rough_lattice(N, h, w, seed=151) * F32(0.05)).permute(0, 2, 3, 1).contiguous()
    theta = dev(affine_thetas(N, seed=152))
    gout = dev(synth.make_gout(N, C, Ho, Wo, seed=153) * F32(2) - F32(1))
    loss = lambda o: (o * gout).sum()   # noqa: E731
    pre = PRE
    if case == "u8_pre":
        frame = torch.from_numpy(np.random.default_rng(154).integers(0, 256, (N, H, W, C), dtype=np.uint8)).cuda()
        frame, pre = frame.permute(0, 3, 1, 2), (-127.5, 1.0 / 127.5)
    else:
        frame = dev(frames_pm1(N, C, H, W, seed=154))
    kw = dict(base="affine", upsample=upsample, out_size=(Ho, Wo), pre=pre, post=POST)
    if case == "broadcast_drift":
        one = lat[:1].clone()
        for want_theta in (False, True):
            leaf = one.detach().requires_grad_(True)
            th = theta.detach().requires_grad_(want_theta)
            pw.warp_fused(frame, drift=leaf.expand(N, h, w, 2), theta=th, **kw).backward(gout)
            ref = FusedBackwardRef(host(frame), host(one.expand(N, h, w, 2)).transpose(0, 3, 1, 2), "affine",
                                   host(theta), False, upsample, host(gout), "zeros", False, pre, POST)
            got, want = host(leaf.grad)[0].astype(np.float64), ref.glat64.sum(0)
            bound = ref.tol.sum(0) + (N - 1) * U * np.abs(ref.glat64).sum(0)   # + autograd's fp32 sum over the items
            assert (np.abs(got - want) <= bound).all()
            if want_theta:
                check_gtheta(host(th.grad), ref)
        return
    ref = FusedBackwardRef(host(frame), host(lat).transpose(0, 3, 1, 2), "affine", host(theta), False, upsample,
                           host(gout), "zeros", False, pre, POST)
    wants = [(a, b, c) for a in (False, True) for b in (False, True) for c in (False, True) if a or b or c]
    for want in wants:
        if case == "u8_pre" and want == (True, False, False):
            continue                     # a uint8 frame alone asks for no gradient: no backward runs
        grads, _, kernels = fused_autograd_run(pw, frame, lat, theta, want, loss, **kw)
        assert kernels and set(kernels) == {"bwd_fused"}, (want, kernels)
        check_autograd_grads(grads, want, ref, frame, lat, f"{case}, requires_grad {want}")


@gpu
def test_fused_backward_c_entry_edges(pw):
    """N = 0 and C = 0 leave defined (zero) gradients in NaN-filled buffers; N = 65536 and an output taller than
    65535 tiles of 16 rows are PWS_EUNSUPPORTED and leave the buffers untouched."""
    from pwstablenet_b200 import _lib
    for N, C, base in ((2, 0, "affine"), (0, 3, "none")):      # (an empty theta has no pointer to hand over)
        frame = torch.zeros((N, C, 5, 6), device="cuda")
        drift = dev(np.zeros((N, 3, 4, 2), F32))
        gout = torch.zeros((N, C, 7, 9), device="cuda")
        rc, gin, glat, gtheta, _ = fused_backward_raw(frame, drift, gout, base, dev(affine_thetas(N, 161)),
                                                      upsample="aligned")
        assert rc == _lib.PWS_OK and gin.numel() == 0
        assert glat.numel() == N * 24 and (glat == 0).all()
        assert gtheta is None or (gtheta == 0).all()
    # C = 0 through autograd: the (N, 0, H, W) grad_input torch allocates keeps strides (H*W, H*W, W, 1)
    f = torch.zeros((2, 0, 5, 6), device="cuda", requires_grad=True)
    d = torch.zeros((2, 3, 4, 2), device="cuda", requires_grad=True)
    pw.warp_fused(f, drift=d, upsample="aligned", out_size=(7, 9)).sum().backward()
    assert f.grad.shape == f.shape and d.grad.shape == d.shape and (d.grad == 0).all()
    big = 65536
    rc, gin, glat, gtheta, _ = fused_backward_raw(torch.zeros((big, 1, 1, 1), device="cuda"),
                                                  torch.zeros((big, 2, 2, 2), device="cuda"),
                                                  torch.zeros((big, 1, 2, 2), device="cuda"),
                                                  theta=torch.zeros((big, 2, 3), device="cuda"), base="affine")
    assert rc == _lib.PWS_EUNSUPPORTED
    assert all(torch.isnan(t).all() for t in (gin, glat, gtheta))
    tall = 65535 * 16 + 1
    rc, gin, glat, _, _ = fused_backward_raw(torch.zeros((1, 1, 2, 2), device="cuda"),
                                             torch.zeros((1, 2, 1, 2), device="cuda"),
                                             torch.zeros((1, 1, tall, 1), device="cuda"), upsample="aligned")
    assert rc == _lib.PWS_EUNSUPPORTED
    assert torch.isnan(gin).all() and torch.isnan(glat).all()


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
    lines.append("")
    lines.append("Every float-output call above also runs its backward (bwd_fused) against FusedBackwardRef.")
    row("test_fused_backward_window_and_scan", "bwd_fused", "rough lattice; affine base on the planar layout", "-",
        "the census cases below; f32 / bf16 lattices, interleaved, planar, one element in; with and without kGin")
    row("test_fused_autograd_layouts", "bwd_fused", "affine + drift, half_pixel", "-",
        "channels-last, channel slice, cropped window frames; channels-last output; grad_output strides 0 / C stride 0")
    row("test_fused_autograd_routing", "bwd_fused", "affine + drift, none / aligned", "-",
        "every requires_grad combination, N = 3 distinct thetas; uint8 frame with a pre scale; N-broadcast drift")
    row("test_fused_backward_c_entry_edges", "-", "-", "-", "N = 0, C = 0 (zeros); N = 65536, > 65535 row tiles")
    lines += ["", "| backward census case | lattice -> output | tiles and runs |", "|---|---|---|"]
    for mh, mw, Ho, Wo, up, what in BWD_CASES:
        lines.append(f"| {what} | {mh}x{mw} -> {Ho}x{Wo} {up} | {census_row(backward_census(mh, mw, Ho, Wo, up))} |")
    return "\n".join(lines)


if __name__ == "__main__":
    print(coverage_report())
