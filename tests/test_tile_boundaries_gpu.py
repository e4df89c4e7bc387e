"""Boundary tests of the TMA warp kernels (csrc/warp_fwd_tma.cu, csrc/warp_bwd_tma.cu) and of the lean kernels behind them.

The TMA kernels sort every 64x16 tile of output pixels into one of four classes (pws_pipe.cuh, box_of_range):
  interior  the tile is full and every tap of every pixel lies inside the frame: mask-free body on a staged box;
  masked    some tap may be outside: per-tap masks, taps still read from the staged box;
  fallback  the box fits no shape, or the map holds NaN / inf / a coordinate beyond +-2^30: gather from global memory;
  empty     no tap is inside the frame: nothing is staged or read;
and stage one of three box shapes (72x20, 80x24, 88x27 pixels; 84 in place of 88 for channels-last frames).  A wrong
rule there does not fault: the kernel reads a neighbouring box row, or runs the mask-free body on a tap that needs a mask,
and the result is silently off.  So the outputs whose contract is bit-exactness -- the forward and grad_grid -- are
compared with the CPU oracle bit for bit, on inputs built to sit on each boundary, and a host-side restatement of the
tile classifier (`tile_classes`, pinned on the CPU below) proves which class and box each tile really took.  grad_input
keeps the suite's standard: <= 1e-4 of its maximum against the float64-accumulated oracle, plus the checksum
sum(grad_input) == sum(grad_out * valid tap weights).

`PYTHONPATH=.:tests python tests/test_tile_boundaries_gpu.py` prints the classifier's census of every case and probe (no GPU needed)."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch

import synth
from oracle import oracle

gpu = pytest.mark.gpu
PAD = {"zeros": 0, "border": 1}
TW, TH = 64, 16                       # output pixels per tile (pws_pipe.cuh kTW, kTH)
BOX_W, BOX_H = (72, 80, 88), (20, 24, 27)
BOX_W_CL = (72, 80, 84)               # channels-last RGB: a TMA box row holds at most 256 elements
SANE = np.float32(2.0 ** 30)          # beyond it ATen's -100 guard breaks monotonicity: the tile takes the fallback
INTERIOR, MASKED, FALLBACK, EMPTY = "interior", "masked", "fallback", "empty"
CLASSES = (INTERIOR, MASKED, FALLBACK, EMPTY)
F32 = np.float32


# ---------------------------------------------------------------------------------------------------------------------
# host-side tile classifier
# ---------------------------------------------------------------------------------------------------------------------
def unnorm(coord, size, align):
    """The kernels' raw unnormalised source coordinate (no clip, no guard), float32.
    align_corners: ((x + 1) * 0.5) * (size - 1), each op rounded in float32.  Otherwise fma(x + 1, size, -1) * 0.5: the
    product is exact in float64 and so is the subtraction below 2^53 (every coordinate the +-2^30 test lets through), so
    one rounding to float32 is the fma's."""
    t = np.asarray(coord, F32) + F32(1)
    with np.errstate(all="ignore"):
        if align:
            return (t * F32(0.5)) * F32(size - 1)
        return (t.astype(np.float64) * size - 1.0).astype(F32) * F32(0.5)


def source_floors(grid, H, W, align):
    """floor of the unnormalised coordinate of every pixel, float64 (NaN / inf kept)."""
    g = np.asarray(grid, F32)
    return np.floor(unnorm(g[..., 0], W, align).astype(np.float64)), np.floor(unnorm(g[..., 1], H, align).astype(np.float64))


def tile_classes(grid, H, W, padding="zeros", align=False, xal=4, cl=False):
    """box_of_range over the 64x16 tile walk of an (N, Ho, Wo, 2) fp32 map, for an H x W frame.  xal: pixels per 16 bytes
    of a frame row (4 for fp32 frames, 8 for 16-bit ones; the box start rounds down to it); cl: channels-last frame.
    Returns a dict of (N, tiles_y, tiles_x) arrays: 'cls' (one of CLASSES), 'shape' (0..2, -1 without a box), 'bx', 'by',
    'bw', 'bh' (the box extent the shape was chosen for)."""
    g = np.asarray(grid, F32)
    N, Ho, Wo, _ = g.shape
    ty, tx = -(-Ho // TH), -(-Wo // TW)

    def extreme(v, fill, red):   # min.NaN / max.NaN over a tile's valid pixels: numpy's min / max propagate NaN too
        p = np.full((N, ty * TH, tx * TW), fill, F32)
        p[:, :Ho, :Wo] = v
        return red(p.reshape(N, ty, TH, tx, TW), axis=(2, 4))

    xlo, xhi = extreme(g[..., 0], np.inf, np.min), extreme(g[..., 0], -np.inf, np.max)
    ylo, yhi = extreme(g[..., 1], np.inf, np.min), extreme(g[..., 1], -np.inf, np.max)
    full = np.zeros((N, ty, tx), bool)
    full[:, :Ho // TH, :Wo // TW] = True
    fxlo, fxhi, fylo, fyhi = unnorm(xlo, W, align), unnorm(xhi, W, align), unnorm(ylo, H, align), unnorm(yhi, H, align)
    with np.errstate(invalid="ignore"):
        sane = (fxlo >= -SANE) & (fxhi <= SANE) & (fylo >= -SANE) & (fyhi <= SANE)
    fl = lambda v: np.floor(np.where(sane, v, 0)).astype(np.int64)   # noqa: E731
    x0lo, x0hi, y0lo, y0hi = fl(fxlo), fl(fxhi), fl(fylo), fl(fyhi)
    interior = (x0lo >= 0) & (x0hi + 1 <= W - 1) & (y0lo >= 0) & (y0hi + 1 <= H - 1) & full
    if padding == "border":
        with np.errstate(invalid="ignore"):
            interior &= (fxlo > 0) & (fylo > 0)
        x0lo, x0hi = np.clip(x0lo, 0, W - 1), np.clip(x0hi, 0, W - 1)
        y0lo, y0hi = np.clip(y0lo, 0, H - 1), np.clip(y0hi, 0, H - 1)
    bx, by = np.maximum(x0lo, 0) & ~(xal - 1), np.maximum(y0lo, 0)
    bw, bh = np.minimum(x0hi + 1, W - 1) - bx + 1, np.minimum(y0hi + 1, H - 1) - by + 1
    widths = BOX_W_CL if cl else BOX_W
    shape = np.select([(bw <= widths[s]) & (bh <= BOX_H[s]) for s in range(3)], [0, 1, 2], -1)
    empty = (bw <= 0) | (bh <= 0)
    cls = np.where(~sane | (~empty & (shape < 0)), FALLBACK, np.where(empty, EMPTY, np.where(interior, INTERIOR, MASKED)))
    boxed = (cls == INTERIOR) | (cls == MASKED)
    return {"cls": cls, "shape": np.where(boxed, shape, -1), "bx": bx, "by": by, "bw": bw, "bh": bh}


def census(tc):
    return {c: int((tc["cls"] == c).sum()) for c in CLASSES}


def box_shape_for(bw, bh, cl=False):
    widths = BOX_W_CL if cl else BOX_W
    for s in range(3):
        if bw <= widths[s] and bh <= BOX_H[s]:
            return s
    return -1


# ---------------------------------------------------------------------------------------------------------------------
# probe maps: one affine patch per tile, each on a classification boundary
# ---------------------------------------------------------------------------------------------------------------------
def coord_to_map(X, size, align):
    """inverse of unnorm in float64 (source coordinate -> map value)"""
    X = np.asarray(X, np.float64)
    return 2.0 * X / (size - 1) - 1.0 if align else (2.0 * X + 1.0) / size - 1.0


def _key(x):       # float32 -> int, monotone in the value (both zeros -> 0)
    i = int(np.asarray(x, F32).view(np.int32))
    return i if i >= 0 else -(i & 0x7FFFFFFF)


def _unkey(k):
    return np.asarray(k if k >= 0 else (-k) | -0x80000000, np.int32).view(F32)[()]


def solve(target, size, align, side="le"):
    """A float32 map value whose unnormalised coordinate relates to `target` as `side` says: 'eq' exactly target, 'le'
    the largest reachable value <= target, 'lt' the largest < target, 'gt' the smallest > target, 'ge' the smallest
    >= target.  unnorm is monotone: a bisection over the ordered float32 values, started at the float64 inverse."""
    strict = side in ("lt", "ge")
    below = lambda k: (float(unnorm(_unkey(k), size, align)) < target) if strict else \
        (float(unnorm(_unkey(k), size, align)) <= target)   # noqa: E731
    lim = _key(F32(np.inf))
    k0 = _key(F32(coord_to_map(target, size, align)))
    step, lo, hi = 1, k0, k0                 # bracket: below(lo), not below(hi)
    if below(k0):
        while hi < lim and below(hi):
            lo, hi, step = hi, min(k0 + step, lim), step * 2
    else:
        while lo > -lim and not below(lo):
            hi, lo, step = lo, max(k0 - step, -lim), step * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if below(mid) else (lo, mid)
    x = _unkey(lo) if side in ("le", "lt", "eq") else _unkey(hi)
    if side == "eq":
        assert float(unnorm(x, size, align)) == target, f"{target} is not reachable (closest below: {unnorm(x, size, align)!r})"
    return x


def patch(H, W, align, xr, yr, override=None):
    """A 16x64 tile of map values whose source x runs from xr[0] (first column) to xr[1] (last column) and source y
    from yr[0] (first row) to yr[1] (last row).  An end may be a number (the largest reachable coordinate <= it) or
    (number, side) for `solve`.  override: (row, col, x map value or None, y map value or None)."""
    def ends(r, size):
        a, b = ((v, "le") if np.isscalar(v) else v for v in r)
        return solve(a[0], size, align, a[1]), solve(b[0], size, align, b[1]), float(a[0]), float(b[0])

    x_a, x_b, X0, X1 = ends(xr, W)
    y_a, y_b, Y0, Y1 = ends(yr, H)
    mx = coord_to_map(np.linspace(X0, X1, TW), W, align).astype(F32)
    my = coord_to_map(np.linspace(Y0, Y1, TH), H, align).astype(F32)
    mx[0], mx[-1], my[0], my[-1] = x_a, x_b, y_a, y_b
    t = np.empty((TH, TW, 2), F32)
    t[..., 0] = mx[None, :]
    t[..., 1] = my[:, None]
    if override is not None:
        r, c, vx, vy = override
        if vx is not None:
            t[r, c, 0] = vx
        if vy is not None:
            t[r, c, 1] = vy
    return t


PROBE_H, PROBE_W = 64, 256            # powers of two: coordinate 0 is reachable without align_corners too
PROBE_TILES_X = 4


def assemble(tiles):
    """tiles -> one (1, Ho, 256, 2) map, four tiles per tile row; the spare tiles repeat the first probe."""
    rows = -(-len(tiles) // PROBE_TILES_X)
    tiles = tiles + [tiles[0]] * (rows * PROBE_TILES_X - len(tiles))
    m = np.concatenate([np.concatenate(tiles[r * PROBE_TILES_X:(r + 1) * PROBE_TILES_X], axis=1) for r in range(rows)], axis=0)
    return m[None]


def extent_probes(frame, pad, align):
    """Box extents at and around every shape threshold, with and without the alignment slack of the box start.
    frame: 'f32' (NCHW), 'cl' (fp32 channels-last) or 'f16' (16-bit).  Returns [(tile, expected dict)]."""
    xal = 8 if frame == "f16" else 4
    bws = [71, 72, 73, 79, 80, 81, 87, 88, 89] + ([83, 84, 85] if frame == "cl" else [])
    bhs = [19, 20, 21, 23, 24, 25, 26, 27, 28]
    bx0, by0 = 64, 8
    out = []
    for slack in (0, xal - 1):
        for bw in bws:
            for bh in bhs:
                # first column floors to bx0 + slack (the box start rounds down to bx0), last column to bx0 + bw - 2:
                # the box spans bx0 .. bx0 + bw - 1 (the east taps); the same in y without the rounding
                t = patch(PROBE_H, PROBE_W, align, (bx0 + slack + 0.25, bx0 + bw - 1.5), (by0 + 0.25, by0 + bh - 1.5))
                shape = box_shape_for(bw, bh, frame == "cl")
                out.append((t, {"probe": f"box {bw}x{bh} slack {slack}", "bw": bw, "bh": bh, "shape": shape,
                                "cls": INTERIOR if shape >= 0 else FALLBACK}))
    return out


def edge_probes(pad, align):
    """The extreme tap coordinate of an otherwise interior tile on each side of the interior test."""
    H, W = PROBE_H, PROBE_W
    below = lambda v: (v, "lt")               # noqa: E731   largest reachable coordinate below v
    yr, xr = (10.3, 25.7), (40.3, 100.7)
    low_in = MASKED if pad == "border" else INTERIOR   # a coordinate exactly on 0: border padding zeroes its map gradient
    cases = [
        ("x max = largest float below W-1", (W - 60.3, below(W - 1.0)), yr, INTERIOR),
        ("x max = W-1", (W - 60.3, (W - 1.0, "eq")), yr, MASKED),
        ("x max = W-2", (W - 60.3, (W - 2.0, "eq")), yr, INTERIOR),
        ("y max = largest float below H-1", xr, (H - 12.3, below(H - 1.0)), INTERIOR),
        ("y max = H-1", xr, (H - 12.3, (H - 1.0, "eq")), MASKED),
        ("y max = H-2", xr, (H - 12.3, (H - 2.0, "eq")), INTERIOR),
        ("x min = 0", ((0.0, "eq"), 60.7), yr, low_in),
        ("x min = smallest coordinate above 0", ((0.0, "gt"), 60.7), yr, INTERIOR),
        ("x min = largest coordinate below 0", ((0.0, "lt"), 60.7), yr, MASKED),
        ("y min = 0", xr, ((0.0, "eq"), 14.7), low_in),
        ("y min = smallest coordinate above 0", xr, ((0.0, "gt"), 14.7), INTERIOR),
        ("y min = largest coordinate below 0", xr, ((0.0, "lt"), 14.7), MASKED),
    ]
    return [(patch(H, W, align, x, y), {"probe": name, "cls": cls}) for name, x, y, cls in cases]


def guard_probes(pad, align):
    """One pixel of a tile on either side of the +-2^30 'sane' bound and of ATen's int-range guard (+-2^31), and NaN /
    +-inf in an otherwise interior tile.  Beyond-the-frame coordinates inside the bound keep a box (it is clamped to the
    frame): the tile stays masked.  Beyond it, the tile gathers from global memory."""
    H, W = PROBE_H, PROBE_W
    right, left, mid, yr = (W - 50.3, W - 2.5), (1.3, 50.7), (40.3, 100.7), (10.3, 25.7)
    sx = lambda v, side: solve(v, W, align, side)   # noqa: E731
    b30, b31 = float(2 ** 30), float(2 ** 31)
    cases = [
        ("x = 2^30 or just below", right, (sx(b30, "le"), None), MASKED),
        ("x just above 2^30", right, (sx(b30, "gt"), None), FALLBACK),
        ("x = -2^30 or just above", left, (sx(-b30, "ge"), None), MASKED),
        ("x just below -2^30", left, (sx(-b30, "lt"), None), FALLBACK),
        ("x = 2^31 or just below (int-range guard)", right, (sx(b31, "le"), None), FALLBACK),
        ("x just above 2^31 (-100 guard)", right, (sx(b31, "gt"), None), FALLBACK),
        ("x = -2^31 or just above", left, (sx(-b31, "ge"), None), FALLBACK),
        ("x just below -2^31 (-100 guard)", left, (sx(-b31, "lt"), None), FALLBACK),
        ("x NaN", mid, (F32(np.nan), None), FALLBACK),
        ("y NaN", mid, (None, F32(np.nan)), FALLBACK),
        ("x +inf", mid, (F32(np.inf), None), FALLBACK),
        ("y -inf", mid, (None, F32(-np.inf)), FALLBACK),
    ]
    return [(patch(H, W, align, xr, yr, (5, 30) + ov), {"probe": name, "cls": cls}) for name, xr, ov, cls in cases]


def probe_map(kind, frame, pad, align):
    probes = extent_probes(frame, pad, align) if kind == "extents" else edge_probes(pad, align) if kind == "edges" \
        else guard_probes(pad, align)
    return assemble([t for t, _ in probes]), [e for _, e in probes]


def check_probe_classes(grid, expect, frame, pad, align):
    """The classifier confirms every probe tile's intended class (and box, for the extent probes)."""
    tc = tile_classes(grid, PROBE_H, PROBE_W, pad, align, xal=8 if frame == "f16" else 4, cl=frame == "cl")
    for i, e in enumerate(expect):
        r, c = divmod(i, PROBE_TILES_X)
        got = {k: tc[k][0, r, c] for k in ("cls", "shape", "bw", "bh")}
        assert got["cls"] == e["cls"], (e["probe"], got)
        if "bw" in e:
            assert (got["bw"], got["bh"], got["shape"]) == (e["bw"], e["bh"], e["shape"]), (e["probe"], got)
    return tc


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the classifier and the probe builder
# ---------------------------------------------------------------------------------------------------------------------
def _pin_floors(grid, H, W, align):
    fx, fy = source_floors(grid, H, W, align)
    x0, y0, _, _ = oracle.taps(np.ascontiguousarray(grid), H, W, "zeros", align, want_weights=False)
    for f, o in ((fx, x0), (fy, y0)):
        with np.errstate(invalid="ignore"):
            ok = (f >= -2.0 ** 31) & (f < 2.0 ** 31)
            guarded = ~np.isfinite(f) | (np.abs(f) > 2.0 ** 31)     # ATen's guard: -100 for NaN / inf / beyond the int range
        np.testing.assert_array_equal(f[ok].astype(np.int64), o[ok])
        assert (o[guarded] == -100).all()
        # (exactly 2^31 passes the guard, and its floor does not fit an int: left out)


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("kind", ["smooth", "identity", "random", "centre", "noisy"])
def test_classifier_floors_match_the_oracle_on_synth_maps(kind, align):
    for H, W in ((270, 480), (40, 72), (1, 64), (2000, 4)):
        _pin_floors(synth.make_map(kind, 2, min(H, 64), 96, align, seed=7), H, W, align)


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("kind,frame", [("extents", "f32"), ("extents", "cl"), ("extents", "f16"), ("edges", "f32"),
                                        ("guards", "f32")])
def test_probe_maps_sit_where_they_were_built(kind, frame, pad, align):
    grid, expect = probe_map(kind, frame, pad, align)
    _pin_floors(grid, PROBE_H, PROBE_W, align)
    check_probe_classes(grid, expect, frame, pad, align)
    if kind == "edges":
        H, W = PROBE_H, PROBE_W
        for (t, e) in edge_probes(pad, align):
            ux, uy = unnorm(t[..., 0], W, align), unnorm(t[..., 1], H, align)
            if "W-1" in e["probe"]:
                want = np.nextafter(F32(W - 1), F32(0)) if "below" in e["probe"] else F32(W - 1)
                assert ux.max() == want
            if e["probe"] == "x min = 0":
                assert ux.min() == 0.0
            if e["probe"] == "x min = smallest coordinate above 0":
                assert ux.min() > 0.0 and unnorm(np.nextafter(t[0, 0, 0], F32(-np.inf)), W, align) <= 0.0


def test_classifier_hand_computed_tiles():
    H, W = 64, 256

    def one(X, Y):     # a full tile whose every pixel samples the source point (X, Y) (or the closest one below)
        g = np.empty((1, TH, TW, 2), F32)
        g[..., 0] = solve(X, W, False)
        g[..., 1] = solve(Y, H, False)
        return g

    tc = tile_classes(one(10.5, 5.5), H, W)             # taps x 10..11, y 5..6; box from x 8: 4 x 2
    assert (tc["cls"][0, 0, 0], tc["shape"][0, 0, 0], tc["bx"][0, 0, 0], tc["bw"][0, 0, 0], tc["bh"][0, 0, 0]) == (INTERIOR, 0, 8, 4, 2)
    tc = tile_classes(one(13.5, 5.5), H, W, xal=8)      # a 16-bit box starts on a multiple of 8 pixels
    assert (tc["bx"][0, 0, 0], tc["bw"][0, 0, 0]) == (8, 7)
    assert tile_classes(one(-5.0, 5.5), H, W)["cls"][0, 0, 0] == EMPTY          # every tap left of the frame
    assert tile_classes(one(300.0, 5.5), H, W)["cls"][0, 0, 0] == EMPTY
    assert tile_classes(one(-5.0, 5.5), H, W, "border")["cls"][0, 0, 0] == MASKED   # border padding clamps onto column 0
    assert tile_classes(one(254.5, 5.5), H, W)["cls"][0, 0, 0] == INTERIOR     # the east tap is column 255 == W - 1
    assert tile_classes(one(254.5, 62.5), H, W)["cls"][0, 0, 0] == INTERIOR    # the south tap is row 63 == H - 1
    assert tile_classes(one(254.5, 63.0), H, W)["cls"][0, 0, 0] == MASKED      # the south tap is row H
    assert tile_classes(one(255.0, 5.5), H, W)["cls"][0, 0, 0] == MASKED       # the east tap is column W
    nan = one(10.5, 5.5)
    nan[0, 3, 7, 1] = np.nan
    assert tile_classes(nan, H, W)["cls"][0, 0, 0] == FALLBACK
    assert tile_classes(nan, H, W, "border")["cls"][0, 0, 0] == FALLBACK
    partial = one(10.5, 5.5)[:, :, :60]                 # a partial tile never takes the mask-free body
    assert tile_classes(partial, H, W)["cls"][0, 0, 0] == MASKED
    # 84 wide: the widest channels-last box, the middle NCHW one is too narrow; 85 wide: no channels-last box
    g = patch(H, W, False, (64.25, 64 + 84 - 1.5), (8.25, 8 + 20 - 1.5))[None]
    assert (tile_classes(g, H, W)["shape"][0, 0, 0], tile_classes(g, H, W, cl=True)["shape"][0, 0, 0]) == (2, 2)
    g = patch(H, W, False, (64.25, 64 + 85 - 1.5), (8.25, 8 + 20 - 1.5))[None]
    assert tile_classes(g, H, W)["shape"][0, 0, 0] == 2 and tile_classes(g, H, W, cl=True)["cls"][0, 0, 0] == FALLBACK
    # 2 x 2 frames of smooth maps at 40 x 72 (the size of the older oracle test): no tile is interior there
    g = synth.make_map("smooth", 2, 40, 72, False, seed=4)
    assert census(tile_classes(g, 40, 72))[INTERIOR] == 0


def test_descriptor_spanning_2_31_elements_is_refused():
    # The kernels address a frame with 32-bit in-frame offsets, so one batch item may span at most 2^31 - 1 elements.  The
    # check fires on the descriptor, before any device access: no allocation is needed and the data pointer is never read.
    from pwstablenet_b200 import _lib
    lib = _lib.load()

    def desc(sizes, strides, dtype=_lib.PWS_F32):
        t = _lib.PwsTensor()
        t.data = 0x1000; t.dtype = dtype; t.device = 0
        for i in range(4):
            t.size[i], t.stride[i] = sizes[i], strides[i]
        return t

    grid = desc((1, 8, 8, 2), (128, 16, 2, 1))
    out = desc((1, 1, 8, 8), (64, 64, 8, 1))
    gout = out
    for frame in (desc((1, 1, 32768, 65536), (2 ** 31, 2 ** 31, 65536, 1)),     # 2^31 elements, dense
                  desc((1, 1, 2, 1), (2 ** 31, 2 ** 31, 2 ** 31 - 1, 1))):         # 2 elements, 2^31 apart
        rc = lib.pws_warp2d_forward(ctypes.byref(frame), ctypes.byref(grid), ctypes.byref(out), 0, 0, 0, None)
        assert rc == _lib.PWS_EUNSUPPORTED and b"2^31" in lib.pws_last_error()
        rc = lib.pws_warp2d_backward(ctypes.byref(gout), ctypes.byref(frame), ctypes.byref(grid), None, None, 0, 0, 0, None)
        assert rc == _lib.PWS_EUNSUPPORTED and b"2^31" in lib.pws_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pw():
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib
    _lib.load()
    return pw


@contextlib.contextmanager
def small_problem_elems(v):
    """pws_small_problem_elems(v) for the block: 0 sends every eligible call to the TMA kernels."""
    from pwstablenet_b200 import _lib
    prev = _lib.small_problem_elems(v)
    try:
        yield
    finally:
        _lib.small_problem_elems(prev)


def last_kernel():
    from pwstablenet_b200 import _lib
    return _lib.last_kernel()


def planar(g):
    return g.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)


DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


class Ref:
    """The oracle's answers for fp32 inputs (16-bit frames: the upcast frame and grad_output)."""

    def __init__(self, frames, grid, gout, pad, align, backward=True):
        N, C, H, W = frames.shape
        self.out = oracle.forward(frames, grid, pad, align)
        if not backward:
            return
        _, self.gg, self.gin64 = oracle.backward(gout, frames, grid, pad, align, want_f64_accum=True)
        _, _, mask, w = oracle.taps(grid, H, W, pad, align)
        valid = ((mask[..., None] >> np.arange(4)) & 1).astype(np.float64)
        wsum = (w.astype(np.float64) * valid).sum(-1)
        if pad == "border":     # the backward's clip keeps a NaN (-> -100 guard, no tap); the forward's drops it
            wsum[np.isnan(grid).any(-1)] = 0.0
        g64 = gout.astype(np.float64)
        self.checksum = float((g64 * wsum[:, None]).sum())
        self.checksum_scale = float((np.abs(g64) * wsum[:, None]).sum())


def check_forward(out, ref, dtype):
    if dtype == torch.float32:
        np.testing.assert_array_equal(out.cpu().numpy(), ref.out)
    else:   # one rounding of the fp32 result to the frame type
        assert torch.equal(out.cpu(), torch.from_numpy(ref.out).to(dtype))


def check_backward(gin, gg, ref):
    if gg is not None:
        np.testing.assert_array_equal(gg.cpu().numpy(), ref.gg)
    if gin is not None:
        gi = gin.cpu().numpy().astype(np.float64)
        assert np.abs(gi - ref.gin64).max() <= 1e-4 * max(np.abs(ref.gin64).max(), 1e-30)
        assert abs(gi.sum() - ref.checksum) <= 1e-6 * ref.checksum_scale + 1e-30


MASKS = [(True, True), (True, False), (False, True)]


def run_case(pw, frames, g, gout, pad, align, ref, fwd_kernel, bwd_kernel, masks=MASKS, aten=False):
    """forward + each output mask of the backward on the device tensors; kernels asserted, results against `ref`."""
    out = pw.warp2d_forward(frames, g, PAD[pad], align)
    assert last_kernel() == fwd_kernel
    check_forward(out, ref, frames.dtype)
    if aten:
        up = torch.ops.aten.grid_sampler_2d(frames.float(), g, 0, PAD[pad], align)
        assert torch.equal(out, up.to(frames.dtype))
    half = frames.dtype != torch.float32
    for mask in masks if bwd_kernel else ():
        acc = torch.full(frames.shape, 7.0, dtype=torch.float32, device="cuda") if (half and mask[0]) else None
        gin, gg = pw.warp2d_backward(gout, frames, g, PAD[pad], align, mask, grad_input=acc)
        assert last_kernel() == bwd_kernel, mask
        check_backward(gin if mask[0] else None, gg if mask[1] else None, ref)


def device_inputs(frames, grid, gout, dtype, layout):
    g = torch.from_numpy(grid).cuda()
    if layout == "planar":
        g = planar(g)
    f = torch.from_numpy(frames).cuda().to(dtype)
    go = torch.from_numpy(gout).cuda().to(dtype)
    # the oracle sees exactly what the kernel sees: the upcast 16-bit values
    return f, g, go, f.float().cpu().numpy(), go.float().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# B. every bwd_tma_kernel instantiation, bit-exact against the oracle
# ---------------------------------------------------------------------------------------------------------------------
FRAMES = [("f32", 1), ("f32", 3), ("f16", 3), ("bf16", 3)]


def matrix_inputs(dt, C, kind, pad, align, N=2, H=270, W=480, seed=21):
    if kind == "offframe":      # the smooth map moved 0.6 frame widths right: the tiles on the right sample nothing
        grid = synth.make_map("smooth", N, H, W, align, seed=seed)
        grid[..., 0] += F32(1.2)
    else:
        grid = synth.make_map(kind, N, H, W, align, seed=seed)
    return synth.make_frames(N, C, H, W, seed=seed + 1), grid, synth.make_gout(N, C, H, W, seed=seed + 2)


def kernels_for(dt):
    return ("fwd_tma", "bwd_tma") if dt == "f32" else ("fwd_tma_16", "bwd_tma_16")


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("dt,C", FRAMES)
def test_tma_matrix_bit_exact_at_270p(pw, dt, C, pad, align):
    # 2 map layouts x 3 output masks per case: with the 16 cases, all 96 bwd_tma_kernel instantiations
    frames, grid, gout = matrix_inputs(dt, C, "smooth", pad, align)
    H, W = frames.shape[2:]
    tc = census(tile_classes(grid, H, W, pad, align, xal=4 if dt == "f32" else 8))
    assert tc[INTERIOR] > 0 and tc[MASKED] > 0
    assert tc[INTERIOR] >= 0.6 * sum(tc.values()), tc
    fk, bk = kernels_for(dt)
    ref = None
    with small_problem_elems(0):
        for layout in ("planar", "interleaved"):
            f, g, go, f_np, go_np = device_inputs(frames, grid, gout, DTYPES[dt], layout)
            ref = ref or Ref(f_np, grid, go_np, pad, align)
            run_case(pw, f, g, go, pad, align, ref, fk, bk)


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_tma_bit_exact_at_1080p(pw, pad, align):
    # the bench's shape and map (2 x 3 x 1080 x 1920, smooth, planar): interior_strip takes ~90 % of the tiles
    frames, grid, gout = matrix_inputs("f32", 3, "smooth", pad, align, H=1080, W=1920, seed=31)
    tc = census(tile_classes(grid, 1080, 1920, pad, align))
    assert tc[MASKED] > 0 and tc[INTERIOR] >= 0.85 * sum(tc.values()), tc
    f, g, go, f_np, go_np = device_inputs(frames, grid, gout, torch.float32, "planar")
    with small_problem_elems(0):
        run_case(pw, f, g, go, pad, align, Ref(f_np, grid, go_np, pad, align), "fwd_tma", "bwd_tma")


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("kind", ["noisy", "random", "centre", "offframe"])
def test_tma_rough_maps_bit_exact_at_270p(pw, kind, pad, align):
    tcs = []
    for dt, layout in (("f32", "planar"), ("f16", "interleaved")):
        frames, grid, gout = matrix_inputs(dt, 3, kind, pad, align, seed=41)
        H, W = frames.shape[2:]
        tcs.append(census(tile_classes(grid, H, W, pad, align, xal=4 if dt == "f32" else 8)))
        f, g, go, f_np, go_np = device_inputs(frames, grid, gout, DTYPES[dt], layout)
        with small_problem_elems(0):
            run_case(pw, f, g, go, pad, align, Ref(f_np, grid, go_np, pad, align), *kernels_for(dt))
    if kind == "random":
        assert all(t[FALLBACK] > 0 for t in tcs), tcs
    if kind == "offframe":
        assert all(t[EMPTY] > 0 for t in tcs) or pad == "border", tcs   # (border padding clamps: nothing is empty)
        assert all(t[MASKED] > 0 and t[INTERIOR] > 0 for t in tcs), tcs


# ---------------------------------------------------------------------------------------------------------------------
# C. probe maps on each classification boundary, through the TMA kernels and the lean ones
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
@pytest.mark.parametrize("kind,frame", [("extents", "f32"), ("extents", "cl"), ("extents", "f16"), ("edges", "f32"),
                                        ("edges", "f16"), ("guards", "f32"), ("guards", "f16")])
def test_probes_bit_exact(pw, kind, frame, pad, align):
    grid, expect = probe_map(kind, frame, pad, align)
    check_probe_classes(grid, expect, frame, pad, align)
    N, Ho, Wo, _ = grid.shape
    C = 3
    frames = synth.make_frames(N, C, PROBE_H, PROBE_W, seed=51)
    gout = synth.make_gout(N, C, Ho, Wo, seed=52)
    dtype = torch.float16 if frame == "f16" else torch.float32
    ref = None
    for layout in ("planar", "interleaved"):
        f, g, go, f_np, go_np = device_inputs(frames, grid, gout, dtype, layout)
        ref = ref or Ref(f_np, grid, go_np, pad, align, backward=frame != "cl")
        if frame == "cl":   # the forward's channels-last boxes (the backward has no channels-last instantiation)
            cl = f.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
            with small_problem_elems(0):
                run_case(pw, cl, g, None, pad, align, ref, "fwd_tma_cl", None, aten=True)
            continue
        half = frame == "f16"
        # ATen's CUDA forward is left out of the guard probes: on them it stopped with an illegal memory access (most
        # likely at the coordinate of exactly 2^31, which passes its int-range guard and floors to a saturated int).  The
        # oracle, which restates its arithmetic on the CPU, stays the reference there.
        aten = kind != "guards"
        with small_problem_elems(0):
            run_case(pw, f, g, go, pad, align, ref, *kernels_for("f16" if half else "f32"), aten=aten)
        # the one-wave kernels at the default threshold, with their own per-warp "inside" tests
        run_case(pw, f, g, go, pad, align, ref, "fwd_lean", "bwd_lean_16" if half else "bwd_lean", aten=aten)


# ---------------------------------------------------------------------------------------------------------------------
# D. launch geometry and size limits
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_tall_output_on_the_small_problem_forward(pw):
    # 1 100 000 output rows: more than 65535 blocks of 16 rows.  The lean forward must not accept the call (its grid's
    # y dimension would be refused at launch); the direct kernel takes it and the result equals ATen's.
    Ho = 1_100_000
    rng = np.random.default_rng(61)
    for dtype, W, Wo in ((torch.float32, 4, 3), (torch.float16, 8, 8)):
        frame = torch.from_numpy(rng.random((1, 1, 4, W), dtype=np.float32) * 255).cuda().to(dtype)
        grid = torch.from_numpy((rng.random((1, Ho, Wo, 2), dtype=np.float32) * 2.2 - 1.1)).cuda().to(dtype)
        for pad in ("zeros", "border"):
            for align in (False, True):
                out = pw.warp2d_forward(frame, grid, PAD[pad], align)
                ref = torch.ops.aten.grid_sampler_2d(frame.float(), grid.float(), 0, PAD[pad], align).to(dtype)
                assert torch.equal(out, ref)
        assert last_kernel() == "fwd_direct"
        fr, gr = frame.float().cpu().numpy(), grid.float().cpu().numpy()
        check_forward(out, Ref(fr, gr, None, "border", True, backward=False), dtype)


@gpu
@pytest.mark.parametrize("W", [2 ** 22, 2 ** 22 + 4])
def test_width_at_the_floor_limit(pw, W):
    # floor_small / the backward's add.rm floor hold for coordinates below 2^22; the TMA kernels take W <= 2^22.  The map
    # samples the last ~5000 columns, where a coordinate's ulp is 0.25.
    H, Ho, Wo = 20, 32, 4992
    rng = np.random.default_rng(62)
    X = (W - 5000.0) + np.arange(Wo) * (4998.0 / Wo) + rng.random((1, Ho, Wo)) * 0.9
    Y = np.linspace(0.3, H - 1.2, Ho)[None, :, None] + rng.random((1, Ho, Wo)) * 0.5
    for align in (False, True):
        grid = np.stack([coord_to_map(X, W, align), coord_to_map(Y, H, align)], -1).astype(F32)
        for pad in ("zeros", "border"):
            tc = census(tile_classes(grid, H, W, pad, align))
            assert tc[INTERIOR] > 0 and tc[MASKED] > 0, tc
            frames = synth.make_frames(1, 1, H, W, seed=63)
            gout = synth.make_gout(1, 1, Ho, Wo, seed=64)
            f, g, go = torch.from_numpy(frames).cuda(), planar(torch.from_numpy(grid).cuda()), torch.from_numpy(gout).cuda()
            ref = Ref(frames, grid, gout, pad, align)
            kernels = ("fwd_tma", "bwd_tma") if W <= 2 ** 22 else ("fwd_lean", "bwd_lean")
            with small_problem_elems(0):
                run_case(pw, f, g, go, pad, align, ref, *kernels, masks=[(True, True)])


@gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_thin_frames_and_outputs(pw, pad, align):
    rng = np.random.default_rng(65)
    # (N, C, H, W, Ho, Wo, kernels at threshold 0 or None): one-row / one-column frames and outputs
    cases = [(2, 3, 1, 64, 16, 64, ("fwd_tma", "bwd_tma")),          # one row, still TMA-eligible
             (2, 3, 2000, 4, 40, 4, ("fwd_tma", "bwd_tma")),         # four columns, still TMA-eligible
             (2, 3, 1, 5, 16, 64, None), (2, 1, 37, 1, 16, 64, None), (2, 3, 1, 1, 8, 8, None),
             (2, 3, 48, 64, 1, 64, None), (2, 3, 48, 64, 40, 1, None), (2, 1, 48, 64, 1, 1, None)]
    for N, C, H, W, Ho, Wo, kernels in cases:
        grid = (rng.random((N, Ho, Wo, 2), dtype=np.float32) * 2.4 - 1.2).astype(F32)
        frames, gout = synth.make_frames(N, C, H, W, seed=66), synth.make_gout(N, C, Ho, Wo, seed=67)
        ref = Ref(frames, grid, gout, pad, align)
        for layout in ("planar", "interleaved"):
            f, g, go, _, _ = device_inputs(frames, grid, gout, torch.float32, layout)
            for thr in (0, None):
                with small_problem_elems(thr) if thr is not None else contextlib.nullcontext():
                    out = pw.warp2d_forward(f, g, PAD[pad], align)
                    if kernels and thr == 0:
                        assert last_kernel() == kernels[0]
                    check_forward(out, ref, torch.float32)
                    assert torch.equal(out, torch.ops.aten.grid_sampler_2d(f, g, 0, PAD[pad], align))
                    gin, gg = pw.warp2d_backward(go, f, g, PAD[pad], align, (True, True))
                    if kernels and thr == 0:
                        assert last_kernel() == kernels[1]
                    check_backward(gin, gg, ref)


@gpu
def test_more_frames_than_one_grid_z(pw):
    # 65537 frames: bwd_lean launches its frames in z-chunks of 65535; the fused entries refuse such a batch cleanly
    N, C, H, W = 65537, 1, 4, 4
    grid = synth.make_map("noisy", N, H, W, False, seed=68)
    frames, gout = synth.make_frames(N, C, H, W, seed=69), synth.make_gout(N, C, H, W, seed=70)
    ref = Ref(frames, grid, gout, "zeros", False)
    f, g, go = (torch.from_numpy(a).cuda() for a in (frames, grid, gout))
    out = pw.warp2d_forward(f, g, 0, False)
    check_forward(out, ref, torch.float32)
    gin, gg = pw.warp2d_backward(go, f, g, 0, False, (True, True))
    assert last_kernel() == "bwd_lean"
    check_backward(gin, gg, ref)
    assert float(gin[-1].abs().sum()) > 0 and float(gg[-1].abs().sum()) > 0
    with pytest.raises(RuntimeError, match="too large"):
        pw.warp_stages(f, [g])
    with pytest.raises(RuntimeError, match="too large"):
        pw.warp_fused(f, drift=g)


@gpu
def test_frame_span_just_under_2_31(pw):
    # one fp32 frame of 32764 x 65536 = 2^31 - 262144 elements (8.6 GB), read with 32-bit in-frame offsets; the map samples
    # its last rows and columns, some taps beyond them
    H, W, Ho, Wo = 32764, 65536, 32, 64
    rng = np.random.default_rng(71)
    X = (W - 45.0) + np.arange(Wo)[None, None, :] * (46.0 / Wo) + rng.random((1, Ho, Wo)) * 0.5
    Y = (H - 22.0) + np.arange(Ho)[None, :, None] * (23.0 / Ho) + rng.random((1, Ho, Wo)) * 0.5
    grid_np = np.stack([coord_to_map(X, W, False), coord_to_map(Y, H, False)], -1).astype(F32)
    frame = torch.rand((1, 1, H, W), generator=torch.Generator("cuda").manual_seed(72), device="cuda") * 255
    g = torch.from_numpy(grid_np).cuda()
    go = torch.from_numpy(synth.make_gout(1, 1, Ho, Wo, seed=73)).cuda()
    x0, y0, mask, w = pw.warp_taps(g, H, W, "zeros", False)
    valid = torch.stack([(mask >> k) & 1 for k in range(4)], dim=-1).to(torch.float64)
    expect = float((go[:, 0].double() * (w.double() * valid).sum(-1)).sum())
    ys, xs = slice(H - 24, H), slice(W - 48, W)
    ref_out = torch.ops.aten.grid_sampler_2d(frame, g, 0, 0, False)
    _, ref_gg = torch.ops.aten.grid_sampler_2d_backward(go, frame, g, 0, 0, False, [False, True])
    ref_gin, _ = torch.ops.aten.grid_sampler_2d_backward(go, frame, g, 0, 0, False, [True, False])
    ref_win = ref_gin[0, 0, ys, xs].clone()
    assert abs(float(ref_gin.double().sum()) - expect) <= 1e-6 * abs(expect)
    del ref_gin
    torch.cuda.empty_cache()
    try:
        for thr in (None, 0):
            with small_problem_elems(thr) if thr is not None else contextlib.nullcontext():
                out = pw.warp2d_forward(frame, g, 0, False)
                assert torch.equal(out, ref_out), last_kernel()
                gin, gg = pw.warp2d_backward(go, frame, g, 0, False, (True, True))
                kern = last_kernel()
                assert float((gg - ref_gg).abs().max()) <= 1e-5 * float(ref_gg.abs().max()), kern
                assert abs(float(gin.double().sum()) - expect) <= 1e-6 * abs(expect), kern
                win = gin[0, 0, ys, xs]
                assert float((win - ref_win).abs().max()) <= 1e-4 * float(ref_win.abs().max()), kern
                gin[0, 0, ys, xs] = 0
                assert float(gin.abs().max()) == 0.0, kern      # nothing lands outside the window the taps reach
                del gin, gg
    finally:
        del frame
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# the coverage table: which tiles each case and probe ran through (host-side, no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def coverage_report():
    lines = ["| case | frames | padding | align | interior | masked | fallback | empty | interior share |", "|" + "---|" * 9]

    def row(case, dt, C, pad, align, tc):
        n = sum(tc.values())
        lines.append(f"| {case} | {dt} C={C} | {pad} | {align} | {tc[INTERIOR]} | {tc[MASKED]} | {tc[FALLBACK]} | "
                     f"{tc[EMPTY]} | {tc[INTERIOR] / n:.1%} |")

    for dt, C in FRAMES:
        for pad in PAD:
            for align in (False, True):
                frames, grid, _ = matrix_inputs(dt, C, "smooth", pad, align)
                row("270p smooth (x 2 layouts x 3 masks)", dt, C, pad, align,
                    census(tile_classes(grid, 270, 480, pad, align, xal=4 if dt == "f32" else 8)))
    for pad in PAD:
        for align in (False, True):
            _, grid, _ = matrix_inputs("f32", 3, "smooth", pad, align, H=1080, W=1920, seed=31)
            row("1080p smooth, planar", "f32", 3, pad, align, census(tile_classes(grid, 1080, 1920, pad, align)))
    for kind in ("noisy", "random", "centre", "offframe"):
        for dt in ("f32", "f16"):
            for pad in PAD:
                for align in (False, True):
                    _, grid, _ = matrix_inputs(dt, 3, kind, pad, align, seed=41)
                    row(f"270p {kind}", dt, 3, pad, align, census(tile_classes(grid, 270, 480, pad, align, xal=4 if dt == "f32" else 8)))
    lines += ["", "| probe set | frames | probe | class | box shape | bw x bh |", "|" + "---|" * 6]
    for kind, frame in (("extents", "f32"), ("extents", "cl"), ("extents", "f16"), ("edges", "f32"), ("guards", "f32")):
        grid, expect = probe_map(kind, frame, "zeros", False)
        tc = check_probe_classes(grid, expect, frame, "zeros", False)
        for i, e in enumerate(expect):
            r, c = divmod(i, PROBE_TILES_X)
            box = f"{tc['bw'][0, r, c]} x {tc['bh'][0, r, c]}" if tc["shape"][0, r, c] >= 0 else "-"
            lines.append(f"| {kind} | {frame} | {e['probe']} | {tc['cls'][0, r, c]} | {tc['shape'][0, r, c]} | {box} |")
    return "\n".join(lines)


if __name__ == "__main__":
    print(coverage_report())
