"""Seeded synthetic inputs shared by tests/ and bench.py (SURVEY.md 8(d))."""
import numpy as np


def identity_map(N, H, W, align_corners, dtype=np.float32):
    """Identity sampling map (N,H,W,2) in the given align_corners convention."""
    if align_corners:
        xs = np.linspace(-1.0, 1.0, W, dtype=np.float64) if W > 1 else np.zeros(1)
        ys = np.linspace(-1.0, 1.0, H, dtype=np.float64) if H > 1 else np.zeros(1)
    else:
        xs = (np.arange(W, dtype=np.float64) * 2 + 1) / W - 1
        ys = (np.arange(H, dtype=np.float64) * 2 + 1) / H - 1
    g = np.empty((N, H, W, 2), dtype)
    g[..., 0] = xs[None, None, :]
    g[..., 1] = ys[None, :, None]
    return g


def smooth_drift(N, H, W, rng, amp=0.03, ncell=8):
    """amp * tanh(low-pass noise): mimics netG's +-0.035 drift (SURVEY 0.7).  The noise
    lives on an (ncell+1)^2 control lattice spanning the frame and is bilinearly
    interpolated, so the local stretch is amp*ncell/2 of a pixel per pixel at most
    (12 % for the defaults) whatever the resolution -- a stabilisation warp, not noise."""
    gh = gw = ncell + 1
    coarse = rng.standard_normal((N, gh, gw, 2))
    ys = np.linspace(0, gh - 1.001, H)
    xs = np.linspace(0, gw - 1.001, W)
    y0 = ys.astype(int); x0 = xs.astype(int)
    fy = (ys - y0)[None, :, None, None]; fx = (xs - x0)[None, None, :, None]
    c = coarse
    top = c[:, y0][:, :, x0] * (1 - fx) + c[:, y0][:, :, x0 + 1] * fx
    bot = c[:, y0 + 1][:, :, x0] * (1 - fx) + c[:, y0 + 1][:, :, x0 + 1] * fx
    return (amp * np.tanh(top * (1 - fy) + bot * fy)).astype(np.float32)


def make_map(kind, N, H, W, align_corners, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "smooth":      # realistic: identity + smooth +-0.03 drift
        return (identity_map(N, H, W, align_corners) + smooth_drift(N, H, W, rng)).astype(np.float32)
    if kind == "identity":
        return identity_map(N, H, W, align_corners)
    if kind == "random":      # stress: uniform random gather, ~31% with an out-of-range coordinate
        return (rng.random((N, H, W, 2), dtype=np.float32) * 2.4 - 1.2).astype(np.float32)
    if kind == "centre":      # degenerate random-init main_new maps: everything near the centre
        return ((rng.random((N, H, W, 2), dtype=np.float32) - 0.5) * 0.06).astype(np.float32)
    if kind == "noisy":       # identity + per-pixel noise of a few pixels
        return (identity_map(N, H, W, align_corners) + (rng.random((N, H, W, 2), dtype=np.float32) - 0.5) * 0.05).astype(np.float32)
    raise ValueError(kind)


def drift_plus_plane(drift, theta):
    """float32(drift + theta[c] . (x, y, 1)) for a planar drift (2,H,W) and a (2,3) float64 plane, x / y at the pixel
    centres (align_corners=False); evaluated in float64 and rounded once, so it is the same on every host."""
    g = identity_map(1, drift.shape[1], drift.shape[2], False, np.float64)[0]
    plane = theta[:, 0, None, None] * g[None, ..., 0] + theta[:, 1, None, None] * g[None, ..., 1] + theta[:, 2, None, None]
    return (drift.astype(np.float64) + plane).astype(np.float32)


def config1_netg_maps(z):
    """The reference netG's three cascade maps stored in tests/golden/config1_netg.npz, planar (2,H,W): stages 1 and 2
    as every 8th row (map_rows8), stage 3 in full.  Stage 3 is drift3 + F.affine_grid(theta) in netG, so it is stored
    as drift3, the least-squares plane of map - drift3 and each element's offset in ulps from drift_plus_plane: exact."""
    pred = drift_plus_plane(z["drift3_planar"][0], z["map2_theta"])
    m2 = (pred.view(np.int32) + z["map2_ulps"].astype(np.int32)).view(np.float32)
    return [z["map_rows8"][0], z["map_rows8"][1], m2]


def make_frames(N, C, H, W, seed=0):
    rng = np.random.default_rng(seed + 1000)
    return (rng.random((N, C, H, W), dtype=np.float32) * 255).astype(np.float32)


def make_gout(N, C, H, W, seed=0):
    rng = np.random.default_rng(seed + 2000)
    return rng.random((N, C, H, W), dtype=np.float32)
