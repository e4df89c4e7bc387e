"""Forward + backward of the fused map composition at the inference-site geometry, against the unfused sequence.

Workload: 16 x 1080p frames, C = 3, a 256^2 planar lattice (netG's drift, permuted) + affine base, aligned bilinear
upsample to the frame (R/main_new.py:706-710), the loss gradient flowing back to the lattice and theta, and optionally to
the frame:
    (a) fused:           pw.warp_fused(frame, drift, base="affine", theta, upsample="aligned") -> one forward kernel, one
                         backward kernel (+ theta's reduction)
    (b) unfused, pw:     affine_grid + drift, F.interpolate, pw.grid_sample and their autograd
    (c) unfused, ATen:   the same sequence with torch's own grid_sample
Cases: uint8 frames (grad -> lattice/theta), f32 frames (grad -> lattice/theta), f32 frames with grad -> frame as well.
Each mode is timed with CUDA events over a warmed region of at least --seconds, modes alternating, --rounds times (the
median is reported).  The fused gradients are checked against (c) in the same run, with (c) sampling at the fused
kernel's map (its gradient path unchanged) and at its own map.

Bytes model of the fused pair, per output pixel: forward taps C*s_in + out C*4, backward gout C*4 + taps C*s_in (+ gin
4*C when the frame gradient is wanted), plus the lattice and its gradient.  The working set (~0.4 GB of f32 frames per
tensor) is several times the 126 MB L2.

    python tools/fused_backward_bench.py [--n 16] [--seconds 1.0] [--rounds 3] [--json out.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pwstablenet_b200 as pw  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        lim = r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        lim = "unknown"
    return name, lim


def make(n, H, W, h, w, frame_u8, want_frame, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if frame_u8:
        frame = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, device="cuda", generator=g).permute(0, 3, 1, 2)
    else:
        frame = (torch.rand(n, 3, H, W, device="cuda", generator=g) * 255).requires_grad_(want_frame)
    planar = (torch.tanh(torch.randn(n, 2, h, w, device="cuda", generator=g)) * 0.02).requires_grad_(True)
    theta = (torch.tensor([[1.0, 0.01, 0.0], [-0.01, 1.0, 0.0]], device="cuda").repeat(n, 1, 1) +
             torch.randn(n, 2, 3, device="cuda", generator=g) * 0.005).requires_grad_(True)
    gout = torch.randn(n, 3, H, W, device="cuda", generator=g)
    return frame, planar, theta, gout


def run(mode, frame, planar, theta, gout, pin=None):
    n, _, H, W = gout.shape
    drift = planar.permute(0, 2, 3, 1)
    if mode == "fused":
        out = pw.warp_fused(frame, drift=drift, base="affine", theta=theta, upsample="aligned", out_size=(H, W))
    else:
        x = frame.float() if frame.dtype == torch.uint8 else frame           # the reference's `now = hwc.float()`
        h, w = planar.shape[2], planar.shape[3]
        lat = drift + F.affine_grid(theta, (n, 3, h, w), align_corners=False)
        grid = F.interpolate(lat.permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
        if pin is not None:   # sample at the fused kernel's map, keep the sequence's gradient path
            grid = grid + (pin - grid).detach()
        sample = pw.grid_sample if mode == "unfused_pw" else F.grid_sample
        out = sample(x, grid, mode="bilinear", padding_mode="zeros", align_corners=False)
    out.backward(gout)


def grads(mode, frame, planar, theta, gout, pin=None):
    for t in (frame, planar, theta):
        if t.grad is not None:
            t.grad = None
    run(mode, frame, planar, theta, gout, pin)
    return [t.grad.clone() if t.grad is not None else None for t in (frame, planar, theta)]


def time_mode(mode, args, seconds):
    for _ in range(3):
        run(mode, *args)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); run(mode, *args); e.record(); e.synchronize()
    iters = max(5, int(seconds * 1e3 / max(s.elapsed_time(e), 1e-3)) + 1)
    s.record()
    for _ in range(iters):
        run(mode, *args)
    e.record(); e.synchronize()
    return s.elapsed_time(e) / iters, iters


def rel(a, b):
    if a is None or b is None:
        return None
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--lattice", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fused_backward_bench: needs a CUDA device (no CPU timing)")
    name, lim = card()
    print(f"device: {name}; power.limit, clocks.max.sm: {lim}")
    n, H, W, L = a.n, a.height, a.width, a.lattice
    results = []
    for case, u8, want_frame in (("u8 frames, grad -> lattice/theta", True, False),
                                 ("f32 frames, grad -> lattice/theta", False, False),
                                 ("f32 frames, grad -> frame/lattice/theta", False, True)):
        args = make(n, H, W, L, L, u8, want_frame)
        frame, planar, theta, gout = args
        pin = pw.compose_map(n, (H, W), planar.detach().permute(0, 2, 3, 1), "affine", theta.detach(), False, "aligned")
        ref = grads("unfused_aten", *args, pin=pin)
        fz = grads("fused", *args)
        errs = {"frame": rel(fz[0], ref[0]), "drift": rel(fz[1], ref[1]), "theta": rel(fz[2], ref[2])}
        # torch composes the map a few ulp away from the fused one; on white-noise frames that moves some taps across
        # a cell boundary, whose gradient differs by O(1): reported, not a parity measure
        ref_free = grads("unfused_aten", *args)
        errs_free = {"drift": rel(fz[1], ref_free[1]), "theta": rel(fz[2], ref_free[2])}
        del pin, ref_free
        s_in = 1 if u8 else 4
        px = n * H * W
        model = px * (3 * s_in + 3 * 4) + px * (3 * 4 + 3 * s_in + (4 * 3 if want_frame else 0)) + 2 * n * L * L * 2 * 4
        times = {m: [] for m in ("fused", "unfused_pw", "unfused_aten")}
        for _ in range(a.rounds):
            for m in times:
                times[m].append(time_mode(m, args, a.seconds)[0])
        med = {m: sorted(v)[len(v) // 2] for m, v in times.items()}
        row = dict(case=case, n=n, H=H, W=W, lattice=L, ms=med, all_ms=times, grad_rel_err_vs_aten_at_fused_map=errs,
                   grad_rel_err_vs_aten_own_map=errs_free,
                   fused_model_bytes=model, fused_model_GBps=model / (med["fused"] * 1e-3) / 1e9,
                   speedup_vs_pw=med["unfused_pw"] / med["fused"], speedup_vs_aten=med["unfused_aten"] / med["fused"])
        results.append(row)
        print(f"{case}: fused {med['fused']:.3f} ms, unfused+pw {med['unfused_pw']:.3f} ms, unfused+aten "
              f"{med['unfused_aten']:.3f} ms (x{row['speedup_vs_pw']:.2f}, x{row['speedup_vs_aten']:.2f}); "
              f"fused bytes model {model / 1e9:.3f} GB -> {row['fused_model_GBps']:.0f} GB/s; "
              f"grad rel err vs (c) at the fused map {errs}, at torch's own map {errs_free}")
        del args, ref, fz
        torch.cuda.empty_cache()
    out = dict(device=name, power_limit_and_max_sm_clock=lim, results=results)
    print(json.dumps(out))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
