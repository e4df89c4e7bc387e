"""Per-call times of `pw.warp_stages` with half-precision frames and maps, at the reference's training shape
(16 x 3 x 256 x 256, three cascade maps; the working set is L2-resident, as it is in training).

    python tools/stages_half_bench.py [--iters 200] [--repeats 3] [--out DIR]

For f16 and bf16 frames, each with fp32 maps and with maps of the frame's type (planar, as netG stores them), and the
`(x+1)*127.5 ... /127.5-1` scales of R/main_new.py:103-110:
  * warp_stages forward, and forward + backward through autograd (grad -> every map);
  * the unfused 16-bit sequence it replaces (three pw.grid_sample calls with torch's elementwise ops around them),
    forward and forward + backward;
  * fp32 warp_stages on the same values, for scale.
A time is CUDA events around `iters` back-to-back calls divided by `iters` (the calls are host-bound at this size, so this
is the rate a training loop sees); each table is measured `repeats` times with the arms interleaved and reported as
min-max.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PRE, POST = (1.0, 127.5), (127.5, -1.0)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else torch.cuda.get_device_name()


def per_call_ms(fn, iters, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3, help="every table is measured this many times, arms interleaved")
    ap.add_argument("--out", default=None, help="directory for stages_half_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("stages_half_bench.py needs a CUDA device")

    import numpy as np
    import synth
    import pwstablenet_b200 as pw
    N, C, H, W = 16, 3, 256, 256
    base = synth.make_map("smooth", N, H, W, False, seed=3)
    rng = np.random.default_rng(103)
    maps32 = []
    for i in range(3):   # three maps that refine each other, stored planar
        m = torch.from_numpy((base + rng.standard_normal(base.shape).astype(np.float32) * (0.004 * i)).astype(np.float32)).cuda()
        maps32.append(m.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1))
    frame32 = torch.from_numpy(synth.make_frames(N, C, H, W, seed=4)).cuda() / 127.5 - 1
    gouts32 = [torch.from_numpy(synth.make_gout(N, C, H, W, seed=5 + k)).cuda() for k in range(3)]

    def fused(frame, maps):
        return pw.warp_stages(frame, maps, "zeros", False, pre=PRE, post=POST)

    def unfused(frame, maps):
        x = (frame + PRE[0]) * PRE[1]
        return [pw.grid_sample(x, g, "bilinear", "zeros", False) / POST[0] + POST[1] for g in maps]

    def fwd_bwd(fn, frame, maps, gouts):
        gs = [g.detach().requires_grad_(True) for g in maps]
        torch.autograd.backward(list(fn(frame, gs)), gouts)

    rows = []
    for dtype in (torch.float16, torch.bfloat16):
        frame = frame32.to(dtype)
        gouts = [g.to(dtype) for g in gouts32]
        for map_kind in ("fp32", "same"):
            maps = maps32 if map_kind == "fp32" else [m.to(dtype) for m in maps32]
            arms = {
                "warp_stages": {
                    "forward": lambda: fused(frame, maps),
                    "forward_backward": lambda: fwd_bwd(fused, frame, maps, gouts),
                },
                "unfused_16bit": {
                    "forward": lambda: unfused(frame, maps),
                    "forward_backward": lambda: fwd_bwd(unfused, frame, maps, gouts),
                },
                "warp_stages_fp32": {
                    "forward": lambda: fused(frame32, maps32),
                    "forward_backward": lambda: fwd_bwd(fused, frame32, maps32, gouts32),
                },
            }
            times = {arm: {op: [] for op in ops} for arm, ops in arms.items()}
            for _ in range(args.repeats):
                for op in ("forward", "forward_backward"):
                    for arm, ops in arms.items():
                        times[arm][op].append(per_call_ms(ops[op], args.iters))
            for arm in arms:
                for op in ("forward", "forward_backward"):
                    t = sorted(times[arm][op])
                    rows.append({"shape": [N, C, H, W], "dtype": str(dtype).replace("torch.", ""), "maps": map_kind, "arm": arm,
                                 "op": op, "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4)})
    res = {"gpu": gpu_info(), "iters": args.iters, "repeats": args.repeats, "rows": rows}
    print(f"GPU (name, power limit, max SM clock): {res['gpu']}")
    print(f"{'dtype':>9} {'maps':>5} {'op':>17} {'warp_stages':>15} {'unfused 16-bit':>15} {'fp32 warp_stages':>17}  "
          f"(ms per call, min-max; {N}x{C}x{H}x{W}, 3 maps)")
    table = {}
    for r in rows:
        table.setdefault((r["dtype"], r["maps"], r["op"]), {})[r["arm"]] = f"{r['ms_min']:.4f}-{r['ms_max']:.4f}"
    for (dt, mk, op), a in table.items():
        print(f"{dt:>9} {mk:>5} {op:>17} {a['warp_stages']:>15} {a['unfused_16bit']:>15} {a['warp_stages_fp32']:>17}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "stages_half_bench.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
