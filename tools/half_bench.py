"""Per-call times of the 16-bit warp: f16 / bf16 frames with maps of the same 16-bit type, against ATen's native 16-bit
kernels on the same tensors and against this library with fp32 maps (the same frames, the map upcast).

    python tools/half_bench.py [--iters 200] [--out DIR]

For each shape (the reference's training call 16 x 3 x 256 x 256, and 2 x 3 x 720 x 1280) and dtype, with a smooth
near-identity map stored planar as netG stores it: forward, backward with both gradients, backward grad -> map only.
A time is CUDA events around `iters` back-to-back calls divided by `iters`, so a host-bound call (the 256^2 shapes are)
is measured at its host rate, as a training loop sees it.  This library is called through its compiled shim
(pwstablenet_b200._pws_torch, what pw.grid_sample uses).  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


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
    ap.add_argument("--repeats", type=int, default=3, help="the whole table is measured this many times, arms interleaved")
    ap.add_argument("--out", default=None, help="directory for half_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("half_bench.py needs a CUDA device")

    import synth
    from pwstablenet_b200 import functional
    ext = functional.torch_ext()
    if not ext:
        sys.exit("half_bench.py: the compiled shim _pws_torch.so is not built (run __graft_entry__.build())")
    aten = torch.ops.aten
    rows = []
    for (N, C, H, W) in [(16, 3, 256, 256), (2, 3, 720, 1280)]:
        g32 = torch.from_numpy(synth.make_map("smooth", N, H, W, False, seed=3)).cuda()
        g32 = g32.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
        for dtype in (torch.float16, torch.bfloat16):
            f = torch.from_numpy(synth.make_frames(N, C, H, W, seed=4)).cuda().to(dtype)
            go = torch.from_numpy(synth.make_gout(N, C, H, W, seed=5)).cuda().to(dtype)
            g16 = g32.to(dtype)
            arms = {
                "aten_native_16bit": {
                    "forward": lambda: aten.grid_sampler_2d(f, g16, 0, 0, False),
                    "backward_both": lambda: aten.grid_sampler_2d_backward(go, f, g16, 0, 0, False, [True, True]),
                    "backward_map_only": lambda: aten.grid_sampler_2d_backward(go, f, g16, 0, 0, False, [False, True]),
                },
                "pw_16bit_map": {
                    "forward": lambda: ext.warp2d_forward(f, g16, 0, False),
                    "backward_both": lambda: ext.warp2d_backward(go, f, g16, 0, False, True, True),
                    "backward_map_only": lambda: ext.warp2d_backward(go, f, g16, 0, False, False, True),
                },
                "pw_fp32_map": {
                    "forward": lambda: ext.warp2d_forward(f, g32, 0, False),
                    "backward_both": lambda: ext.warp2d_backward(go, f, g32, 0, False, True, True),
                    "backward_map_only": lambda: ext.warp2d_backward(go, f, g32, 0, False, False, True),
                },
            }
            times = {arm: {op: [] for op in ops} for arm, ops in arms.items()}
            for _ in range(args.repeats):
                for op in ("forward", "backward_both", "backward_map_only"):
                    for arm, ops in arms.items():
                        times[arm][op].append(per_call_ms(ops[op], args.iters))
            for arm in arms:
                for op in ("forward", "backward_both", "backward_map_only"):
                    t = sorted(times[arm][op])
                    rows.append({"shape": [N, C, H, W], "dtype": str(dtype).replace("torch.", ""), "arm": arm, "op": op,
                                 "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4)})
    res = {"gpu": gpu_info(), "iters": args.iters, "repeats": args.repeats, "rows": rows}
    print(f"GPU (name, power limit, max SM clock): {res['gpu']}")
    print(f"{'shape':>18} {'dtype':>9} {'op':>18} {'ATen native 16-bit':>20} {'pw, 16-bit map':>16} {'pw, fp32 map':>14}  (ms per call, min-max)")
    key = lambda r: (tuple(r["shape"]), r["dtype"], r["op"])
    table = {}
    for r in rows:
        table.setdefault(key(r), {})[r["arm"]] = f"{r['ms_min']:.4f}-{r['ms_max']:.4f}"
    for (shape, dt, op), arms_ in table.items():
        print(f"{'x'.join(map(str, shape)):>18} {dt:>9} {op:>18} {arms_['aten_native_16bit']:>20} {arms_['pw_16bit_map']:>16} "
              f"{arms_['pw_fp32_map']:>14}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "half_bench.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
