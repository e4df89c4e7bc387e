#!/usr/bin/env python
"""bench.py -- 1080p warped frames/s of the pixel-wise warp hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one resident batch of synthetic frames: forward warp + backward warp
(gradients to BOTH the frame and the map) of FRAMES 1080p fp32 RGB frames per GPU, through the C ABI of libpwswarp.so.
The timed region is exactly K steps.  For the sustained clocks and power state rather than those of a short burst, give
a K for which the region (`timed_region_s`) lasts a second or more.

--dump-outputs DIR writes what the last timed step returned (rank 0): output, grad_input and grad_grid as
DIR/<name>.npy, float32, each a sample of DUMP_ELEMS elements at flat indices drawn by torch.randint with a fixed seed.
The inputs depend only on the seeds, so two builds can be compared output for output.

  value        frames/s, whole job, inputs resident in HBM (inputs are 0.9 GB per GPU,
               larger than the 126 MB L2, so every pass streams from DRAM)
  e2e          same metric through the user-facing host API (pwstablenet_b200.HostWarpPipeline) with PINNED HOST
               buffers: H2D of frames/map/grad_output and D2H of output/grad_frame/grad_map inside the timed region
  e2e_inference  the inference site (R/main_new.py:679-684,697-721) end to end: uint8 HWC 1080p frames + the 256x256 map
               lattice up, ONE fused kernel (upsample + sample + uint8), uint8 frames down (HostInferencePipeline)
  roofline     backward kernel (bwd_tma_kernel, the dominant one): algorithmic bytes (52 B/pixel, DESIGN.md) / CUDA-event
               time of the backward call, against MEASURED_PEAKS.json; `traffic` = DRAM bytes of the same launch from the
               ncu capture recorded in profiles/traffic.json -- null when the kernel source has changed since
  aten_cuda    torch's own CUDA grid_sample fwd+bwd on the same device tensors (what the reference executes on a GPU box)
  cpu_baseline the reference's CPU path -- torch.nn.functional.grid_sample on CPU tensors exactly as
               R/main_new.py:106,116,716 call it -- timed on this box's host cores over a bounded sample
  --impl reference   times only that CPU path (rank 0), K steps after W warm-up steps, and prints the same JSON line

N > 1 (torchrun): every rank owns its own frames (frame/clip sharding, no collective on
the warp path); the timed region is bracketed by barrier + synchronize and the MAX over
ranks is taken.  scaling = weak.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

H, W, C = 1080, 1920, 3
FRAMES = 16                      # frames per GPU per step
DUMP_ELEMS = 1 << 22             # per dumped array: 3 x 16 MiB of float32
FWD_BYTES_PX, BWD_BYTES_PX = 32, 52   # algorithmic bytes per output pixel, fp32 C=3 (DESIGN.md section 4)
WORKLOAD = ("1080p (1920x1080) fp32 RGB bilinear warp, forward + backward (grad to frame and map), "
            f"{FRAMES} frames/GPU/pass, zeros padding, align_corners=False, NCHW frames, planar-stored map "
            "= identity + 0.03*tanh(low-pass noise)")


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_inputs(n_frames, seed, device):
    """Frames U(0,255), grad_output U(0,1) on the device; the map is built on the host
    from the seeded generator shared with the tests (tests/synth.py) and stored planar."""
    import synth
    g = torch.Generator(device="cpu").manual_seed(seed)
    nmap = min(n_frames, 4)
    m = torch.from_numpy(synth.make_map("smooth", nmap, H, W, False, seed=seed))
    m = m.repeat((n_frames + nmap - 1) // nmap, 1, 1, 1)[:n_frames]
    planar = m.permute(0, 3, 1, 2).contiguous()          # (N,2,H,W) storage, as netG returns it
    frames = torch.rand((n_frames, C, H, W), generator=g) * 255
    gout = torch.rand((n_frames, C, H, W), generator=g)
    if device is not None:
        frames, gout, planar = frames.to(device), gout.to(device), planar.to(device)
    return frames, planar.permute(0, 2, 3, 1), gout       # map view: strides (2HW, W, 1, HW)


def dump_outputs(path, arrays):
    """DIR/<name>.npy: float32 values of each array (in its logical index order) at DUMP_ELEMS flat indices drawn with a
    fixed seed, so the same arguments always sample the same elements."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        flat = t.detach().reshape(-1)
        idx = torch.randint(flat.numel(), (min(DUMP_ELEMS, flat.numel()),), generator=torch.Generator().manual_seed(0))
        np.save(os.path.join(path, name + ".npy"), flat[idx.to(flat.device)].float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        if os.environ.get("PWS_BENCH_NO_SMI"):
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:  # region shorter than the sampling period: take the nearest samples
            for ts, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); mx = float(f[2])
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_inputs(threads):
    """The reference arm's batch: ATen parallelises this op over the batch only (SURVEY 2.2), so the bounded sample is
    one frame per thread (= FRAMES on a 16-core box), cloned and flagged for autograd ONCE, outside any timed region."""
    frames, grid, gout = make_inputs(threads, seed=7, device=None)
    return frames.clone().requires_grad_(True), grid.clone().requires_grad_(True), gout


def cpu_reference_pass(fi, gi, gout):
    """The reference's CPU path, timed: F.grid_sample + autograd backward (R/main_new.py:106,116,197,214)."""
    import torch.nn.functional as F
    fi.grad = None
    gi.grad = None
    t0 = time.perf_counter()
    out = F.grid_sample(fi, gi, mode="bilinear", padding_mode="zeros", align_corners=False)
    out.backward(gout)
    return time.perf_counter() - t0


def host_threads():
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(cores, 32)), cores


def cpu_baseline(budget_s=20.0):
    """Bounded sample of the bench workload on the host cores (reported beside the GPU numbers, not the target)."""
    threads, cores = host_threads()
    torch.set_num_threads(threads)
    fi, gi, gout = cpu_inputs(threads)
    cpu_reference_pass(fi, gi, gout)       # warm the op
    t, spent = [], 0.0
    while len(t) < 3 and (spent < budget_s or not t):
        dt = cpu_reference_pass(fi, gi, gout)
        t.append(dt); spent += dt
    best = min(t)
    return {"value": threads / best, "unit": "frames/s", "cores": threads, "kind": "reference",
            "sample": f"torch.nn.functional.grid_sample fwd+bwd on CPU tensors (ATen CPU kernel, the op the reference's "
                      f"call sites run), batch {threads} 1080p fp32 frames, best of {len(t)} passes, "
                      f"{threads} threads of {cores} host cores; only the op is timed",
            "ms_per_pass": best * 1e3}


def shared_config(world):
    """Identical in both arms: the workload, not the implementation."""
    return {"workload": WORKLOAD, "frames_per_gpu_per_pass": FRAMES, "global_frames_per_pass": FRAMES * world,
            "sharding": f"frames split over {world} rank(s), no collective on the warp path",
            "l2": "inputs (0.9 GB/GPU) exceed the 126 MB L2; no explicit flush needed"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores, K steps after W warm-up steps;
    a step is a bounded sample of the workload (one 1080p frame per host thread); only the op is inside the timer."""
    if rank != 0:
        return
    threads, cores = host_threads()
    torch.set_num_threads(threads)
    fi, gi, gout = cpu_inputs(threads)
    for _ in range(args.warmup):
        cpu_reference_pass(fi, gi, gout)
    steps = max(1, args.steps)
    total = 0.0
    for _ in range(steps):
        total += cpu_reference_pass(fi, gi, gout)
    dt = total / steps
    value = threads / dt
    line = {
        "impl": "reference", "metric": "1080p warped frames/s (forward+backward)", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(world),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "reference",
                         "sample": f"torch CPU grid_sample fwd+bwd (the reference's call), {threads} 1080p frames per step on "
                                   f"{threads} threads of {cores} host cores, op only (inputs prepared outside the timer)"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "frames_per_step": threads,
    }
    print(json.dumps(line), flush=True)


def kernel_source_hash():
    """sha256 over the sources the backward kernel is built from: keys profiles/traffic.json."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "pwstablenet_b200", "csrc")
    for name in ("warp_bwd_tma.cu", "pws_pipe.cuh", "pws_tma.cuh", "pws_tile.cuh", "pws_common.cuh", "pws_f32x2.cuh"):
        with open(os.path.join(csrc, name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def recorded_traffic():
    """DRAM bytes per 16-frame backward launch from the ncu capture of THIS kernel source, else None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            rec = json.load(f).get("bwd_tma_kernel", {})
    except Exception:
        return None, "profiles/traffic.json missing"
    if rec.get("source_sha16") != kernel_source_hash():
        return None, f"stale: captured for kernel source {rec.get('source_sha16')}, current {kernel_source_hash()}"
    if rec.get("frames_per_launch") != FRAMES:
        return None, "captured at another launch size"
    return int(rec["dram_bytes"]), rec.get("from", "profiles/traffic.json")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="headline", choices=["headline", "train", "clip"],
                    help="headline: the BASELINE metric (default); train: BASELINE config 3 (netG training step, DDP); "
                         "clip: BASELINE config 4 (300-frame 1080p clip inference, frame-sharded)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the last timed step's output, grad_input and grad_grid to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.config != "headline" or args.impl != "ours"):
        ap.error("--dump-outputs records the headline workload of --impl ours")
    if args.config != "headline":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        if args.config == "train":
            from harness import train_step
            return train_step.run(args)
        from harness import clip_inference
        return clip_inference.run(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    import pwstablenet_b200 as pw
    from pwstablenet_b200 import _lib, numa
    _lib.load()  # fails loudly when the CUDA library is missing: there is no fallback

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # run on (and pin host buffers from) the NUMA node this rank's GPU hangs off -- before anything is allocated
    placement = numa.bind_to_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    steps = max(args.steps, 1)

    frames, grid, gout = make_inputs(FRAMES, seed=100 + rank, device=dev)
    px = FRAMES * H * W

    def one_pass():
        out = pw.warp2d_forward(frames, grid, 0, False)
        gin, ggrid = pw.warp2d_backward(gout, frames, grid, 0, False, (True, True))
        return out, gin, ggrid

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- warm-up (same allocation pattern as the timed loop)
    for _ in range(warmup):
        out, gin, ggrid = one_pass()
    barrier()

    # ---------------- a burst, for comparison with round 1's 13 ms measurement: 20 passes after the GPU has idled
    time.sleep(0.5)
    bev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(20)]
    for k in range(20):
        bev[k][0].record()
        out = pw.warp2d_forward(frames, grid, 0, False)
        bev[k][1].record()
        gin, ggrid = pw.warp2d_backward(gout, frames, grid, 0, False, (True, True))
        bev[k][2].record()
    torch.cuda.synchronize()
    burst_fwd = float(np.mean([e[0].elapsed_time(e[1]) for e in bev]))
    burst_bwd = float(np.mean([e[1].elapsed_time(e[2]) for e in bev]))
    burst_ms = bev[0][0].elapsed_time(bev[-1][2]) / 20
    time.sleep(0.25)

    # ---------------- device-resident throughput (`value`) + per-call CUDA-event split
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    l0 = _lib.launch_count()
    barrier()
    t_wall0 = time.time()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for k in range(steps):
        ev[k][0].record()
        out = pw.warp2d_forward(frames, grid, 0, False)
        ev[k][1].record()
        gin, ggrid = pw.warp2d_backward(gout, frames, grid, 0, False, (True, True))
        ev[k][2].record()
    stop.record()
    barrier()
    t_wall1 = time.time()
    launches = _lib.launch_count() - l0
    clocks = sampler.stop(t_wall0, t_wall1)
    elapsed_ms = start.elapsed_time(stop)
    fwd_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    bwd_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    del ev
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"output": out, "grad_input": gin, "grad_grid": ggrid})

    # ---------------- what the reference executes on a GPU box: ATen's CUDA kernels on the same tensors (a few passes)
    aten = None
    if rank == 0:
        fr = frames.clone().requires_grad_(True)
        gr = grid.clone().requires_grad_(True)
        ta = []
        for k in range(4):
            a0, a1, a2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            fr.grad = None; gr.grad = None
            a0.record()
            o = torch.ops.aten.grid_sampler_2d(fr, gr, 0, 0, False)
            a1.record()
            o.backward(gout)
            a2.record()
            torch.cuda.synchronize()
            if k:
                ta.append((a0.elapsed_time(a1), a1.elapsed_time(a2)))
        af, ab = float(np.mean([x[0] for x in ta])), float(np.mean([x[1] for x in ta]))
        aten = {"value": FRAMES / ((af + ab) * 1e-3), "unit": "frames/s", "fwd_ms": af, "bwd_ms": ab,
                "what": "torch.ops.aten.grid_sampler_2d + autograd backward (both gradients) on the same device tensors, "
                        "CUDA events, 3 passes after 1 warm-up; backward time includes autograd's zero-fill of grad_input"}
        del fr, gr, o
    del out, gin, ggrid
    torch.cuda.empty_cache()

    # ---------------- end to end through the public host API with pinned host buffers
    hf, hg, hgo = (t.cpu().pin_memory() for t in (frames, grid.permute(0, 3, 1, 2).contiguous(), gout))
    h_out = torch.empty_like(hf).pin_memory()
    h_gin = torch.empty_like(hf).pin_memory()
    h_gg = torch.empty_like(hg).pin_memory()
    h2d = hf.numel() * 4 + hg.numel() * 4 + hgo.numel() * 4
    d2h = h_out.numel() * 4 + h_gin.numel() * 4 + h_gg.numel() * 4
    pipe = pw.HostWarpPipeline(2, C, (H, W), device=dev, backward=True)
    e2e_steps = max(3, min(steps, 40))
    for _ in range(2):
        pipe.run(hf, hg, h_out, hgo, h_gin, h_gg)
    barrier()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    for _ in range(e2e_steps):
        pipe.run(hf, hg, h_out, hgo, h_gin, h_gg)   # returns when the results are in the host buffers
    e2.record()
    barrier()
    e2e_ms = s2.elapsed_time(e2)
    del pipe, hf, hg, hgo, h_out, h_gin, h_gg

    # ---------------- the inference site end to end: uint8 HWC frames + 256x256 lattices up, uint8 frames down
    import synth
    INF_FRAMES = 32
    g8 = torch.Generator(device="cpu").manual_seed(1000 + rank)
    h_u8 = torch.randint(0, 256, (INF_FRAMES, H, W, 3), dtype=torch.uint8, generator=g8).pin_memory()
    lat = torch.from_numpy(np.ascontiguousarray(synth.make_map("smooth", 4, 256, 256, False, seed=5 + rank).transpose(0, 3, 1, 2)))
    h_lat = lat.repeat(INF_FRAMES // 4, 1, 1, 1).contiguous().pin_memory()
    h_o8 = torch.empty_like(h_u8).pin_memory()
    ipipe = pw.HostInferencePipeline(4, (H, W), (256, 256), device=dev)
    inf_steps = max(3, min(steps, 20))
    for _ in range(2):
        ipipe.run(h_u8, h_lat, h_o8)
    barrier()
    s3, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s3.record()
    for _ in range(inf_steps):
        ipipe.run(h_u8, h_lat, h_o8)
    e3.record()
    barrier()
    inf_ms = s3.elapsed_time(e3)
    inf_h2d, inf_d2h = h_u8.numel() + h_lat.numel() * 4, h_o8.numel()

    # ---------------- max over ranks
    if world > 1:
        t = torch.tensor([elapsed_ms, e2e_ms, fwd_ms, bwd_ms, inf_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms, fwd_ms, bwd_ms, inf_ms = [float(x) for x in t.tolist()]
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())

    if rank == 0:
        peak, peak_src = peaks()
        value = world * FRAMES * steps / (elapsed_ms * 1e-3)
        bwd_gbs = BWD_BYTES_PX * px / (bwd_ms * 1e-3) / 1e9
        fwd_gbs = FWD_BYTES_PX * px / (fwd_ms * 1e-3) / 1e9
        step_gbs = (FWD_BYTES_PX + BWD_BYTES_PX) * px * steps / (elapsed_ms * 1e-3) / 1e9
        traffic, traffic_src = recorded_traffic()
        line = {
            "metric": "1080p warped frames/s (forward+backward)", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": elapsed_ms / steps,
            "ms_per_pass": elapsed_ms / steps, "timed_region_s": elapsed_ms * 1e-3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(world),
            "clocks": clocks,
            "e2e": {"value": world * FRAMES * e2e_steps / (e2e_ms * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": "pwstablenet_b200.HostWarpPipeline.run(): pinned host buffers in and out, 2-frame chunks, H2D / fwd+bwd through the C ABI / D2H overlapped on 3 streams; returns when the results are in host memory",
                    "host_placement": placement},
            "e2e_inference": {"value": world * INF_FRAMES * inf_steps / (inf_ms * 1e-3), "unit": "frames/s",
                              "h2d_bytes_per_step": inf_h2d, "d2h_bytes_per_step": inf_d2h, "steps": inf_steps, "frames_per_step": INF_FRAMES,
                              "api": "pwstablenet_b200.HostInferencePipeline.run(): uint8 HWC 1080p frames + 256x256 fp32 map lattice up, one fused kernel "
                                     "(map upsample + bilinear sample + uint8 truncation: R/main_new.py:679-684,697-721), uint8 HWC frames down"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "bwd_tma_kernel (pws_warp2d_backward)", "achieved": bwd_gbs, "peak": peak,
                         "unit": "GB/s", "frac": bwd_gbs / peak, "peak_source": peak_src,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch_set": BWD_BYTES_PX * px, "ms": bwd_ms,
                         "frac_of_8TBs_nominal": bwd_gbs / 8000.0,
                         "forward": {"achieved": fwd_gbs, "frac": fwd_gbs / peak, "ms": fwd_ms},
                         "whole_step": {"achieved": step_gbs, "frac": step_gbs / peak}},
            "aten_cuda": aten,
            "burst": {"value": world * FRAMES / (burst_ms * 1e-3), "unit": "frames/s", "fwd_ms": burst_fwd, "bwd_ms": burst_bwd, "passes": 20,
                      "what": "rank 0's first 20 passes after 0.5 s of idle (SM clock at its maximum): what a ~13 ms timed region "
                              "measures; `value` above is the sustained figure (>= 1 s, under the power cap the kernel runs into)"},
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
