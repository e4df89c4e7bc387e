"""Generates tests/golden/*.npz from the REFERENCE itself, in the build container.

Run (CPU, ~1 min):   python tests/golden/make_golden.py

What is the reference here?  PWStableNet has no arithmetic of its own on the
warp path: R/main_new.py:106,116,197,716 call torch.nn.functional.grid_sample
and R/lib/networks_cascading.py:152-237 / R/lib/utils.py:386-403 build the
maps.  So the vectors are produced by
  * importing the reference's lib/ from /root/reference (unmodified) and running
    its random-init cascading netG (BASELINE config 1: seed 123 = opt.seed,
    R/lib/cfg.py:22; define_G(31,2,64,'normal',0.02), R/main_new.py:28 analogue),
  * the reference's generate_maps() (its `.cuda()` is patched to a no-op, the
    only change, because this container has no GPU),
  * torch's CPU grid_sample / affine_grid / Upsample called exactly as the
    reference calls them.
/root/reference does not exist on the GPU box, so only the outputs travel.
Large outputs are stored as a sha256 of their bytes plus a strided subsample.
"""
import hashlib
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.path.insert(0, os.path.dirname(HERE))
import synth  # noqa: E402


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def config1_vectors(frame, gout, maps_planar, drift3_planar, genmaps_planar):
    """config1_netg.npz from netG's outputs: maps_planar (3,2,256,256), drift3_planar / genmaps_planar (1,2,256,256),
    frame / gout (1,3,256,256) float32.  A full map is 512 KiB and does not compress, so to keep the file under 1 MB
    stages 1 and 2 keep every 8th row (each output pixel and its grad_grid depend on its own map row only) and stage 3
    is stored as drift3 + plane + ulp offsets (tests/synth.py:config1_netg_maps).  Every case is then torch's CPU
    grid_sample fwd + bwd on the map the tests rebuild."""
    import torch
    import torch.nn.functional as F

    d3 = drift3_planar[0]
    g = synth.identity_map(1, 256, 256, False, np.float64)[0].reshape(-1, 2)
    a = np.concatenate([g, np.ones((g.shape[0], 1))], 1)
    resid = maps_planar[2].astype(np.float64) - d3.astype(np.float64)
    theta = np.stack([np.linalg.lstsq(a, resid[c].ravel(), rcond=None)[0] for c in range(2)])
    ulps = maps_planar[2].view(np.int32).astype(np.int64) - synth.drift_plus_plane(d3, theta).view(np.int32)
    assert np.abs(ulps).max() < 2 ** 15
    out = {
        "frame_sha": sha(frame),
        "map_rows8": np.ascontiguousarray(maps_planar[:2, :, ::8, :]),
        "map2_theta": theta,
        "map2_ulps": ulps.astype(np.int16),
        "drift3_planar": drift3_planar,
        "genmaps_sha": sha(genmaps_planar),
        "genmaps_sub": genmaps_planar[:, :, ::8, ::8].copy(),
    }
    maps = synth.config1_netg_maps(out)
    assert np.array_equal(maps[2], maps_planar[2])
    sub = (slice(None), slice(None), slice(None, None, 8), slice(None, None, 8))
    # the three cascade maps (align_corners unset -> False on torch>=1.3) and the
    # generate_maps map under both conventions (torch 0.4 behaved as True)
    cases = [("m0", maps[0], False), ("m1", maps[1], False), ("m2", maps[2], False),
             ("gm_f", genmaps_planar[0], False), ("gm_t", genmaps_planar[0], True)]
    for name, planar, align in cases:
        # planar storage (N,2,H,W): what the reference really hands to grid_sample
        m = torch.from_numpy(planar[None]).permute(0, 2, 3, 1)
        go = torch.from_numpy(np.ascontiguousarray(gout[:, :, ::gout.shape[2] // planar.shape[1]]))  # the map's rows
        for pad in ("zeros", "border"):
            fi = torch.from_numpy(frame).requires_grad_(True)
            mi = m.clone().requires_grad_(True)
            o = F.grid_sample(fi, mi, mode="bilinear", padding_mode=pad, align_corners=align)
            o.backward(go)
            key = f"{name}_{pad}"
            out[key + "_out_sha"] = sha(o.detach().numpy())
            out[key + "_out_sub"] = o.detach().numpy()[sub].copy()
            out[key + "_gin_sub"] = fi.grad.numpy()[sub].copy()
            out[key + "_gin_sum"] = np.float64(fi.grad.double().sum().item())
            gg = mi.grad.contiguous().numpy()  # (1,H,256,2)
            out[key + "_ggrid_sub"] = gg[:, ::8, ::8, :].copy()
            out[key + "_ggrid_abssum"] = np.float64(np.abs(gg.astype(np.float64)).sum())
    return out


def main():
    only_inference = "--inference-only" in sys.argv   # regenerate inference_site.npz without touching the other files
    warnings.filterwarnings("ignore")
    sys.dont_write_bytecode = True
    sys.argv = ["x"]  # lib/cfg.py parses argv at import (R/lib/cfg.py:43)
    sys.path.insert(0, REF)
    import torch
    import torch.nn.functional as F

    torch.set_num_threads(1)  # fixed reduction order inside the conv stack
    from lib.networks_cascading import define_G
    from lib import utils as ref_utils

    # ------------------------------------------------------------------ config 1
    torch.manual_seed(123)
    netG = define_G(31, 2, 64, "normal", 0.02)
    stack = torch.rand(1, 31, 256, 256) * 2 - 1
    # frame and grad_output come from a numpy generator so that they need not be stored
    frng = np.random.default_rng(123)
    frame = torch.from_numpy((frng.random((1, 3, 256, 256), dtype=np.float32) * 255).astype(np.float32))  # (x+1)*127.5 range, R/main_new.py:106
    gout = torch.from_numpy(frng.random((1, 3, 256, 256), dtype=np.float32))
    with torch.no_grad():
        maps, drifts = netG(stack)  # train mode: 3 maps + 3 drifts, planar-stored views
    assert maps[0].stride() == (131072, 256, 1, 65536)

    # reference generate_maps on the stage-3 drift (R/main.py:104 pattern)
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        gm = ref_utils.generate_maps(drifts[2].permute(0, 3, 1, 2), 1)  # (1,2,256,256)
    finally:
        torch.Tensor.cuda = orig_cuda

    out = config1_vectors(frame.numpy(), gout.numpy(),
                          np.stack([m.permute(0, 3, 1, 2).contiguous().numpy()[0] for m in maps]),
                          drifts[2].permute(0, 3, 1, 2).contiguous().numpy(), gm.contiguous().numpy())
    if not only_inference:
        np.savez_compressed(os.path.join(HERE, "config1_netg.npz"), **out)

    # ------------------------------------------------------------------ inference site (R/main_new.py:679-684,697-721)
    # cv2-style uint8 HWC frame -> float -> permute view; netG's 256x256 map -> permute -> UpsamplingBilinear2d to the
    # frame size -> permute -> grid_sample (defaults) -> astype(uint8).  The map is the stage-3 map of the netG run
    # above (train-mode output; process() runs the same ops on the eval-mode output), once as netG emits it at random
    # init (degenerate: everything samples the centre, SURVEY 0.7) and once with the identity added (what a trained
    # theta looks like), so that the vector also covers a geometry worth testing.
    ih, iw = 144, 256
    irng = np.random.default_rng(716)
    hwc = irng.integers(0, 256, (ih, iw, 3), dtype=np.uint8)   # regenerated by the tests from the same seed
    now = torch.from_numpy(hwc.astype(np.float32))[None].permute(0, 3, 1, 2)       # :679-684
    ident = F.affine_grid(torch.tensor([[[1.0, 0, 0], [0, 1.0, 0]]]), (1, 3, 256, 256), align_corners=False)
    site = {"frame_sha": sha(hwc)}
    for name, grid in (("netg", maps[2].detach()), ("netg_plus_identity", (maps[2].detach() + ident))):
        g = grid.permute(0, 3, 1, 2)                                               # :706
        grid_resize = torch.nn.UpsamplingBilinear2d(size=(ih, iw))(g).permute(0, 2, 3, 1)   # :708-710
        fake = F.grid_sample(now, grid_resize)                                     # :716
        samples = fake[0].numpy().transpose((1, 2, 0))                             # :717-719
        site[name + "_out_u8"] = np.array(samples.astype(np.uint8))                # :721
        site[name + "_out_f32_sub"] = fake.numpy()[:, :, ::4, ::4].copy()
    np.savez_compressed(os.path.join(HERE, "inference_site.npz"), **site)
    print("inference_site.npz", os.path.getsize(os.path.join(HERE, "inference_site.npz")) // 1024, "KiB")
    if only_inference:
        return

    # ------------------------------------------------------------------ small KATs (stored in full)
    rng = np.random.default_rng(20261017)
    kat = {}
    idx = 0
    for (N, C, H, W, Ho, Wo) in [(2, 3, 13, 17, 13, 17), (1, 1, 5, 7, 9, 4), (2, 4, 8, 8, 3, 11), (1, 3, 1, 1, 2, 2)]:
        for pad in ("zeros", "border"):
            for align in (False, True):
                inp = (rng.random((N, C, H, W), dtype=np.float32) * 255).astype(np.float32)
                # coordinates well outside [-1,1], exact integers/borders, and a few specials
                g = (rng.random((N, Ho, Wo, 2), dtype=np.float32) * 2.8 - 1.4).astype(np.float32)
                g.reshape(-1)[:: 7] = np.float32(-1.0)
                g.reshape(-1)[3:: 11] = np.float32(1.0)
                g.reshape(-1)[5:: 13] = np.float32(0.0)
                go = rng.random((N, C, Ho, Wo), dtype=np.float32)
                ti = torch.from_numpy(inp).requires_grad_(True)
                tg = torch.from_numpy(g).requires_grad_(True)
                o = F.grid_sample(ti, tg, mode="bilinear", padding_mode=pad, align_corners=align)
                o.backward(torch.from_numpy(go))
                k = f"k{idx}"
                kat[k + "_meta"] = np.array([N, C, H, W, Ho, Wo, 0 if pad == "zeros" else 1, int(align)], np.int64)
                kat[k + "_in"], kat[k + "_grid"], kat[k + "_gout"] = inp, g, go
                kat[k + "_out"] = o.detach().numpy()
                kat[k + "_gin"] = ti.grad.numpy()
                kat[k + "_ggrid"] = tg.grad.numpy()
                idx += 1
    kat["count"] = np.int64(idx)
    np.savez_compressed(os.path.join(HERE, "kat_small.npz"), **kat)

    # ------------------------------------------------------------------ composition helpers
    comp = {}
    theta = torch.tensor([[[1.02, 0.03, -0.01], [-0.02, 0.97, 0.04]],
                          [[0.9, -0.1, 0.2], [0.05, 1.1, -0.3]]], dtype=torch.float32)
    comp["theta"] = theta.numpy()
    for align in (False, True):
        comp[f"affine_{int(align)}"] = F.affine_grid(theta, (2, 3, 16, 24), align_corners=align).numpy()
    small = torch.from_numpy((rng.random((1, 2, 32, 32), dtype=np.float32) * 2 - 1).astype(np.float32))
    comp["up_src"] = small.numpy()
    # R/main_new.py:708 (UpsamplingBilinear2d == align_corners=True) and R/main.py:639 (default False)
    comp["up_1"] = torch.nn.UpsamplingBilinear2d(size=(54, 96))(small).numpy()
    comp["up_0"] = torch.nn.Upsample(size=(54, 96), mode="bilinear")(small).numpy()
    np.savez_compressed(os.path.join(HERE, "composition.npz"), **comp)

    for f in ("config1_netg.npz", "kat_small.npz", "composition.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
    print("torch", torch.__version__)


if __name__ == "__main__":
    main()
