#!/usr/bin/env python
"""Masked sampling (inpainting / outpainting) on one GPU, against plain sample() on the headline model:
   bs 64, 32x32 latents, 8-step CFG (cfg 8, T 1.0 -> 0.2, as bench.py's sample workload).
Per workload: ms per call and images/s (CUDA events, profiler off), then the fused_sampler ms per step from one profiled call
(pb200_profile_*), and the needed-slot fraction of the mask (the share of the shared-Philox sampler's work that remains).
Also decode_composite vs decode_indices_u8 at bs 64 (32x32 tokens -> 128x128 px) and an outpaint of a 32x32 latent image on a
32x64 latent canvas.  Records the card's name and power limit in the same run.  Prints one JSON object; --out writes it too."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from paella_b200 import _lib  # noqa: E402
from paella_b200 import utils as U  # noqa: E402
from paella_b200.synth import synthetic_conditioning  # noqa: E402


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def profiled(fn):
    """One call with CUDA events around every library launch: {kernel family: ms}."""
    L = _lib.lib()
    torch.cuda.synchronize()
    L.pb200_profile_enable(1)
    fn()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(65536)
    _lib.check(L.pb200_profile_report(buf, 65536), "profile_report")
    L.pb200_profile_enable(0)
    return {k: v["ms"] for k, v in json.loads(buf.value.decode()).items()}


def slot_fraction(mask, num_labels):
    """Share of the shared-Philox sampler's slots (4 rows sharing one Philox call per label) with a masked row."""
    sm, thr = ctypes.c_int(), ctypes.c_int()
    _lib.check(_lib.lib().pb200_device_info(ctypes.byref(sm), ctypes.byref(thr)), "device_info")
    R = mask.numel()
    grid = min((R * num_labels + 255) // 256, sm.value * (thr.value // 256))
    rs = 256 * grid // num_labels
    n_blocks = (R + 4 * rs - 1) // (4 * rs)
    m = torch.zeros(n_blocks * 4 * rs, dtype=torch.bool)
    m[:R] = mask.reshape(-1).cpu()
    return float(m.view(n_blocks, 4, rs).any(dim=1).float().mean())


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    model = bench.build_model(dev)
    model.pack_weights()
    B, H, steps = bench.BATCH, bench.LATENT, bench.SAMPLE_STEPS
    K = model.num_labels
    cond, uncond = synthetic_conditioning(B, bench.BYT5_LEN, device=dev)
    known = torch.randint(0, K, (B, H, H), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    masks = {"ones": torch.ones(H, H, dtype=torch.bool)}
    c = torch.zeros(H, H, dtype=torch.bool)
    c[8:24, 8:24] = True
    masks["centre16"] = c
    lh = torch.zeros(H, H, dtype=torch.bool)
    lh[:, :H // 2] = True
    masks["left_half"] = lh
    c8 = torch.zeros(H, H, dtype=torch.bool)
    c8[12:20, 12:20] = True
    masks["centre8"] = c8
    kw = dict(steps=steps, renoise_steps=steps - 1, temperature=(1.0, 0.2))
    res = {"card": card(), "workload": f"bs {B}, {H}x{H} latents, {steps}-step CFG 8, T 1.0->0.2", "sample": {}}

    def run(name, fn, extra):
        ms = timed(fn, 1, args.iters)
        prof = profiled(fn)
        res["sample"][name] = dict(extra, ms_per_call=ms, images_per_s=B / ms * 1e3,
                                   fused_sampler_ms_per_step=prof.get("fused_sampler", 0.0) / steps)
        print(json.dumps({name: res["sample"][name]}), flush=True)

    run("plain_sample", lambda: U.sample(model, cond, (B, H, H), uncond, cfg=8.0, **kw), {"token_fraction": 1.0, "slot_fraction": 1.0})
    for name, mk in masks.items():
        mk_d = mk.to(dev)
        run(f"mask_{name}", lambda: U.sample_masked(model, cond, known, mk_d, uncond, cfg=(8.0, 8.0), **kw),
            {"token_fraction": float(mk.float().mean()), "slot_fraction": slot_fraction(mk.expand(B, H, H), K)})

    # outpaint: a 32x32 latent image in the middle of a 32x64 latent canvas (2^30-element draw: two sampler kernels per step)
    CW = 2 * H
    known_o = torch.randint(0, K, (B, H, CW), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    mo = torch.ones(H, CW, dtype=torch.bool)
    mo[:, H // 2:H // 2 + H] = False
    mo_d = mo.to(dev)
    run("outpaint_32x32_to_32x64", lambda: U.sample_masked(model, cond, known_o, mo_d, uncond, cfg=(8.0, 8.0), **kw),
        {"token_fraction": float(mo.float().mean()), "slot_fraction": slot_fraction(mo.expand(B, H, CW), K)})
    run("plain_sample_32x64", lambda: U.sample(model, cond, (B, H, CW), uncond, cfg=8.0, **kw), {"token_fraction": 1.0, "slot_fraction": 1.0})

    vq = bench.build_vqgan(dev)
    vq.pack_weights()
    idx = torch.randint(0, K, (B, H, H), device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    orig = torch.rand(B, 3, 4 * H, 4 * H, device=dev, generator=torch.Generator(device=dev).manual_seed(4))
    pm = torch.zeros(4 * H, 4 * H, dtype=torch.bool, device=dev)
    pm[32:96, 32:96] = True
    ms_u8 = timed(lambda: vq.decode_indices_u8(idx), 2, 10)
    ms_cmp = timed(lambda: vq.decode_composite(idx, orig, pm, "uint8"), 2, 10)
    out_u8, out_cmp = profiled(lambda: vq.decode_indices_u8(idx)), profiled(lambda: vq.decode_composite(idx, orig, pm, "uint8"))
    res["decode"] = {"what": f"bs {B}, {H}x{H} tokens -> {4 * H}x{4 * H} px uint8 NHWC",
                     "decode_indices_u8_ms": ms_u8, "decode_composite_ms": ms_cmp,
                     "vq_out_block_ms": {"decode_indices_u8": out_u8.get("vq_out_block"), "decode_composite": out_cmp.get("vq_out_block")}}
    print(json.dumps({"decode": res["decode"]}), flush=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
