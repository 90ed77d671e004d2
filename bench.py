#!/usr/bin/env python
"""Benchmark of the hot path: images/s of the 8-step CFG sample() at 32x32 latents, bs=64 per GPU.

  python bench.py --gpus N --steps K --warmup W                        (our CUDA path; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W       (the UNMODIFIED reference on the host CPU cores)
  python bench.py --impl reference-cuda --steps K --warmup W           (the UNMODIFIED reference on cuda:0, fp32 and autocast)
  python bench.py --workload {sample,sample64,vqgan} ...               (BASELINE.json configs[1] (default) / [3] / [4])

One "step" = one full pass of the workload over one batch:
  sample    BASELINE.json configs[1]: bs=64/GPU, 32x32 latents, 8 denoising steps with classifier-free guidance (16 denoiser
            sample-forwards + 8 resamples per image), the reference-default 1.008 B denoiser (SURVEY.md F1), synthetic
            ByT5/CLIP embeddings (L=128), re-randomised weights (paella_b200/synth.py)
  sample64  configs[3]: bs=16, 64x64 latents, 12 steps, + CLIP-image conditioning (unconditional side without it)
  vqgan     configs[4]: f4 VQGAN encode -> indices -> decode_indices round trip, bs=256/GPU, 256x256 images
Prints ONE JSON line (rank 0).

  --dump-outputs DIR  rank 0 writes what the timed (HBM-resident) path returned in its last timed step as float32 .npy
                      files: tokens.npy for the sample workloads, images_sample.npy + images_sample_index.npy (a fixed,
                      seeded sample of the decoded images and its flat indices) for vqgan.  Inputs and seeds depend only
                      on the arguments, so two builds run with the same arguments can be compared output for output.

  value     images/s with the inputs already resident in HBM
  e2e       images/s through the public API with HOST (pinned) inputs: H2D of the step's inputs and D2H of its result
            inside the timed region, every step
  roofline  tcgen05 GEMM family: algorithmic FLOPs of one step / summed CUDA-event durations of its launches,
            measured live by one extra profiled step after the timed region (events on the launching stream)
  cpu_baseline        the unmodified reference (baseline/_ref; oracle port if absent) on a bounded sample, rank 0, N=1 only
  torch_cuda_baseline the unmodified reference on the same GPU (fp32 w/ cuDNN TF32 default, and torch.autocast fp16)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYT5_LEN = 128
WORKLOADS = {
    "sample": dict(
        metric="images/sec @256x256-class (32x32 latent, 8192 codes), 8-step CFG sample, bs=64 per GPU",
        desc=("sample() 8-step CFG, 32x32 latents, 8192 codes, 1.008B denoiser (reference default; readme says 573M), "
              "L_byt5=128+clip, synthetic embeddings, re-randomised weights"),
        latent=32, steps=8, batch=64, clip_image=False, baseline_config=1),
    "sample64": dict(
        metric="images/sec @512x512-class (64x64 latent, 8192 codes), 12-step CFG sample with CLIP-image cond, bs=16",
        desc=("sample() 12-step CFG, 64x64 latents, 8192 codes, 1.008B denoiser, L_byt5=128+clip+clip_image (uncond without "
              "clip_image), synthetic embeddings, re-randomised weights"),
        latent=64, steps=12, batch=16, clip_image=True, baseline_config=3),
    "vqgan": dict(
        metric="images/sec VQGAN f4 encode->indices->decode round trip @256x256, bs=256 per GPU",
        desc="VQModel.encode -> indices -> decode_indices, 256x256 U[0,1) images, re-randomised f4 VQGAN (gammas, BN stats, codebook)",
        batch=256, image=256, baseline_config=4),
}
# kept as module constants for tools/ that import bench
LATENT, SAMPLE_STEPS, RENOISE, BATCH = 32, 8, 7, 64
METRIC, WORKLOAD = WORKLOADS["sample"]["metric"], WORKLOADS["sample"]["desc"]
DUMP_MAX_ELEMS = 1 << 22    # --dump-outputs: larger outputs are sampled (4 Mi float32 values + float64 indices = 48 MB)


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def host_threads():
    """CPU threads this process may really use: affinity mask capped by the cgroup CPU quota (what os.cpu_count() and
    torchrun's OMP_NUM_THREADS=1 both get wrong), and torch is told to use exactly that many."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                n = max(1, min(n, int(float(quota) / period)))
            break
        except Exception:  # noqa: BLE001
            continue
    torch.set_num_threads(n)
    return n


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def ncu_traffic():
    """DRAM bytes per launch of the dominant (GEMM) kernels from the committed `ncu --set full` capture: the
    launch-weighted mean over the main-path shapes of one forward (bench.py cannot run ncu itself)."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        try:
            ks = json.load(open(path))["kernels"]
            n = sum(k["launches_per_forward"] for k in ks)
            mean = sum(k["launches_per_forward"] * k["dram_bytes"] for k in ks) / n
            alg = sum(k["launches_per_forward"] * k["algorithmic_bytes"] for k in ks) / n
            return mean, f"profiles/{name} (launch-weighted mean of {len(ks)} shapes; algorithmic {alg / 1e6:.0f} MB)"
        except (OSError, KeyError, ValueError, ZeroDivisionError):
            continue
    return None, None


def dump_arrays(name, out):
    """--dump-outputs: one output tensor as float32 arrays, whole up to DUMP_MAX_ELEMS elements, else a fixed seeded sample
    of its flattened elements plus their flat indices (float64, exact)."""
    out = out.detach()
    if out.numel() <= DUMP_MAX_ELEMS:
        return {name: out.float().cpu().numpy()}
    idx = torch.randint(out.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
    return {f"{name}_sample": out.reshape(-1)[idx.to(out.device)].float().cpu().numpy(),
            f"{name}_sample_index": idx.double().numpy()}


def build_model(device):
    from paella_b200.modules import Paella
    from paella_b200.synth import rerandomize_
    torch.manual_seed(0)
    m = Paella(byt5_embd=2560).eval()
    rerandomize_(m.state_dict(), seed=0)
    return m.to(device)


def build_vqgan(device):
    from paella_b200.synth import rerandomize_
    from paella_b200.vqgan import VQModel
    torch.manual_seed(0)
    vq = VQModel().eval()
    rerandomize_(vq.state_dict(), seed=1)
    return vq.to(device)


# ---------------------------------------------------------------------------------------------- baseline arms
def _reference_models(workload, device):
    """The unmodified reference's modules with the same re-randomised weights as our arm (baseline/_ref)."""
    from baseline import ref_loader
    from paella_b200.synth import rerandomize_
    ref = ref_loader.load()
    torch.manual_seed(0)
    if workload == "vqgan":
        m = ref.vqgan.VQModel().eval()
        rerandomize_(m.state_dict(), seed=1)
    else:
        m = ref.modules.Paella(byt5_embd=2560).eval()
        rerandomize_(m.state_dict(), seed=0)
    return ref, m.to(device).requires_grad_(False)


def _reference_step(workload, ref, model, B, device):
    from paella_b200.synth import synthetic_conditioning
    w = WORKLOADS[workload]
    if workload == "vqgan":
        img = torch.rand(B, 3, w["image"], w["image"], generator=torch.Generator().manual_seed(5)).to(device)

        def one():
            with torch.inference_mode():
                idx = model.encode(img)[2]
                return model.decode_indices(idx)
        return one
    cond, uncond = synthetic_conditioning(B, BYT5_LEN, with_clip_image=w["clip_image"], device=device)

    def one():
        return ref.sample(model, cond, (B, w["latent"], w["latent"]), unconditional_inputs=uncond, steps=w["steps"],
                          renoise_steps=w["steps"] - 1, temperature=(1.0, 0.2), cfg=8.0, device=device)
    return one


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation on the box's host cores (all threads it can use): the
    UNMODIFIED ref/src/modules.py + ref/src/utils.py::sample from baseline/_ref (kind "reference"); if that tree did not
    travel, the oracle port (kind "port").  A step = one bounded sample of the workload: the full sample() at batch
    --ref-batch (default 1)."""
    if rank != 0:
        return
    from baseline import ref_loader
    w = WORKLOADS[args.workload]
    cores = host_threads()
    B = args.ref_batch
    if ref_loader.available():
        kind = "reference"
        ref, model = _reference_models(args.workload, "cpu")
        one = _reference_step(args.workload, ref, model, B, "cpu")
        what = "unmodified ref/src (baseline/_ref)"
    else:
        assert args.workload == "sample", "the oracle-port fallback covers the default workload only"
        kind, what = "port", "oracle port (baseline/_ref absent)"
        one = _oracle_port_step(B)
    log(f"reference arm: {what} on {cores} host threads, bs={B}")
    torch.manual_seed(1)
    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = time.perf_counter() - t0
    val = B * args.steps / dt
    sample = (f"full {w['desc'].split(',')[0]} at bs={B} (of the bs={w['batch']} workload), {what}, torch CPU fp32, {cores} threads, "
              f"torch {torch.__version__}")
    print(json.dumps({
        "impl": "reference", "metric": w["metric"], "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "batch_per_step": B},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def _oracle_port_step(B):
    from oracle import paella_oracle as po
    from paella_b200.modules import Paella
    from paella_b200.synth import rerandomize_, synthetic_conditioning
    torch.manual_seed(0)
    m = Paella(byt5_embd=2560).eval()
    rerandomize_(m.state_dict(), seed=0)
    sd = {k: v for k, v in m.state_dict().items()}
    oc = po.PaellaConfig(byt5_embd=2560)
    cond, uncond = synthetic_conditioning(B, BYT5_LEN)
    g = torch.Generator().manual_seed(1)

    def one():
        draws = {"init": torch.randint(0, 8192, (B, LATENT, LATENT), generator=g),
                 "q": [torch.empty(B * LATENT * LATENT, 8192).exponential_(1, generator=g) for _ in range(SAMPLE_STEPS)],
                 "u": [torch.rand(B, LATENT, LATENT, generator=g) for _ in range(RENOISE)]}
        with torch.inference_mode():
            return po.sample(sd, oc, cond, (B, LATENT, LATENT), uncond, steps=SAMPLE_STEPS, renoise_steps=RENOISE,
                             temperature=(1.0, 0.2), cfg_scale=8.0, draws=draws)
    return one


def reference_cuda_arm(args):
    """--impl reference-cuda: the UNMODIFIED reference (baseline/_ref) on cuda:0 through its own API, same workload, batch and
    weights as our arm — BASELINE.json north_star's "reference's own PyTorch-CUDA path".  Two stock modes:
      fp32      torch defaults (cuDNN convs may use TF32, matmuls fp32) — what `python train.py`-style code gets
      autocast  `with torch.autocast("cuda")` (fp16), as paella_inference.ipynb does (nb:349)
    Prints one JSON line; `value` is the faster mode."""
    from baseline import ref_loader
    w = WORKLOADS[args.workload]
    if not ref_loader.available():
        print(json.dumps({"impl": "reference-cuda", "unavailable": "baseline/_ref is empty (reference tree did not travel)"}), flush=True)
        return
    assert torch.cuda.is_available()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ref, model = _reference_models(args.workload, dev)
    B = args.batch or w["batch"]
    one = _reference_step(args.workload, ref, model, B, dev)
    modes = {}
    for mode in ("fp32", "autocast"):
        def run():
            if mode == "autocast":
                with torch.autocast("cuda"):
                    return one()
            return one()
        torch.manual_seed(1)
        try:
            for _ in range(max(1, args.warmup)):
                run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                run()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            modes[mode] = {"images_per_s": B / ms * 1e3, "ms_per_step": ms}
            log(f"reference-cuda {mode}: {ms:.1f} ms/step = {B / ms * 1e3:.1f} img/s")
        except Exception as e:  # noqa: BLE001 — e.g. OOM at bs=256 for the codec: report, do not die
            modes[mode] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.empty_cache()
    ok = {k: v for k, v in modes.items() if "images_per_s" in v}
    best = max(ok, key=lambda k: ok[k]["images_per_s"]) if ok else None
    print(json.dumps({
        "impl": "reference-cuda", "metric": w["metric"], "value": ok[best]["images_per_s"] if best else None, "unit": "images/s",
        "n_gpus": 1, "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": ok[best]["ms_per_step"] if best else None,
        "higher_is_better": True, "best_mode": best, "modes": modes, "data": "synthetic",
        "config": {"workload": w["desc"], "batch_per_gpu": B},
        "what": ("unmodified ref/src/modules.py + ref/src/utils.py::sample (baseline/_ref) on cuda:0, torch "
                 f"{torch.__version__}, cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}, "
                 f"matmul.allow_tf32={torch.backends.cuda.matmul.allow_tf32}")}), flush=True)


def _child_json(extra, timeout):
    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + extra, capture_output=True, text=True, timeout=timeout)
    return json.loads(r.stdout.strip().splitlines()[-1])


# ---------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default="sample", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--ref-batch", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after timing, write the last timed step's outputs to DIR as float32 .npy files "
                    "(the tokens; for vqgan a fixed, seeded sample of the images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.impl == "reference-cuda":
        if rank == 0:
            reference_cuda_arm(args)
        return

    import torch.distributed as dist
    from paella_b200 import _lib
    from paella_b200 import utils as U
    from paella_b200.synth import synthetic_conditioning
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    w = WORKLOADS[args.workload]
    B = args.batch or w["batch"]
    bsrc = 0 if world > 1 else None
    extra = {}

    if args.workload == "vqgan":
        vq = build_vqgan(dev)
        vq.pack_weights(broadcast_src=bsrc)       # the one collective: weight blob broadcast (+ checksum all-reduce)
        S = w["image"]
        img_h = torch.rand(B, 3, S, S, generator=torch.Generator().manual_seed(5 + rank)).pin_memory()
        img_d = img_h.to(dev)
        out_h = torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory()

        def step_resident():
            return vq.decode_indices(vq.encode(img_d)[2])
        dump_name = "images"

        def step_e2e():
            x = img_h.to(dev, non_blocking=True)
            out_h.copy_(vq.decode_indices_u8(vq.encode(x)[2]), non_blocking=True)
        h2d, d2h = img_h.numel() * 4, out_h.numel()
        e2e_note = "H2D fp32 images; D2H uint8 NHWC images (fused clamp(0,1)*255 writer)"
    else:
        model = build_model(dev)
        model.pack_weights(broadcast_src=bsrc)    # the one collective: weight blob broadcast (+ checksum all-reduce)
        H, steps = w["latent"], w["steps"]
        cond_h, uncond_h = synthetic_conditioning(B, BYT5_LEN, with_clip_image=w["clip_image"], seed=1234 + rank, pin=True)
        cond_d = {k: v.to(dev) for k, v in cond_h.items()}
        uncond_d = {k: v.to(dev) for k, v in uncond_h.items()}
        shape = (B, H, H)
        torch.manual_seed(1234 + rank)
        kw = dict(steps=steps, renoise_steps=steps - 1, temperature=(1.0, 0.2), cfg=8.0)

        def step_resident():
            return U.sample(model, cond_d, shape, uncond_d, **kw)
        dump_name = "tokens"

        host_tokens = torch.empty(shape, dtype=torch.int64).pin_memory()

        def step_e2e():
            c = {k: v.to(dev, non_blocking=True) for k, v in cond_h.items()}
            u = {k: v.to(dev, non_blocking=True) for k, v in uncond_h.items()}
            toks = U.sample(model, c, shape, u, **kw)
            host_tokens.copy_(toks, non_blocking=True)
            return toks
        h2d = sum(v.numel() * v.element_size() for v in list(cond_h.values()) + list(uncond_h.values()))
        d2h = host_tokens.numel() * host_tokens.element_size()
        e2e_note = "H2D byt5/clip embeddings (cond + uncond); D2H int64 tokens"
        if world > 1:
            # data-plane proof: every rank samples the SAME inputs with the SAME seed; token checksums must agree, i.e. the
            # broadcast weights and the whole kernel path are identical on every GPU (a short / failed broadcast cannot pass)
            cs, us = synthetic_conditioning(2, 16, with_clip_image=w["clip_image"], seed=99, device=dev)
            torch.manual_seed(4242)
            tk = U.sample(model, cs, (2, 16, 16), us, steps=3, renoise_steps=2)
            torch.manual_seed(1234 + rank)
            mine = (tk.view(-1) * torch.arange(1, tk.numel() + 1, device=dev)).sum().view(1)
            allc = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allc, mine)
            sums = [int(c) for c in allc]
            assert len(set(sums)) == 1, f"cross-rank token checksum mismatch (weights differ between ranks?): {sums}"
            extra["cross_rank_token_checksum"] = {"value": sums[0], "ranks_agree": world}

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms), last

    log(f"rank {rank}: weights packed; warm-up x{max(args.warmup, 3)}")
    for _ in range(max(args.warmup, 3)):
        step_resident()
    torch.cuda.synchronize()
    log(f"timing {args.steps} steps (HBM-resident inputs)")
    launches0 = L.pb200_launch_count()
    with ClockSampler(local_rank) as clk:
        ms, last = timed(step_resident, args.steps)
    launches = L.pb200_launch_count() - launches0
    dumped = dump_arrays(dump_name, last) if args.dump_outputs and rank == 0 else {}
    del last
    log(f"  {ms / args.steps:.1f} ms/step; timing {args.steps} steps end to end (host inputs)")
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    log(f"  {ms_e2e / args.steps:.1f} ms/step; profiled step")
    value = world * B * args.steps / (ms / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)

    if args.workload == "sample" and world == 1:
        # the step after the path (SURVEY.md §8 f2): sample() with the decode fused on its tail, uint8 NHWC images out
        try:
            vq = build_vqgan(dev)
            vq.pack_weights()

            def step_dec():
                return U.sample(model, cond_d, shape, uncond_d, decode=vq, **kw)
            for _ in range(2):
                step_dec()
            ms_dec, _ = timed(step_dec, args.steps)
            extra["with_decode"] = {"value": B * args.steps / (ms_dec / 1e3), "unit": "images/s", "ms_per_step": ms_dec / args.steps,
                                    "what": "sample(..., decode=vqmodel): tokens -> f4 VQGAN decode_indices -> clamp(0,1) -> uint8 NHWC, on-stream"}
        except Exception as e:  # noqa: BLE001
            extra["with_decode"] = {"error": f"{type(e).__name__}: {str(e)[:160]}"}

    # one extra profiled step: CUDA events around every launch, by kernel family
    L.pb200_profile_enable(1)
    step_resident()
    cbuf = ctypes.create_string_buffer(65536)
    _lib.check(L.pb200_profile_report(cbuf, 65536), "profile_report")
    prof = json.loads(cbuf.value.decode())
    L.pb200_profile_enable(0)
    pk = peaks()
    tensor_tags = [k for k in prof if k.startswith("gemm") or k.startswith("conv")]
    gemm_ms = sum(prof[k]["ms"] for k in tensor_tags)
    gemm_fl = sum(prof[k]["work"] for k in tensor_tags)
    gemm_n = sum(prof[k]["launches"] for k in tensor_tags)
    total_ms = sum(v["ms"] for v in prof.values())
    achieved = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic() if args.workload == "sample" else (None, None)

    def fam(k, v):
        tensor = k in tensor_tags or k == "fused_sampler"
        rate = v["work"] / (v["ms"] / 1e3) / (1e12 if tensor else 1e9) if v["ms"] > 0 else None
        peak = pk["tflops"] if tensor else pk["hbm_gbs"]
        return {"ms": round(v["ms"], 3), "launches": v["launches"], "rate": rate, "unit": "TFLOP/s" if tensor else "GB/s",
                "frac": (rate / peak if rate else None), "bound": "alu(philox)" if k == "fused_sampler" else ("tensor" if tensor else "hbm")}
    roofline = {"bound": "tensor", "kernel": "gemm_f16_cg2_kernel / gemm_f16_kernel (tcgen05 GEMM family)", "achieved": achieved,
                "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": pk["src"] + " bf16 sustained", "launches_per_step": gemm_n,
                "avg_launch_ms": gemm_ms / max(gemm_n, 1), "share_of_step": gemm_ms / total_ms if total_ms else None,
                "families": {k: fam(k, v) for k, v in prof.items()}}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {"metric": w["metric"], "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
           "data": "synthetic",
           "config": {"workload": w["desc"], "baseline_config": w["baseline_config"], "batch_per_gpu": B, "global_batch": B * world,
                      "parallelism": f"batch-shard x{world}, 1 weight broadcast",
                      "l2": "inputs larger than L2 (weights + activations per step far exceed 126 MB)"},
           "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": ms_e2e / args.steps, "copies": e2e_note},
           "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roofline}
    out.update(extra)
    if world == 1 and not args.no_cuda_baseline:
        log("torch-CUDA baseline: the unmodified reference on this GPU (child process) ...")
        try:
            out["torch_cuda_baseline"] = _child_json(["--impl", "reference-cuda", "--workload", args.workload, "--steps", "2", "--warmup", "1",
                                                      "--batch", str(B)], timeout=420)
            v = out["torch_cuda_baseline"].get("value")
            if v:
                out["torch_cuda_baseline"]["ours_over_reference_cuda"] = {"value": value / v, "e2e": e2e / v}
        except Exception as e:  # noqa: BLE001
            out["torch_cuda_baseline"] = {"value": None, "error": f"{type(e).__name__}: {str(e)[:160]}"}
    if world == 1 and not args.no_cpu_baseline:
        # in a child process with a hard limit, so the GPU line is printed whatever the host CPU does
        log("cpu baseline (the unmodified reference on the host cores, bounded to one image) ...")
        try:
            r = _child_json(["--impl", "reference", "--workload", args.workload, "--steps", "1", "--warmup", "0", "--ref-batch", "1"],
                            timeout=300)
            out["cpu_baseline"] = r["cpu_baseline"]
        except Exception as e:  # noqa: BLE001
            out["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": host_threads(), "kind": "reference",
                                   "sample": f"not measured: {type(e).__name__} (300 s limit)"}
    if dumped:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{k}.npy"), a)
        log(f"outputs of the last timed step: {', '.join(f'{k}{list(a.shape)}' for k, a in dumped.items())} -> {args.dump_outputs}")
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
