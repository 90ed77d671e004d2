#!/usr/bin/env python
"""Generate the committed golden fixtures by running the REAL reference on CPU.

Needs a checkout of the original dome272/Paella, named by PAELLA_REFERENCE:
    PAELLA_REFERENCE=<checkout> python tests/golden/make_golden.py
It imports ref/src/modules.py, ref/utils/modules.py, ref/utils/alter_attention.py,
ref/src/vqgan.py and ref/src/utils.py UNMODIFIED.  ``torchtools`` (third-party,
absent) is stubbed only so those files import; the stub's quantiser is our
restatement (oracle/vqgan_oracle.py) and is NOT what these fixtures pin — the
fixtures record the conv stacks' pre-quantisation latents and decoder outputs.

Outputs (small, committed):  tests/golden/paella_tiny.npz, vqgan_tiny.npz, sample_tiny.npz, reference_default.npz
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("PAELLA_REFERENCE", "")
sys.path.insert(0, ROOT)

from oracle import vqgan_oracle as vo          # noqa: E402
from paella_b200.synth import rerandomize_, synthetic_conditioning     # noqa: E402

TINY = dict(c_in=16, c_out=16, num_labels=64, c_r=64, patch_size=2, c_cond=32, c_hidden=[32, 64, 64],
            nhead=[-1, 4, 4], blocks=[1, 2, 1], level_config=["CT", "CTA", "CTA"], clip_embd=24,
            byt5_embd=40, clip_seq_len=4, kernel_size=3, dropout=0.1, self_attn=True)
TINY_VQ = dict(levels=2, bottleneck_blocks=2, c_hidden=32, c_latent=4, codebook_size=64)


def install_torchtools_stub():
    class VectorQuantize(nn.Module):
        def __init__(self, embedding_size, k, ema_decay=0.99, ema_loss=False):
            super().__init__()
            self.codebook = nn.Embedding(k, embedding_size)
            self.codebook.weight.data.uniform_(-1. / k, 1. / k)

        def forward(self, x, get_losses=True, dim=-1):
            return vo.vq_forward(x, self.codebook.weight.data, dim)

        def idx2vq(self, idx, dim=-1):
            return vo.idx2vq(idx, self.codebook.weight.data, dim)

    tt = types.ModuleType("torchtools")
    ttnn = types.ModuleType("torchtools.nn")
    ttnn.VectorQuantize = VectorQuantize
    tt.nn = ttnn
    sys.modules["torchtools"] = tt
    sys.modules["torchtools.nn"] = ttnn


def load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    if not os.path.isdir(os.path.join(REF, "src")):
        raise SystemExit("set PAELLA_REFERENCE to a checkout of dome272/Paella")
    install_torchtools_stub()
    ref_modules = load_by_path("ref_src_modules", os.path.join(REF, "src", "modules.py"))
    ref_nb_modules = load_by_path("ref_utils_modules", os.path.join(REF, "utils", "modules.py"))
    ref_alter = load_by_path("ref_alter_attention", os.path.join(REF, "utils", "alter_attention.py"))
    ref_vqgan = load_by_path("vqgan", os.path.join(REF, "src", "vqgan.py"))     # src/utils.py does `from vqgan import VQModel`
    try:
        ref_utils = load_by_path("ref_src_utils", os.path.join(REF, "src", "utils.py"))
    except Exception as e:  # torchvision / transformers import trouble: fall back to the function source
        src = open(os.path.join(REF, "src", "utils.py")).read()
        fn = src[src.index("def sample("):]
        ns = {"torch": torch}
        exec(compile(fn, "ref_src_utils_sample", "exec"), ns)
        ref_utils = types.SimpleNamespace(sample=ns["sample"])
    return ref_modules, ref_nb_modules, ref_alter, ref_vqgan, ref_utils


def sd_to_np(sd, prefix):
    return {prefix + k: v.detach().cpu().numpy() for k, v in sd.items()}


def fingerprint(tensors, prefix):
    """Names plus float64 sum and sum of squares of every tensor: pins seeded data too large to store."""
    ts = [v.detach().double() for v in tensors.values()]
    return {prefix + "keys": np.array(list(tensors)), prefix + "sum": np.array([float(t.sum()) for t in ts]),
            prefix + "sumsq": np.array([float(t.pow(2).sum()) for t in ts])}


N_LOGIT_SAMPLES = 8192


def make_reference_default(ref_modules, ref_vqgan):
    """reference_default.npz: the reference-default denoiser (1.008 B) and f4 VQGAN, weights re-randomised from seeds.
    Weights and the seeded float inputs are recorded as fingerprints, the 8.4 M denoiser logits as a seeded sample plus
    their per-channel and per-position means; the token inputs and the codec outputs are stored whole."""
    torch.manual_seed(0)
    m = ref_modules.Paella(byt5_embd=2560).eval()
    rerandomize_(m.state_dict(), seed=0)
    cond, _ = synthetic_conditioning(1, 16, with_clip_image=True)
    x = torch.randint(0, 8192, (1, 32, 32), generator=torch.Generator().manual_seed(1))
    r = torch.tensor([0.6])
    logits = m(x, r, cond["byt5"], clip=cond["clip"], clip_image=cond["clip_image"])
    flat = logits.reshape(-1).numpy()
    idx = np.sort(np.random.default_rng(0).choice(flat.size, N_LOGIT_SAMPLES, replace=False)).astype(np.int32)
    out = {"x": x.numpy().astype(np.int16), "r": r.numpy(), "logits_shape": np.array(logits.shape),
           "logits_std": np.array(float(logits.std())), "logits_idx": idx, "logits_sample": flat[idx],
           "logits_channel_mean": logits.mean((0, 2, 3)).numpy(), "logits_position_mean": logits.mean(1).reshape(-1).numpy()}
    out.update(fingerprint(cond, "cond_"))
    out.update(fingerprint(m.state_dict(), "denoiser_sd_"))
    del m, logits

    torch.manual_seed(0)
    vq = ref_vqgan.VQModel().eval()
    rerandomize_(vq.state_dict(), seed=4)
    img = torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(7))
    idx_v = torch.randint(0, 8192, (1, 16, 16), generator=torch.Generator().manual_seed(8))
    out.update({"vq_latents": vq.down_blocks(vq.in_block(img)).numpy(), "vq_idx": idx_v.numpy().astype(np.int16),
                "vq_dec_indices": vq.decode_indices(idx_v).numpy()})
    out.update(fingerprint({"img": img}, "vq_img_"))
    out.update(fingerprint(vq.state_dict(), "vqgan_sd_"))
    np.savez_compressed(os.path.join(HERE, "reference_default.npz"), **out)
    print("reference_default.npz:", {k: v.shape for k, v in out.items()})


def main():
    torch.set_grad_enabled(False)
    torch.set_num_threads(4)
    ref_modules, ref_nb_modules, ref_alter, ref_vqgan, ref_utils = load_reference()

    # ------------------------------------------------------------------ denoiser
    torch.manual_seed(0)
    model = ref_nb_modules.Paella(**TINY).eval()
    rerandomize_(model.state_dict(), seed=1)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    g = torch.Generator().manual_seed(2)
    B, H, L = 2, 8, 5
    x = torch.randint(0, TINY["num_labels"], (B, H, H), generator=g)
    r = torch.rand(B, generator=g)
    byt5 = torch.randn(B, L, TINY["byt5_embd"], generator=g)
    clip = torch.randn(B, TINY["clip_embd"], generator=g)
    clip_image = torch.randn(B, TINY["clip_embd"], generator=g)

    taps = {}

    def hook(name):
        def f(mod, inp, out):
            taps[name] = out.detach().clone()
        return f
    for name, mod in model.named_modules():
        if name.count(".") == 2 and (name.startswith("down_blocks.") or name.startswith("up_blocks.")):
            mod.register_forward_hook(hook(name + "."))
    logits = model(x, r, byt5, clip=clip, clip_image=clip_image)
    logits_noimg = model(x, r, byt5, clip=clip)
    logits_byt5only = model(x, r, byt5)
    out = {"cfg_json": np.array(repr(TINY)), "x": x.numpy(), "r": r.numpy(), "byt5": byt5.numpy(), "clip": clip.numpy(),
           "clip_image": clip_image.numpy(), "logits": logits.numpy(), "logits_noimg": logits_noimg.numpy(),
           "logits_byt5only": logits_byt5only.numpy(),
           "r_embed": model.gen_r_embedding(r).numpy(),
           "c_embed": model.gen_c_embeddings(byt5, clip, clip_image).numpy()}
    # per-block activations of the full-conditioning forward were overwritten by later forwards: redo
    taps.clear()
    model(x, r, byt5, clip=clip, clip_image=clip_image)
    for k, v in taps.items():
        out["tap:" + k] = v.numpy()
    # notebook path: CustomMultiheadAttention + attn_weights on the last n key columns
    ref_alter.replace_attention_layers(model)
    aw = torch.tensor([1.2, 1.2, 0.4, 0.4, 0.4])
    out["attn_weights"] = aw.numpy()
    out["logits_attnw"] = model(x, r, byt5, clip=clip, clip_image=clip_image, attn_weights=aw).numpy()
    out["logits_custom_mha"] = model(x, r, byt5, clip=clip, clip_image=clip_image).numpy()
    # add_noise with explicit mask source
    torch.manual_seed(5)
    t = torch.tensor([0.3, 0.8])
    rx = torch.randint(0, TINY["num_labels"], (B, H, H))
    torch.manual_seed(6)
    u = torch.rand_like(x.float())
    torch.manual_seed(6)
    noised, mask = model.add_noise(x, t, random_x=rx)
    out.update({"an_t": t.numpy(), "an_random_x": rx.numpy(), "an_u": u.numpy(), "an_out": noised.numpy(), "an_mask": mask.numpy()})
    out.update(sd_to_np(sd, "sd:"))
    np.savez_compressed(os.path.join(HERE, "paella_tiny.npz"), **out)
    print("paella_tiny.npz:", {k: v.shape for k, v in out.items() if not k.startswith("sd:") and not k.startswith("tap:")})

    # ------------------------------------------------------------------ sample()
    torch.manual_seed(0)
    model2 = ref_modules.Paella(**TINY).eval()
    model2.load_state_dict(sd)
    Bs, Hs = 2, 8
    cond = {"byt5": byt5, "clip": clip}
    uncond = {"byt5": torch.zeros_like(byt5), "clip": torch.zeros_like(clip)}
    steps, renoise = 4, 3
    torch.manual_seed(11)
    toks = ref_utils.sample(model2, cond, (Bs, Hs, Hs), uncond, steps=steps, renoise_steps=renoise,
                            temperature=(1.0, 0.2), cfg=8.0, device="cpu")
    # replay the CPU generator to record every draw the loop consumed
    torch.manual_seed(11)
    init = torch.randint(0, model2.num_labels, size=(Bs, Hs, Hs))
    qs, us = [], []
    for i in range(steps):
        qs.append(torch.empty(Bs * Hs * Hs, model2.num_labels).exponential_(1))
        if i < renoise:
            us.append(torch.rand(Bs, Hs, Hs))
    so = {"tokens": toks.numpy(), "init": init.numpy(), "q": torch.stack(qs).numpy(), "u": torch.stack(us).numpy(),
          "steps": np.array(steps), "renoise_steps": np.array(renoise), "byt5": byt5.numpy(), "clip": clip.numpy()}
    np.savez_compressed(os.path.join(HERE, "sample_tiny.npz"), **so)
    print("sample_tiny.npz tokens:", toks.flatten().tolist())

    # ------------------------------------------------------------------ VQGAN
    torch.manual_seed(3)
    vq = ref_vqgan.VQModel(**TINY_VQ).eval()
    rerandomize_(vq.state_dict(), seed=4)
    vsd = {k: v.clone() for k, v in vq.state_dict().items()}
    img = torch.rand(2, 3, 16, 16, generator=torch.Generator().manual_seed(7))
    lat = vq.down_blocks(vq.in_block(img))                       # pre-quantisation latents, NCHW
    qe, xs, idx, loss = vq.encode(img)
    dec_idx = vq.decode_indices(idx)
    dec = vq.decode(qe)
    idx_rand = torch.randint(0, TINY_VQ["codebook_size"], (2, 4, 4), generator=torch.Generator().manual_seed(8))
    dec_rand = vq.decode_indices(idx_rand)
    vo_ = {"cfg_json": np.array(repr(TINY_VQ)), "img": img.numpy(), "latents": lat.numpy(), "qe": qe.numpy(), "xs": xs.numpy(),
           "idx": idx.numpy(), "dec_idx": dec_idx.numpy(), "dec": dec.numpy(), "idx_rand": idx_rand.numpy(),
           "dec_rand": dec_rand.numpy()}
    vo_.update(sd_to_np(vsd, "sd:"))
    np.savez_compressed(os.path.join(HERE, "vqgan_tiny.npz"), **vo_)
    print("vqgan_tiny.npz:", {k: v.shape for k, v in vo_.items() if not k.startswith("sd:")})

    make_reference_default(ref_modules, ref_vqgan)


if __name__ == "__main__":
    main()
