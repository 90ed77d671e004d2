"""The sampling loop — ``sample()`` in the reference's three signatures over one fused core.

  sample()               ref/src/utils.py:35-55
  sample_distributed()   ref/src_distributed/utils.py:97-126   (init_x, per-step cfg, sampling_conditional_steps)
  sample_notebook()      paella_inference.ipynb cell 3          (mode, attn_weights, returns intermediates)
  sample_masked()        sample_notebook() regenerating only where a mask is set (inpainting / outpainting)

Per step the reference runs two forwards, materialises 2 x [B,8192,H,W] fp32 logits and makes ~20 passes
over them.  Here: conditional and unconditional rows run as ONE batch of 2B through the denoiser (their
conditioning K/V are computed once per call, not per step), and the out_mapper GEMM, CFG mix, temperature,
softmax and multinomial draw are a single kernel.  All random draws (randint, multinomial's exponential_,
add_noise's rand_like) come from the torch CUDA generator's own Philox stream, consumed op by op like the
reference does, so ``torch.manual_seed`` means the same thing.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch

from . import ops
from ._lib import PaellaB200Error
from .modules import Paella


def _zeros_like_inputs(inputs: Dict[str, torch.Tensor]):
    return {k: (torch.zeros_like(v) if torch.is_tensor(v) else v) for k, v in inputs.items() if v is not None}


def _sample_core(model: Paella, model_inputs, latent_shape, unconditional_inputs, init_x, steps, renoise_steps, temperature,
                 cfgs, t_start, t_end, sampling_conditional_steps, mode, attn_weights, exact, collect, sampling_quant_steps=None,
                 codebook=None, known=None, mask=None):
    """``known`` int64 [B,H,W] / ``mask`` bool [B,H,W] on the model's device (1 = regenerate), or both None: masked
    sampling keeps ``known`` wherever the mask is 0, in the start state and after every draw; the renoise is unchanged
    because the noise it draws from equals ``known`` there."""
    B, H, W = latent_shape
    dev = model._device()
    use_cfg_any = cfgs is not None
    with torch.inference_mode():
        init_noise = ops.randint(model.num_labels, (B, H, W), dev)
        if mask is not None:
            init_noise = torch.where(mask, init_noise, known)
        if init_x is not None:
            sampled = torch.where(mask, init_x.to(dev), known) if mask is not None else init_x.to(dev)
        else:
            sampled = init_noise.clone()
        t_list = torch.linspace(t_start, t_end, steps + 1)
        temperatures = torch.linspace(temperature[0], temperature[1], steps)
        groups = [model_inputs] + ([unconditional_inputs] if use_cfg_any else [])
        cond_full = model.prepare_conditioning(groups, (H, W))
        cond_only = None
        intermediates = []
        for i in range(steps):
            if sampling_quant_steps is not None and i >= sampling_quant_steps:
                mode = "quant"
            guided = use_cfg_any and i < sampling_conditional_steps
            t = float(t_list[i])
            if guided:
                cond, tokens = cond_full, sampled          # one (tokens, r) per CFG pair, see Paella.features
            elif use_cfg_any:
                if cond_only is None:
                    cond_only = model.prepare_conditioning([model_inputs], (H, W))
                cond, tokens = cond_only, sampled
            else:
                cond, tokens = cond_full, sampled
            r = torch.full((tokens.shape[0],), t, dtype=torch.float32, device=dev)
            feats = model.features(tokens, r, cond, attn_weights, B if attn_weights is not None else 0, cfg_pairs=guided)
            cfg_i = float(cfgs[i]) if guided else None
            if mode == "multinomial" and not exact and mask is not None:
                sampled = model.sample_tokens_masked(feats, B, H, W, cfg_i, float(temperatures[i]), known, mask)
            elif mode == "multinomial" and not exact:
                sampled = model.sample_tokens(feats, B, H, W, cfg_i, float(temperatures[i]))
            else:
                n = B * H * W
                lc = model.logits_from_features(feats[:n], B, H, W)
                lu = model.logits_from_features(feats[n:], B, H, W) if guided else None
                if mode == "quant":
                    if codebook is None:
                        raise ValueError("mode='quant' needs the VQGAN codebook: pass vqmodel=... (the notebook uses its global `vqmodel`)")
                    sampled = ops.resample_quant(lc, lu, cfg_i if guided else 0.0, float(temperatures[i]), codebook)
                else:
                    sampled = ops.resample_logits(lc, lu, cfg_i if guided else 0.0, float(temperatures[i]), mode)
                if mask is not None:
                    sampled = torch.where(mask, sampled, known)
            if collect:
                intermediates.append(sampled)
            if i < renoise_steps:
                t_next = torch.full((B,), float(t_list[i + 1]), dtype=torch.float32, device=dev)
                sampled = model.add_noise(sampled, t_next, random_x=init_noise)[0]
                if collect:
                    intermediates.append(sampled)
    return sampled, intermediates


def load_conditional_models(byt5_model_name, vqgan_path, device):
    """ref/src/utils.py:24-32: the f4 codec from ``vqgan_path`` (a ``{'state_dict': ...}`` checkpoint, as saved by the
    reference's training code) and the ByT5 text encoder.  The codec is this package's VQModel; the text encoder is
    the third-party ``transformers`` model exactly as in the reference (outside the hot path, SURVEY.md §8f.4) —
    ``byt5_model_name=None`` skips it."""
    from .vqgan import VQModel
    vqgan = VQModel().to(device)
    ckpt = torch.load(vqgan_path, map_location=device)
    vqgan.load_state_dict(ckpt["state_dict"] if isinstance(ckpt, dict) and "state_dict" in ckpt else ckpt)
    vqgan.eval().requires_grad_(False)
    if byt5_model_name is None:
        return vqgan, None
    from transformers import AutoTokenizer, T5EncoderModel
    byt5 = T5EncoderModel.from_pretrained(byt5_model_name).to(device).eval().requires_grad_(False)
    byt5_tokenizer = AutoTokenizer.from_pretrained(byt5_model_name)
    return vqgan, (byt5_tokenizer, byt5)


def _decode_tail(tokens, decode, decode_output):
    """The step after the path (SURVEY.md §8 f2; ref/src_distributed/train.py:168-171, notebook nb:354-357): the final token
    grid goes straight into the f4 decoder on the same stream -- no host round trip, no separate clamp / byte pass."""
    if decode is None:
        return tokens
    if decode_output == "uint8":
        return decode.decode_indices_u8(tokens)
    if decode_output == "clamp":
        return decode.decode_indices_clamped(tokens)
    if decode_output == "raw":
        return decode.decode_indices(tokens)
    raise ValueError(f"decode_output={decode_output!r}: expected 'uint8', 'clamp' or 'raw'")


def sample(model, model_inputs, latent_shape, unconditional_inputs=None, steps=12, renoise_steps=11, temperature=(1.0, 0.2),
           cfg=8.0, t_start=1.0, t_end=0.0, device="cuda", exact=False, decode=None, decode_output="uint8"):
    """ref/src/utils.py:35-55 (same positional/keyword arguments; ``device`` is accepted and must be the model's).
    ``exact=True`` materialises the logits and uses the op-for-op torch arithmetic (parity path).
    ``decode=vqmodel`` appends the reference callers' next step, ``vqmodel.decode_indices(tokens).clamp(0, 1)``, fused on the
    tail: returns uint8 NHWC images (``decode_output='uint8'``), clamped fp32 NCHW ('clamp') or unclamped fp32 NCHW ('raw')."""
    cfgs = [cfg] * steps if cfg else None
    if cfgs is not None and unconditional_inputs is None:
        raise TypeError("sample(): cfg is set but unconditional_inputs is None")
    out, _ = _sample_core(model, model_inputs, tuple(latent_shape), unconditional_inputs, None, steps, renoise_steps,
                          temperature, cfgs, t_start, t_end, steps, "multinomial", None, exact, False)
    return _decode_tail(out, decode, decode_output)


def sample_distributed(model, model_inputs, unconditional_inputs, latent_shape, init_x=None, steps=12, renoise_steps=None,
                       temperature=(0.7, 0.3), cfg=(8.0, 8.0), t_start=1.0, t_end=0.0, sampling_conditional_steps=None,
                       exact=False):
    """ref/src_distributed/utils.py:97-126."""
    if sampling_conditional_steps is None:
        sampling_conditional_steps = steps
    if renoise_steps is None:
        renoise_steps = steps - 1
    cfgs = torch.linspace(cfg[0], cfg[1], steps).tolist() if cfg is not None else None
    out, _ = _sample_core(model, model_inputs, tuple(latent_shape), unconditional_inputs, init_x, steps, renoise_steps,
                          temperature, cfgs, t_start, t_end, sampling_conditional_steps, "multinomial", None, exact, False)
    return out


def sample_notebook(model, model_inputs, latent_shape, unconditional_inputs=None, init_x=None, steps=12, renoise_steps=None,
                    temperature=(0.7, 0.3), cfg=(8.0, 8.0), mode='multinomial', t_start=1.0, t_end=0.0,
                    sampling_conditional_steps=None, sampling_quant_steps=None, attn_weights=None, exact=False, vqmodel=None):
    """paella_inference.ipynb cell 3: returns (sampled, intermediate_images).  ``vqmodel`` replaces the notebook's global
    of the same name for ``mode='quant'`` / ``sampling_quant_steps`` (softmax @ codebook -> nearest code)."""
    if sampling_conditional_steps is None:
        sampling_conditional_steps = steps
    if renoise_steps is None:
        renoise_steps = steps - 1
    if unconditional_inputs is None:
        unconditional_inputs = _zeros_like_inputs(model_inputs)
    cfgs = torch.linspace(cfg[0], cfg[1], steps).tolist() if cfg is not None else None
    codebook = vqmodel.vquantizer.codebook.weight.data if vqmodel is not None else None
    return _sample_core(model, model_inputs, tuple(latent_shape), unconditional_inputs, init_x, steps, renoise_steps,
                        temperature, cfgs, t_start, t_end, sampling_conditional_steps, mode, attn_weights, exact, True,
                        sampling_quant_steps, codebook)


def _masked_inputs(model, known, mask):
    """Validate (known [B,H,W] tokens, mask [B,H,W] or [H,W]) and move them to the model's device: int64 and bool [B,H,W]."""
    if known.dim() != 3:
        raise PaellaB200Error(f"sample_masked: known must be [B,H,W] tokens, got shape {tuple(known.shape)}")
    B, H, W = known.shape
    if tuple(mask.shape) not in ((B, H, W), (H, W)):
        raise PaellaB200Error(f"sample_masked: mask has shape {tuple(mask.shape)}, expected {(B, H, W)} or {(H, W)}")
    dev = model._device()
    known = known.to(device=dev, dtype=torch.int64).contiguous()
    mask = mask.to(device=dev).bool().expand(B, H, W).contiguous()
    return known, mask


def sample_masked(model, model_inputs, known, mask, unconditional_inputs=None, init_x=None, steps=12, renoise_steps=None,
                  temperature=(0.7, 0.3), cfg=(8.0, 8.0), mode='multinomial', t_start=1.0, t_end=0.0,
                  sampling_conditional_steps=None, sampling_quant_steps=None, attn_weights=None, exact=False, vqmodel=None):
    """Inpainting / outpainting on token grids: ``sample_notebook`` over the latent shape of ``known`` (int64 [B,H,W])
    that regenerates only the positions where ``mask`` ([B,H,W] or [H,W], broadcast over the batch) is 1 -- the meaning
    of ``mask`` in ``Paella.add_noise`` (ref/src/modules.py:277-283).  Returns (tokens, intermediates) like
    ``sample_notebook``; kept positions hold ``known`` in the result and in every intermediate.

    The torch generator is consumed exactly as by the unmasked loop of the same shape (every draw is full-size), so a
    mask of all ones reproduces ``sample_notebook`` from the same seed.  On the fused path the sampler spends work only on
    the positions to regenerate; ``exact=True``, ``mode='argmax'`` and ``'quant'`` merge after the draw."""
    known, mask = _masked_inputs(model, known, mask)
    if sampling_conditional_steps is None:
        sampling_conditional_steps = steps
    if renoise_steps is None:
        renoise_steps = steps - 1
    if unconditional_inputs is None:
        unconditional_inputs = _zeros_like_inputs(model_inputs)
    cfgs = torch.linspace(cfg[0], cfg[1], steps).tolist() if cfg is not None else None
    codebook = vqmodel.vquantizer.codebook.weight.data if vqmodel is not None else None
    return _sample_core(model, model_inputs, tuple(known.shape), unconditional_inputs, init_x, steps, renoise_steps,
                        temperature, cfgs, t_start, t_end, sampling_conditional_steps, mode, attn_weights, exact, True,
                        sampling_quant_steps, codebook, known, mask)
