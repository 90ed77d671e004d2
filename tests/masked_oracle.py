"""Test support for masked sampling (inpainting / outpainting): the masked sampling loop stated on the CPU oracle's
pieces, and the masks the masked-sampling tests run."""
from typing import Optional

import torch
from torch import Tensor

from oracle import paella_oracle as po


def sample(sd, cfg, model_inputs: dict, latent_shape, unconditional_inputs: dict, known: Tensor, mask: Tensor,
           steps=12, renoise_steps=11, temperature=(1.0, 0.2), cfg_scale=8.0, t_start=1.0, t_end=0.0,
           draws: Optional[dict] = None, mm=po.mm_fp32):
    """oracle.paella_oracle.sample (ref/src/utils.py:35-55, every random draw supplied by ``draws``) regenerating only
    where ``mask`` ([B,H,W] or [H,W]; 1 = regenerate, the meaning of ``mask`` in ref/src/modules.py:277-283) is set:
      1. start state and renoise source  init_noise = where(mask, draws['init'], known);
      2. after every draw                 sampled = where(mask, draw, known);
      3. the renoise is the unmasked one on init_noise (kept positions renoise to themselves).
    The draws are the full-size ones of the unmasked loop."""
    B = latent_shape[0]
    mask = mask.bool().expand(draws["init"].shape)
    init_noise = torch.where(mask, draws["init"], known)
    sampled = init_noise.clone()
    t_list = torch.linspace(t_start, t_end, steps + 1)
    temps = torch.linspace(temperature[0], temperature[1], steps)
    for i in range(steps):
        t = torch.ones(B) * t_list[i]
        logits = po.paella_forward(sd, cfg, sampled, t, mm=mm, **model_inputs)
        if cfg_scale:
            logits = logits * cfg_scale + po.paella_forward(sd, cfg, sampled, t, mm=mm, **unconditional_inputs) * (1 - cfg_scale)
        p = logits.div(temps[i]).softmax(dim=1).permute(0, 2, 3, 1).reshape(-1, logits.size(1))
        draw = torch.argmax(p / draws["q"][i], dim=-1).view(logits.size(0), *logits.shape[2:])
        sampled = torch.where(mask, draw, known)
        if i < renoise_steps:
            sampled, _ = po.add_noise(sampled, torch.ones(B) * t_list[i + 1], init_noise, draws["u"][i])
    return sampled


def token_masks(B, H, W, seed=0):
    """The masks (bool [B,H,W], 1 = regenerate) the masked-sampling tests run: all ones, all zeros, a random 30 %, a central
    rectangle, a border ring and a different rectangle per sample."""
    g = torch.Generator().manual_seed(seed)
    ones = torch.ones(B, H, W, dtype=torch.bool)
    rect = torch.zeros(B, H, W, dtype=torch.bool)
    rect[:, H // 4:H - H // 4, W // 4:W - W // 4] = True
    ring = torch.ones(B, H, W, dtype=torch.bool)
    ring[:, 2:H - 2, 2:W - 2] = False
    per = torch.zeros(B, H, W, dtype=torch.bool)
    for b in range(B):
        y, x = b % max(1, H // 2), (3 * b) % max(1, W // 2)
        per[b, y:y + H // 2, x:x + W // 2] = True
    return {"ones": ones, "zeros": ~ones, "random30": torch.rand(B, H, W, generator=g) < 0.3, "rect": rect, "ring": ring,
            "per_sample": per}
