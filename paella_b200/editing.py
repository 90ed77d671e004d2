"""Inpainting and outpainting on images: the pixel <-> token geometry around ``utils.sample_masked``.

The f4 VQGAN maps a 4x4 pixel block to one token, so a token is regenerated when any pixel of its block is masked.  The
denoiser's latent grid must be a multiple of ``patch_size << (levels - 1)`` (16 for the reference config).  Everything is
validated before the first launch; mask preparation runs once per call, the per-step work is the library's kernels.

  inpaint(model, vq, images, pixel_mask, inputs)          regenerate the masked pixels of each image
  outpaint(model, vq, images, canvas_hw, offset_yx, inputs)  place each image on a larger canvas and fill the rest
"""
from __future__ import annotations

import torch

from ._lib import PaellaB200Error
from .utils import _decode_tail, sample_masked

_OUTPUTS = ("uint8", "clamp", "raw", "tokens")


def latent_multiple(model) -> int:
    """The denoiser's latent grid must be a multiple of this (patch_size << (levels - 1))."""
    return int(model._cfg["patch_size"]) << (len(model._cfg["c_hidden"]) - 1)


def token_mask(pixel_mask: torch.Tensor) -> torch.Tensor:
    """bool [..., H, W] pixels -> bool [..., H/4, W/4] tokens: a token is set when any pixel of its 4x4 block is set."""
    *lead, H, W = pixel_mask.shape
    return pixel_mask.bool().reshape(*lead, H // 4, 4, W // 4, 4).any(dim=-1).any(dim=-2)


def _check_output(output):
    if output not in _OUTPUTS:
        raise PaellaB200Error(f"output={output!r}: expected one of {_OUTPUTS}")


def _check_canvas(model, H, W, what):
    if H % 4 or W % 4:
        raise PaellaB200Error(f"{what} {H}x{W} px is not a multiple of 4 px (one token = 4x4 px)")
    mult = latent_multiple(model)
    if (H // 4) % mult or (W // 4) % mult:
        raise PaellaB200Error(f"{what} {H}x{W} px gives a {H // 4}x{W // 4} latent grid; the denoiser needs a multiple of {mult} "
                              f"tokens ({4 * mult} px) on each side")


def _check_images(images, what):
    if images.dim() != 4 or images.shape[1] != 3:
        raise PaellaB200Error(f"{what}: images must be [B,3,H,W], got shape {tuple(images.shape)}")


def _finish(vqmodel, tokens, output, paste_back, orig, pixel_mask):
    if output == "tokens":
        return tokens
    if paste_back:
        return vqmodel.decode_composite(tokens, orig, pixel_mask, output)
    return _decode_tail(tokens, vqmodel, output)


def inpaint(model, vqmodel, images, pixel_mask, model_inputs, unconditional_inputs=None, output="uint8", paste_back=True,
            **sample_kwargs):
    """Regenerate the pixels of ``images`` (fp32 [B,3,H,W] in [0,1]) where ``pixel_mask`` ([B,H,W] or [H,W]) is 1.

    The images are encoded, every token with a masked pixel in its 4x4 block is resampled by ``sample_masked`` (keyword
    arguments as there: steps, temperature, cfg, ...), and the result is decoded.  ``output``: 'uint8' (NHWC), 'clamp' or
    'raw' (fp32 NCHW), or 'tokens' (int64 [B,H/4,W/4]).  ``paste_back=True`` composites the decoded pixels into the input
    in the decoder's last kernel, so pixels outside the mask are the input's own; ``False`` returns the plain decode."""
    _check_output(output)
    _check_images(images, "inpaint")
    B, _, H, W = images.shape
    _check_canvas(model, H, W, "inpaint: image")
    if tuple(pixel_mask.shape) not in ((B, H, W), (H, W)):
        raise PaellaB200Error(f"inpaint: pixel_mask has shape {tuple(pixel_mask.shape)}, expected {(B, H, W)} or {(H, W)}")
    dev = model._device()
    images = images.to(device=dev, dtype=torch.float32).contiguous()
    pixel_mask = pixel_mask.to(device=dev).bool()
    known = vqmodel.encode(images)[2]
    tokens, _ = sample_masked(model, model_inputs, known, token_mask(pixel_mask), unconditional_inputs, **sample_kwargs)
    return _finish(vqmodel, tokens, output, paste_back, images, pixel_mask)


def outpaint(model, vqmodel, images, canvas_hw, offset_yx, model_inputs, unconditional_inputs=None, output="uint8",
             paste_back=True, **sample_kwargs):
    """Place ``images`` (fp32 [B,3,h,w] in [0,1]) at pixel ``offset_yx`` on a ``canvas_hw`` pixel canvas and generate the
    rest.  The image is encoded on its own and its tokens are placed at ``offset_yx // 4`` of the canvas's latent grid;
    every other token is regenerated.  Non-square canvases are fine.  ``output`` / ``paste_back`` as in ``inpaint`` (the
    pasted-back region is the image itself)."""
    _check_output(output)
    _check_images(images, "outpaint")
    B, _, h, w = images.shape
    CH, CW = (int(v) for v in canvas_hw)
    oy, ox = (int(v) for v in offset_yx)
    _check_canvas(model, CH, CW, "outpaint: canvas")
    if h % 4 or w % 4:
        raise PaellaB200Error(f"outpaint: image {h}x{w} px is not a multiple of 4 px")
    if oy % 4 or ox % 4:
        raise PaellaB200Error(f"outpaint: offset {(oy, ox)} px is not a multiple of 4 px")
    if oy < 0 or ox < 0 or oy + h > CH or ox + w > CW:
        raise PaellaB200Error(f"outpaint: a {h}x{w} px image at offset {(oy, ox)} does not fit in a {CH}x{CW} px canvas")
    dev = model._device()
    images = images.to(device=dev, dtype=torch.float32).contiguous()
    idx = vqmodel.encode(images)[2]
    known = torch.zeros(B, CH // 4, CW // 4, dtype=torch.int64, device=dev)
    known[:, oy // 4:(oy + h) // 4, ox // 4:(ox + w) // 4] = idx
    mask = torch.ones(CH // 4, CW // 4, dtype=torch.bool, device=dev)
    mask[oy // 4:(oy + h) // 4, ox // 4:(ox + w) // 4] = False
    tokens, _ = sample_masked(model, model_inputs, known, mask, unconditional_inputs, **sample_kwargs)
    if output == "tokens" or not paste_back:
        return _finish(vqmodel, tokens, output, False, None, None)
    canvas = torch.zeros(B, 3, CH, CW, dtype=torch.float32, device=dev)
    canvas[:, :, oy:oy + h, ox:ox + w] = images
    pixel_mask = torch.ones(CH, CW, dtype=torch.bool, device=dev)
    pixel_mask[oy:oy + h, ox:ox + w] = False
    return _finish(vqmodel, tokens, output, True, canvas, pixel_mask)
