"""Python mirror of the reference denoiser's class surface (ref/src/modules.py, ref/utils/modules.py).

Same class names, constructor kwargs, attribute names and state-dict keys as the reference, so
``load_state_dict(paella_v3.pt)`` and ``paella_inference.ipynb`` work unchanged — but ``forward`` runs the
hand-written sm_100a kernels behind the C ABI (include/paella_b200.h).  The ``torch.nn`` layers created
here are PARAMETER HOLDERS ONLY (they give the reference's key names and initialisation); none of their
``forward`` methods is ever called, and there is no PyTorch or CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
from torch import nn

from . import _lib, ops
from ._lib import PaellaB200Error, check, current_stream, lib, ptr


# ------------------------------------------------------------------------------------------------
# Building blocks — parameter layout AND stand-alone forward of ref/src/modules.py:7-106.
# Inside a Paella the blocks are executed by the fused plan in csrc/paella_model.cu; called on their own
# they compose the same kernels through the block-level C ABI (include/paella_b200.h).  Inference
# semantics (Dropout = identity), fp16 GEMM operands / fp32 accumulation like the model path.
# ------------------------------------------------------------------------------------------------
def _cached(mod: nn.Module, key: str, src: torch.Tensor, make):
    """Derived copy (fp16 cast / repack) of a parameter, rebuilt when the parameter changes."""
    cache = mod.__dict__.setdefault("_pb200_cache", {})
    tag = (src.data_ptr(), src._version, str(src.device))
    hit = cache.get(key)
    if hit is None or hit[0] != tag:
        with torch.no_grad():
            hit = (tag, make(src.detach()))
        cache[key] = hit
    return hit[1]


def _w16(mod, key, w):
    return _cached(mod, key, w, lambda t: t.reshape(t.shape[0], -1).to(torch.float16).contiguous())


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().float().contiguous()


def _to_rows(x: torch.Tensor) -> torch.Tensor:
    """NCHW fp32 -> channels-last rows [B*H*W, C] (a fresh buffer the block may update in place)."""
    if x.dim() != 4:
        raise PaellaB200Error(f"expected an NCHW tensor, got shape {tuple(x.shape)}")
    x = _f32(x)
    B, C, H, W = x.shape
    out = torch.empty(B * H * W, C, dtype=torch.float32, device=x.device)
    check(lib().pb200_nchw_to_nhwc(ptr(x), B, C, H * W, ptr(out), current_stream()), "pb200_nchw_to_nhwc")
    return out


def _to_nchw(rows: torch.Tensor, shape) -> torch.Tensor:
    B, C, H, W = shape
    out = torch.empty(B, C, H, W, dtype=torch.float32, device=rows.device)
    check(lib().pb200_nhwc_to_nchw(ptr(rows), B, C, H * W, ptr(out), current_stream()), "pb200_nhwc_to_nchw")
    return out


def _cast16(x: torch.Tensor, silu: bool = False) -> torch.Tensor:
    x = _f32(x)
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    check(lib().pb200_cast_f16(ptr(x), x.numel(), int(silu), ptr(out), current_stream()), "pb200_cast_f16")
    return out


def _layernorm(rows: torch.Tensor, ln: nn.LayerNorm, half: bool) -> torch.Tensor:
    M, C = rows.shape
    if tuple(ln.normalized_shape) != (C,):
        raise PaellaB200Error(f"LayerNorm over {tuple(ln.normalized_shape)} applied to {C} channels")
    out = torch.empty(M, C, dtype=torch.float16 if half else torch.float32, device=rows.device)
    w = _f32(ln.weight) if ln.weight is not None else None
    b = _f32(ln.bias) if ln.bias is not None else None
    check(lib().pb200_layernorm(ptr(rows), M, C, float(ln.eps), ptr(w), ptr(b), None if half else ptr(out),
                                ptr(out) if half else None, current_stream()), "pb200_layernorm")
    return out


def _mlp_rows(mlp: nn.Sequential, a16: torch.Tensor, resid_rows: torch.Tensor, batch: int) -> torch.Tensor:
    """channelwise = Linear -> GELU -> GRN -> Dropout(eval) -> Linear, added onto resid_rows in place."""
    lin1, grn, lin2 = mlp[0], mlp[2], mlp[4]
    M, c = a16.shape
    n = lin1.out_features
    P = M // batch
    h16 = torch.empty(M, n, dtype=torch.float16, device=a16.device)
    sq = torch.zeros(2, batch, n, dtype=torch.int64, device=a16.device)
    ops.gemm_f16(a16, _w16(lin1, "w16", lin1.weight), _lib.EPI_GELU_F16, h16, bias=_f32(lin1.bias), sqsum=sq[0], rows_per_sample=P)
    mult = torch.empty(batch, n, dtype=torch.float32, device=a16.device)
    check(lib().pb200_grn_f16(ptr(h16), batch, P, n, ptr(sq[0]), ptr(sq[1]), n, ptr(_f32(grn.gamma).view(-1)),
                              ptr(_f32(grn.beta).view(-1)), ptr(mult), current_stream()), "pb200_grn_f16")
    ops.gemm_f16(h16, _w16(lin2, "w16", lin2.weight), _lib.EPI_RESID_F32, resid_rows, bias=_f32(lin2.bias), resid=resid_rows)
    return resid_rows


class Attention2D(nn.Module):
    """ref/src/modules.py:7-19.  ``attn`` holds in_proj_weight/bias and out_proj.* under the reference's keys."""

    def __init__(self, c, nhead, dropout=0.0):
        super().__init__()
        self.attn = torch.nn.MultiheadAttention(c, nhead, dropout=dropout, bias=True, batch_first=True)

    def _core(self, xq16: torch.Tensor, kv16: torch.Tensor, batch: int, self_attn: bool, attn_weights=None) -> torch.Tensor:
        """in-projection + attention core: xq16 [B*P, E] queries (and self keys), kv16 [B*S, E] -> fp16 [B*P, E]."""
        mha = self.attn
        E = mha.embed_dim
        M = xq16.shape[0]
        P = M // batch
        S = kv16.shape[0] // batch if kv16 is not None else 0
        w16 = _w16(mha, "in16", mha.in_proj_weight)
        b32 = _f32(mha.in_proj_bias)
        qkv = torch.empty(M, 3 * E, dtype=torch.float16, device=xq16.device)
        ops.gemm_f16(xq16, w16, _lib.EPI_F16, qkv, bias=b32)
        ckv = None
        if S > 0:
            ckv = torch.empty(batch * S, 2 * E, dtype=torch.float16, device=xq16.device)
            ops.gemm_f16(kv16, w16[E:], _lib.EPI_F16, ckv, bias=b32[E:])
        aw, n_w = None, 0
        if attn_weights is not None:
            aw = _f32(attn_weights).reshape(-1)
            n_w = aw.numel()
        out = torch.empty(M, E, dtype=torch.float16, device=xq16.device)
        check(lib().pb200_attention(ptr(qkv), ptr(ckv), None, ptr(out), batch, P, S, E, mha.num_heads, int(bool(self_attn)),
                                    ptr(aw), n_w, batch, current_stream()), "pb200_attention")
        return out

    def forward(self, x, kv, self_attn=False, **kwargs):
        B, C = x.shape[0], x.shape[1]
        rows16 = _cast16(_to_rows(x))
        kv16 = _cast16(kv).view(-1, C) if kv is not None and kv.numel() > 0 else None
        o16 = self._core(rows16, kv16, B, self_attn, kwargs.get("attn_weights"))
        out = torch.empty(rows16.shape[0], C, dtype=torch.float32, device=x.device)
        ops.gemm_f16(o16, _w16(self.attn, "out16", self.attn.out_proj.weight), _lib.EPI_F32, out, bias=_f32(self.attn.out_proj.bias))
        return _to_nchw(out, x.shape)


class LayerNorm2d(nn.LayerNorm):
    """ref/src/modules.py:22-27 (no parameters when elementwise_affine=False)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)

    def forward(self, x):
        return _to_nchw(_layernorm(_to_rows(x), self, half=False), x.shape)


class GlobalResponseNorm(nn.Module):
    """ref/src/modules.py:30-40 (input NHWC ``[B, H, W, dim]``)."""

    def __init__(self, dim):
        super().__init__()
        self.gamma = nn.Parameter(torch.zeros(1, 1, 1, dim))
        self.beta = nn.Parameter(torch.zeros(1, 1, 1, dim))

    def forward(self, x):
        if x.dim() != 4 or x.shape[-1] != self.gamma.shape[-1]:
            raise PaellaB200Error(f"GlobalResponseNorm({self.gamma.shape[-1]}) got shape {tuple(x.shape)}")
        x = _f32(x)
        B, H, W, N = x.shape
        out = torch.empty_like(x)
        stat = torch.empty(B, N, dtype=torch.float32, device=x.device)
        check(lib().pb200_grn_f32(ptr(x), B, H * W, N, ptr(_f32(self.gamma).view(-1)), ptr(_f32(self.beta).view(-1)), ptr(stat),
                                  ptr(out), current_stream()), "pb200_grn_f32")
        return out


def _mlp_holder(c, dropout):
    return nn.Sequential(nn.Linear(c, c * 4), nn.GELU(), GlobalResponseNorm(c * 4), nn.Dropout(dropout), nn.Linear(c * 4, c))


class ResBlock(nn.Module):
    """ref/src/modules.py:43-62."""

    def __init__(self, c, c_skip=None, kernel_size=3, dropout=0.0):
        super().__init__()
        c_skip = c_skip or 0
        self.depthwise = nn.Conv2d(c + c_skip, c, kernel_size=kernel_size, padding=kernel_size // 2, groups=c)
        self.norm = LayerNorm2d(c, elementwise_affine=False, eps=1e-6)
        self.channelwise = _mlp_holder(c, dropout)

    def forward(self, x, x_skip=None):
        dw = self.depthwise
        c, per, k = dw.out_channels, dw.in_channels // dw.out_channels, dw.kernel_size[0]
        if per not in (1, 2) or dw.in_channels != per * c or (x_skip is not None) != (per == 2):
            raise PaellaB200Error("ResBlock: c_skip must be 0 (no x_skip) or c (with x_skip)")
        if self.norm.elementwise_affine or self.norm.eps != 1e-6:
            raise PaellaB200Error("ResBlock: the fused depthwise+LayerNorm kernel is eps=1e-6 without affine (the reference's setting)")
        B, _, H, W = x.shape
        rows = _to_rows(x)
        skip = _to_rows(x_skip) if x_skip is not None else None
        # [c, per, k, k] -> [k*k][per][c]; with a skip the conv input is cat[x, x_skip], group g reads channels 2g, 2g+1
        wp = _cached(dw, "wp", dw.weight, lambda t: t.float().permute(2, 3, 1, 0).reshape(k * k, per, c).contiguous())
        a16 = torch.empty(B * H * W, c, dtype=torch.float16, device=x.device)
        check(lib().pb200_dwconv_ln(ptr(rows), ptr(skip), ptr(wp), ptr(_f32(dw.bias)), B, H, W, c, k, ptr(a16), current_stream()),
              "pb200_dwconv_ln")
        return _to_nchw(_mlp_rows(self.channelwise, a16, rows, B), x.shape)


class AttnBlock(nn.Module):
    """ref/src/modules.py:65-79 (``attn_weights=`` as in ref/utils/modules.py:76-78)."""

    def __init__(self, c, c_cond, nhead, self_attn=True, dropout=0.0):
        super().__init__()
        self.self_attn = self_attn
        self.norm = LayerNorm2d(c, elementwise_affine=False, eps=1e-6)
        self.attention = Attention2D(c, nhead, dropout)
        self.kv_mapper = nn.Sequential(nn.SiLU(), nn.Linear(c_cond, c))

    def forward(self, x, kv, **kwargs):
        B, C = x.shape[0], x.shape[1]
        rows = _to_rows(x)
        xn16 = _layernorm(rows, self.norm, half=True)
        lin = self.kv_mapper[1]
        kv16 = None
        if kv is not None and kv.numel() > 0:
            s16 = _cast16(kv, silu=True).view(-1, lin.in_features)
            kv16 = torch.empty(s16.shape[0], C, dtype=torch.float16, device=x.device)
            ops.gemm_f16(s16, _w16(lin, "w16", lin.weight), _lib.EPI_F16, kv16, bias=_f32(lin.bias))
        o16 = self.attention._core(xn16, kv16, B, self.self_attn, kwargs.get("attn_weights"))
        mha = self.attention.attn
        ops.gemm_f16(o16, _w16(mha, "out16", mha.out_proj.weight), _lib.EPI_RESID_F32, rows, bias=_f32(mha.out_proj.bias), resid=rows)
        return _to_nchw(rows, x.shape)


class FeedForwardBlock(nn.Module):
    """ref/src/modules.py:82-96."""

    def __init__(self, c, dropout=0.0):
        super().__init__()
        self.norm = LayerNorm2d(c, elementwise_affine=False, eps=1e-6)
        self.channelwise = _mlp_holder(c, dropout)

    def forward(self, x):
        rows = _to_rows(x)
        return _to_nchw(_mlp_rows(self.channelwise, _layernorm(rows, self.norm, half=True), rows, x.shape[0]), x.shape)


class TimestepBlock(nn.Module):
    """ref/src/modules.py:99-106."""

    def __init__(self, c, c_timestep):
        super().__init__()
        self.mapper = nn.Linear(c_timestep, c * 2)

    def forward(self, x, t):
        B, C, H, W = x.shape
        film = torch.empty(B, 2 * C, dtype=torch.float32, device=x.device)
        ops.gemm_f16(_cast16(t).view(B, -1), _w16(self.mapper, "w16", self.mapper.weight), _lib.EPI_F32, film, bias=_f32(self.mapper.bias))
        rows = _to_rows(x)
        check(lib().pb200_film_apply(ptr(rows), B * H * W, C, H * W, ptr(film), 2 * C, 0, current_stream()), "pb200_film_apply")
        return _to_nchw(rows, x.shape)


# ------------------------------------------------------------------------------------------------
class ConditioningCache:
    """x- and t-independent conditioning work of one sample() call: c_embed and every AttnBlock's
    cond K/V for ``batch_total`` samples (conditional rows first, then unconditional rows)."""

    def __init__(self, cache: torch.Tensor, batch_total: int, s_max: int, slots: Optional[int] = None,
                 slot_map: Optional[torch.Tensor] = None):
        self.cache, self.batch_total, self.s_max = cache, batch_total, s_max
        # a group whose samples all carry the same conditioning (the unconditional half of a CFG batch) occupies ONE
        # slot of the cache; slot_map (int32 [batch_total], None = identity) names the slot each sample attends to
        self.slots = batch_total if slots is None else slots
        self.slot_map = slot_map


class Paella(nn.Module):
    """Drop-in for ``Paella`` (ref/src/modules.py:109-283, notebook variant ref/utils/modules.py)."""

    def __init__(self, c_in=256, c_out=256, num_labels=8192, c_r=64, patch_size=2, c_cond=1024,
                 c_hidden=[640, 1280, 1280], nhead=[-1, 16, 16], blocks=[6, 16, 6], level_config=['CT', 'CTA', 'CTA'],
                 clip_embd=1024, byt5_embd=1536, clip_seq_len=4, kernel_size=3, dropout=0.1, self_attn=True):
        super().__init__()
        self.c_r, self.c_cond, self.num_labels = c_r, c_cond, num_labels
        self._cfg = dict(c_in=c_in, c_out=c_out, num_labels=num_labels, c_r=c_r, patch_size=patch_size, c_cond=c_cond,
                         c_hidden=list(c_hidden), nhead=list(nhead), blocks=list(blocks), level_config=list(level_config),
                         clip_embd=clip_embd, byt5_embd=byt5_embd, clip_seq_len=clip_seq_len, kernel_size=kernel_size,
                         self_attn=bool(self_attn))
        if not isinstance(dropout, list):
            dropout = [dropout] * len(c_hidden)

        self.byt5_mapper = nn.Linear(byt5_embd, c_cond)
        self.clip_mapper = nn.Linear(clip_embd, c_cond * clip_seq_len)
        self.clip_image_mapper = nn.Linear(clip_embd, c_cond * clip_seq_len)
        self.seq_norm = nn.LayerNorm(c_cond, elementwise_affine=False, eps=1e-6)
        self.in_mapper = nn.Sequential(nn.Embedding(num_labels, c_in), nn.LayerNorm(c_in, elementwise_affine=False, eps=1e-6))
        self.embedding = nn.Sequential(nn.PixelUnshuffle(patch_size),
                                       nn.Conv2d(c_in * (patch_size ** 2), c_hidden[0], kernel_size=1),
                                       LayerNorm2d(c_hidden[0], elementwise_affine=False, eps=1e-6))

        def make(kind, lvl, c_skip=0):
            c = c_hidden[lvl]
            if kind == 'C':
                return ResBlock(c, c_skip, kernel_size=kernel_size, dropout=dropout[lvl])
            if kind == 'A':
                return AttnBlock(c, c_cond, nhead[lvl], self_attn=self_attn, dropout=dropout[lvl])
            if kind == 'F':
                return FeedForwardBlock(c, dropout=dropout[lvl])
            if kind == 'T':
                return TimestepBlock(c, c_r)
            raise Exception(f'Block type {kind} not supported')

        n = len(c_hidden)
        self.down_blocks = nn.ModuleList()
        for i in range(n):
            level = nn.ModuleList()
            if i > 0:
                level.append(nn.Sequential(LayerNorm2d(c_hidden[i - 1], elementwise_affine=False, eps=1e-6),
                                           nn.Conv2d(c_hidden[i - 1], c_hidden[i], kernel_size=2, stride=2)))
            for _ in range(blocks[i]):
                for kind in level_config[i]:
                    level.append(make(kind, i))
            self.down_blocks.append(level)
        self.up_blocks = nn.ModuleList()
        for i in reversed(range(n)):
            level = nn.ModuleList()
            for j in range(blocks[i]):
                for k, kind in enumerate(level_config[i]):
                    level.append(make(kind, i, c_skip=c_hidden[i] if i < n - 1 and j == k == 0 else 0))
            if i > 0:
                level.append(nn.Sequential(LayerNorm2d(c_hidden[i], elementwise_affine=False, eps=1e-6),
                                           nn.ConvTranspose2d(c_hidden[i], c_hidden[i - 1], kernel_size=2, stride=2)))
            self.up_blocks.append(level)
        self.clf = nn.Sequential(LayerNorm2d(c_hidden[0], elementwise_affine=False, eps=1e-6),
                                 nn.Conv2d(c_hidden[0], c_out * (patch_size ** 2), kernel_size=1),
                                 nn.PixelShuffle(patch_size))
        self.out_mapper = nn.Sequential(LayerNorm2d(c_out, elementwise_affine=False, eps=1e-6),
                                        nn.Conv2d(c_out, num_labels, kernel_size=1, bias=False))
        self._reference_init(blocks, num_labels)

        self._handle = None
        self._blob = None
        self._packed_key = None
        self._workspace = None
        self._cond_single = None

    # -------------------------------------------------------------- initialisation (ref/src/modules.py:189-210)
    def _reference_init(self, blocks, num_labels):
        for mod in self.modules():
            if isinstance(mod, (nn.Conv2d, nn.Linear)):
                nn.init.xavier_uniform_(mod.weight)
                if mod.bias is not None:
                    nn.init.constant_(mod.bias, 0)
        for lin in (self.byt5_mapper, self.clip_mapper, self.clip_image_mapper):
            nn.init.normal_(lin.weight, std=0.02)
        nn.init.xavier_uniform_(self.embedding[1].weight, 0.02)
        nn.init.constant_(self.clf[1].weight, 0)
        nn.init.normal_(self.in_mapper[0].weight, std=np.sqrt(1 / num_labels))
        self.out_mapper[-1].weight.data = self.in_mapper[0].weight.data[:, :, None, None].clone()
        scale = np.sqrt(1 / sum(blocks))
        for level in list(self.down_blocks) + list(self.up_blocks):
            for blk in level:
                if isinstance(blk, (ResBlock, FeedForwardBlock)):
                    blk.channelwise[-1].weight.data *= scale
                elif isinstance(blk, TimestepBlock):
                    nn.init.constant_(blk.mapper.weight, 0)

    # -------------------------------------------------------------- native handle + packed weights
    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                lib().pb200_paella_destroy(self._handle)
        except Exception:
            pass

    def _device(self):
        po = getattr(self, "_packed_only", None)
        return po if po is not None else self.in_mapper[0].weight.device

    def _weights_key(self):
        return (str(self._device()),) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def pack_weights(self, broadcast_src: Optional[int] = None):
        """Convert the reference-layout fp32 parameters into the library's packed blob (fp16 GEMM weights,
        repacked conv kernels, concatenated FiLM mappers).  With ``broadcast_src`` set and
        ``torch.distributed`` initialised, only that rank converts; the blob is then NCCL-broadcast —
        the single collective of a multi-GPU run (no collective inside the step loop)."""
        dev = self._device()
        if dev.type != "cuda":
            raise PaellaB200Error("Paella runs on CUDA only: move the model with .to('cuda') (no CPU fallback)")
        L = lib()
        if self._handle is None:
            c = self._cfg
            cfg = _lib.PaellaConfig()
            for k in ("c_in", "c_out", "num_labels", "c_r", "patch_size", "c_cond", "clip_embd", "byt5_embd",
                      "clip_seq_len", "kernel_size"):
                setattr(cfg, k, int(c[k]))
            cfg.self_attn = int(c["self_attn"])
            cfg.n_levels = len(c["c_hidden"])
            if cfg.n_levels > _lib.PB200_MAX_LEVELS:
                raise PaellaB200Error("too many levels")
            for i in range(cfg.n_levels):
                cfg.c_hidden[i], cfg.nhead[i], cfg.blocks[i] = c["c_hidden"][i], c["nhead"][i], c["blocks"][i]
                cfg.level_config[i].value = c["level_config"][i].encode()
            h = ctypes.c_void_p()
            check(L.pb200_paella_create(ctypes.byref(cfg), ctypes.byref(h)), "pb200_paella_create")
            self._handle = h
        with torch.cuda.device(dev):
            nbytes = L.pb200_paella_weight_bytes(self._handle)
            if self._blob is None or self._blob.numel() != nbytes or self._blob.device != dev:
                self._blob = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
                self._workspace = None
            check(L.pb200_paella_bind_weights(self._handle, ptr(self._blob)), "pb200_paella_bind_weights")
            import torch.distributed as dist
            distributed = broadcast_src is not None and dist.is_available() and dist.is_initialized()
            if not distributed or dist.get_rank() == broadcast_src:
                sd = self.state_dict()
                for i in range(L.pb200_paella_num_params(self._handle)):
                    name = L.pb200_paella_param_name(self._handle, i)
                    t = sd[name.decode()].detach().to(dtype=torch.float32).contiguous()
                    check(L.pb200_paella_load_param(self._handle, name, ptr(t), t.numel(), current_stream()),
                          f"pb200_paella_load_param({name.decode()})")
                torch.cuda.current_stream().synchronize()     # temporaries from .float() must outlive the copies
            if distributed:
                from .parallel import broadcast_blob
                broadcast_blob(self._blob, src=broadcast_src)      # + checksum agreement across ranks (raises on mismatch)
        self._packed_key = self._weights_key()
        self._cond_single = None
        return self

    def _ensure_packed(self):
        if getattr(self, "_packed_only", None) is not None:
            return          # from_packed(): the blob IS the model; the nn parameters are meta placeholders
        if self._handle is None or self._packed_key != self._weights_key():
            self.pack_weights()

    def _apply(self, fn, *a, **k):      # .to()/.cuda()/.half(): repack lazily
        if getattr(self, "_packed_only", None) is not None:
            return self     # a packed-only model lives where from_packed() put it
        self._packed_key = None
        return super()._apply(fn, *a, **k)

    # -------------------------------------------------------------- on-disk packed form (SURVEY.md §8 f3)
    def save_packed(self, path: str):
        """Write the library's packed weight blob (fp16 GEMM weights, repacked conv kernels, fused FiLM table, derived
        row sums) + the constructor config to ``path``: what ``tools/pack_checkpoint.py`` produces from ``paella_v3.pt``
        (nb:178-180).  ``Paella.from_packed`` memory-maps nothing and converts nothing: one H2D copy of 2.0 GB instead of
        materialising 4.0 GB of fp32 parameters and running the pack kernels."""
        from .packed import save_blob
        self._ensure_packed()
        save_blob(path, "paella", dict(self._cfg, dropout=0.0), self._blob)

    @classmethod
    def from_packed(cls, path: str, device="cuda"):
        from .packed import load_blob
        cfg, blob = load_blob(path, "paella", device)
        with torch.device("meta"):
            m = cls(**cfg)
        m.eval().requires_grad_(False)
        L = lib()
        m._packed_only = torch.device(device) if not isinstance(device, torch.device) else device
        if m._packed_only.index is None:
            m._packed_only = torch.device("cuda", torch.cuda.current_device())
        c = m._cfg
        ccfg = _lib.PaellaConfig()
        for k in ("c_in", "c_out", "num_labels", "c_r", "patch_size", "c_cond", "clip_embd", "byt5_embd", "clip_seq_len", "kernel_size"):
            setattr(ccfg, k, int(c[k]))
        ccfg.self_attn = int(c["self_attn"])
        ccfg.n_levels = len(c["c_hidden"])
        for i in range(ccfg.n_levels):
            ccfg.c_hidden[i], ccfg.nhead[i], ccfg.blocks[i] = c["c_hidden"][i], c["nhead"][i], c["blocks"][i]
            ccfg.level_config[i].value = c["level_config"][i].encode()
        h = ctypes.c_void_p()
        check(L.pb200_paella_create(ctypes.byref(ccfg), ctypes.byref(h)), "pb200_paella_create")
        m._handle = h
        if L.pb200_paella_weight_bytes(h) != blob.numel():
            raise PaellaB200Error(f"{path}: packed blob has {blob.numel()} bytes, this build's plan needs {L.pb200_paella_weight_bytes(h)} "
                                  "(packed with a different library version or config)")
        m._blob = blob
        with torch.cuda.device(blob.device):
            check(L.pb200_paella_bind_weights(h, ptr(blob)), "pb200_paella_bind_weights")
        return m

    def _ws(self, nbytes: int) -> torch.Tensor:
        """Scratch for the launches of ONE stream (the library bump-allocates it identically on every call): one buffer per
        CUDA stream the model is driven from, so calls issued on different streams never share scratch."""
        if not isinstance(self._workspace, dict):
            self._workspace = {}
        key = torch.cuda.current_stream(self._device()).cuda_stream
        ws = self._workspace.get(key)
        if ws is None or ws.numel() < nbytes or ws.device != self._device():
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self._device())
            self._workspace[key] = ws
        return ws

    # -------------------------------------------------------------- conditioning
    def prepare_conditioning(self, groups: Sequence[Dict[str, torch.Tensor]], latent_hw=(32, 32),
                             share_uniform: bool = True) -> ConditioningCache:
        """gen_c_embeddings (ref/src/modules.py:223-232) + every AttnBlock's kv_mapper and K/V projection of the
        conditioning rows, for the concatenation of ``groups`` (e.g. [conditional, unconditional]).  A group whose
        samples all carry the same tensors (the usual unconditional group) is projected once and shared."""
        self._ensure_packed()
        L = lib()
        dev = self._device()
        seq = self._cfg["clip_seq_len"]

        def seqlen(g):
            n = (1 if g.get("clip") is not None else 0)
            ci = g.get("clip_image")
            if ci is not None:
                n += len(ci) if isinstance(ci, (list, tuple)) else 1
            return g["byt5"].shape[1] + seq * n
        s_max = max(seqlen(g) for g in groups)
        bt = sum(g["byt5"].shape[0] for g in groups)

        def uniform(g):
            """All samples of the group carry identical conditioning (one host sync per tensor, once per sample() call)."""
            if not share_uniform or g["byt5"].shape[0] < 2:
                return False
            ts = [g["byt5"], g.get("clip")]
            ci = g.get("clip_image")
            ts += list(ci) if isinstance(ci, (list, tuple)) else [ci]
            return all(bool((t == t[:1]).all()) for t in ts if t is not None)
        shared = [uniform(g) for g in groups]
        slots = sum(1 if sh else g["byt5"].shape[0] for g, sh in zip(groups, shared))
        with torch.cuda.device(dev):
            # zero-filled: rows between a slot's own length and s_max are never written by the K/V GEMMs, and the attention
            # kernel multiplies them by exactly-zero probabilities -- they must be finite
            cache = torch.zeros(L.pb200_paella_cond_cache_bytes(self._handle, slots, s_max), dtype=torch.uint8, device=dev)
            ws = self._ws(L.pb200_paella_workspace_bytes(self._handle, bt, latent_hw[0], latent_hw[1], s_max))
            off = 0
            keep = []
            slot_of = []
            for g, sh in zip(groups, shared):
                n_g = g["byt5"].shape[0]
                if sh:
                    ci = g.get("clip_image")
                    g = {"byt5": g["byt5"][:1], "clip": g["clip"][:1] if g.get("clip") is not None else None,
                         "clip_image": ([t[:1] for t in ci] if isinstance(ci, (list, tuple)) else ci[:1]) if ci is not None else None}
                    slot_of += [off] * n_g
                else:
                    slot_of += list(range(off, off + n_g))
                byt5 = g["byt5"].to(device=dev, dtype=torch.float32).contiguous()
                B = byt5.shape[0]
                cond = _lib.Cond()
                cond.byt5, cond.byt5_len = ptr(byt5).value, byt5.shape[1]
                clip = g.get("clip")
                if clip is not None:
                    clip = clip.to(device=dev, dtype=torch.float32).contiguous()
                    cond.clip = ptr(clip).value
                ci = g.get("clip_image")
                if ci is not None:
                    ci = torch.stack([t.to(device=dev, dtype=torch.float32) for t in ci]) if isinstance(ci, (list, tuple)) \
                        else ci.to(device=dev, dtype=torch.float32)[None]
                    ci = ci.contiguous()
                    cond.clip_image, cond.n_clip_image = ptr(ci).value, ci.shape[0]
                keep += [byt5, clip, ci]
                check(L.pb200_paella_prepare_cond(self._handle, ctypes.byref(cond), B, off, slots, s_max, ptr(cache), ptr(ws),
                                                  ws.numel(), current_stream()), "pb200_paella_prepare_cond")
                off += B
            slot_map = torch.tensor(slot_of, dtype=torch.int32, device=dev) if slots != bt else None
        return ConditioningCache(cache, bt, s_max, slots, slot_map)

    def gen_r_embedding(self, r, max_positions=10000):
        """ref/src/modules.py:212-221 -> [B, c_r]."""
        if max_positions != 10000:
            raise PaellaB200Error("gen_r_embedding: only max_positions=10000 is built (the reference's only value)")
        dev = self._device()
        with torch.cuda.device(dev):
            r = r.to(device=dev, dtype=torch.float32).contiguous()
            out = torch.empty(r.shape[0], self.c_r, dtype=torch.float32, device=dev)
            check(lib().pb200_paella_r_embedding(ptr(r), r.shape[0], self.c_r, ptr(out), current_stream()), "pb200_paella_r_embedding")
        return out

    def gen_c_embeddings(self, byt5, clip, clip_image):
        """ref/src/modules.py:223-232 (+ list-valued clip_image, ref/utils/modules.py:228-235) -> [B, S, c_cond]."""
        self._ensure_packed()
        L, dev = lib(), self._device()
        with torch.cuda.device(dev):
            byt5 = byt5.to(device=dev, dtype=torch.float32).contiguous()
            B = byt5.shape[0]
            cond = _lib.Cond()
            cond.byt5, cond.byt5_len = ptr(byt5).value, byt5.shape[1]
            n = 0
            if clip is not None:
                clip = clip.to(device=dev, dtype=torch.float32).contiguous()
                cond.clip = ptr(clip).value
                n += 1
            ci = clip_image
            if ci is not None:
                ci = torch.stack([t.to(device=dev, dtype=torch.float32) for t in ci]) if isinstance(ci, (list, tuple)) \
                    else ci.to(device=dev, dtype=torch.float32)[None]
                ci = ci.contiguous()
                cond.clip_image, cond.n_clip_image = ptr(ci).value, ci.shape[0]
                n += ci.shape[0]
            S = byt5.shape[1] + self._cfg["clip_seq_len"] * n
            out = torch.empty(B, S, self.c_cond, dtype=torch.float32, device=dev)
            ws = self._ws(L.pb200_paella_workspace_bytes(self._handle, B, 2 * self._cfg["patch_size"] * 2 ** (len(self._cfg["c_hidden"]) - 1),
                                                         2 * self._cfg["patch_size"] * 2 ** (len(self._cfg["c_hidden"]) - 1), S))
            check(L.pb200_paella_c_embeddings(self._handle, ctypes.byref(cond), B, ptr(out), ptr(ws), ws.numel(), current_stream()),
                  "pb200_paella_c_embeddings")
        return out

    # -------------------------------------------------------------- forward pieces
    def features(self, x: torch.Tensor, r: torch.Tensor, cond: ConditioningCache, attn_weights=None,
                 attn_weights_batch: int = 0, cfg_pairs: bool = False) -> torch.Tensor:
        """Everything up to out_mapper's LayerNorm: tokens [Bt,H,W] -> fp32 [Bt*H*W, c_out].

        ``cfg_pairs=True``: x [B,H,W] and r [B] are the classifier-free-guidance batch of ref/src/utils.py:42-45 —
        evaluated under the conditional rows [0,B) and the unconditional rows [B,2B) of ``cond``; the result has 2B
        samples, and the conditioning-independent blocks before the first AttnBlock run once per pair."""
        self._ensure_packed()
        L = lib()
        dev = self._device()
        Bt, H, W = x.shape
        if cfg_pairs:
            Bt *= 2
        if Bt != cond.batch_total:
            raise PaellaB200Error(f"batch {Bt} does not match the conditioning cache ({cond.batch_total})")
        with torch.cuda.device(dev):
            x = x.to(device=dev, dtype=torch.int64).contiguous()
            r = r.to(device=dev, dtype=torch.float32).contiguous()
            ws = self._ws(L.pb200_paella_workspace_bytes(self._handle, Bt, H, W, cond.s_max))
            feats = torch.empty(Bt * H * W, self._cfg["c_out"], dtype=torch.float32, device=dev)
            aw = attn_weights.to(device=dev, dtype=torch.float32).contiguous() if attn_weights is not None else None
            check(L.pb200_paella_features(self._handle, ptr(x), ptr(r), Bt, int(cfg_pairs), H, W, ptr(cond.cache), cond.slots,
                                          ptr(cond.slot_map), cond.s_max, ptr(aw),
                                          aw.numel() if aw is not None else 0, attn_weights_batch, ptr(feats), ptr(ws),
                                          ws.numel(), current_stream()), "pb200_paella_features")
        return feats

    def logits_from_features(self, feats: torch.Tensor, batch: int, h: int, w: int) -> torch.Tensor:
        self._ensure_packed()
        L = lib()
        dev = self._device()
        with torch.cuda.device(dev):
            out = torch.empty(batch, self.num_labels, h, w, dtype=torch.float32, device=dev)
            ws = self._ws(feats.numel() * 2 + 256)
            check(L.pb200_paella_logits(self._handle, ptr(feats), batch, h * w, ptr(out), ptr(ws), ws.numel(),
                                        current_stream()), "pb200_paella_logits")
        return out

    def sample_tokens(self, feats: torch.Tensor, batch: int, h: int, w: int, cfg: Optional[float], temperature: float,
                      generator=None) -> torch.Tensor:
        """Fused out_mapper + CFG + temperature + multinomial on torch's random stream (ref/src/utils.py:44-50)."""
        self._ensure_packed()
        L = lib()
        dev = self._device()
        with torch.cuda.device(dev):
            out = torch.empty(batch, h, w, dtype=torch.int64, device=dev)
            ws = self._ws(L.pb200_paella_workspace_bytes(self._handle, batch, h, w, 1))
            n = batch * h * w
            chunks = ops.philox_row_chunks(n, self.num_labels)       # one kernel per 32-bit-indexable piece, like torch
            ops.skip_philox_for_split(chunks, n * self.num_labels, dev, generator)
            flat = out.view(-1)
            for lo, hi in chunks:
                seed, off = ops.take_philox((hi - lo) * self.num_labels, dev, generator)
                if len(chunks) == 1:
                    f = feats
                elif cfg is not None:
                    f = torch.cat([feats[lo:hi], feats[n + lo:n + hi]])
                else:
                    f = feats[lo:hi]
                check(L.pb200_paella_sample_tokens(self._handle, ptr(f), 1, hi - lo, 1 if cfg is not None else 0,
                                                   float(cfg) if cfg is not None else 0.0, float(temperature), seed, off,
                                                   ptr(flat[lo:hi]), ptr(ws), ws.numel(), current_stream()), "pb200_paella_sample_tokens")
        return out

    def sample_tokens_masked(self, feats: torch.Tensor, batch: int, h: int, w: int, cfg: Optional[float], temperature: float,
                             known: torch.Tensor, mask: torch.Tensor, generator=None) -> torch.Tensor:
        """``where(mask, sample_tokens(...), known)`` without drawing the kept rows: ``known`` int64 [B,H,W], ``mask``
        bool/uint8 [B,H,W] (1 = regenerate).  The draw at a masked position is bit-identical to ``sample_tokens``'s and the
        generator advances by the same amount, so a mask of all ones reproduces the unmasked sampler."""
        self._ensure_packed()
        L = lib()
        dev = self._device()
        with torch.cuda.device(dev):
            out = known.to(device=dev, dtype=torch.int64).reshape(batch, h, w).clone()
            m8 = mask.to(device=dev).reshape(batch, h, w)
            m8 = (m8 if m8.dtype == torch.bool else m8 != 0).contiguous().view(torch.uint8)      # bool storage is 0 / 1 bytes
            ws = self._ws(L.pb200_paella_workspace_bytes(self._handle, batch, h, w, 1))
            n = batch * h * w
            chunks = ops.philox_row_chunks(n, self.num_labels)       # the same pieces, offsets and draws as sample_tokens
            ops.skip_philox_for_split(chunks, n * self.num_labels, dev, generator)
            flat, mflat = out.view(-1), m8.view(-1)
            for lo, hi in chunks:
                seed, off = ops.take_philox((hi - lo) * self.num_labels, dev, generator)
                if len(chunks) == 1:
                    f = feats
                elif cfg is not None:
                    f = torch.cat([feats[lo:hi], feats[n + lo:n + hi]])
                else:
                    f = feats[lo:hi]
                check(L.pb200_paella_sample_tokens_masked(self._handle, ptr(f), 1, hi - lo, 1 if cfg is not None else 0,
                                                          float(cfg) if cfg is not None else 0.0, float(temperature), seed, off,
                                                          ptr(mflat[lo:hi]), ptr(flat[lo:hi]), ptr(ws), ws.numel(),
                                                          current_stream()), "pb200_paella_sample_tokens_masked")
        return out

    def forward(self, x, r, byt5, clip=None, clip_image=None, x_cat=None, **kwargs):
        """ref/src/modules.py:263-275 / ref/utils/modules.py:268-282: logits [B, num_labels, H, W] fp32."""
        if x_cat is not None:
            x = torch.cat([x, x_cat], dim=1)
        attn_weights = kwargs.pop("attn_weights", None)
        if kwargs:
            raise TypeError(f"unexpected keyword arguments {sorted(kwargs)}")
        B, H, W = x.shape
        cond = self._cond_for_forward(byt5, clip, clip_image, (H, W))
        feats = self.features(x, r, cond, attn_weights, B if attn_weights is not None else 0)
        return self.logits_from_features(feats, B, H, W)

    def _cond_for_forward(self, byt5, clip, clip_image, hw):
        """The reference's own loop calls ``model(x, t, **inputs)`` twice per step with the SAME conditioning tensors
        (ref/src/utils.py:42-45): the conditioning cache (44 kv_mapper + K/V GEMMs) is memoised on the identity and version
        of those tensor objects (references are held, so an address cannot be recycled under the memo) and the weights."""
        self._ensure_packed()
        ci = list(clip_image) if isinstance(clip_image, (list, tuple)) else [clip_image]
        ts = [byt5, clip] + ci
        try:
            vers = tuple(None if t is None else t._version for t in ts)
        except RuntimeError:        # inference tensors carry no version counter: no memo
            vers = None
        # a few entries, most recent first: the loop alternates between the conditional and the unconditional inputs
        memos = self._cond_single if isinstance(self._cond_single, list) else []
        if vers is not None:
            for i, memo in enumerate(memos):
                if (memo["hw"] == tuple(hw) and memo["vers"] == vers and len(memo["ts"]) == len(ts)
                        and all(a is b for a, b in zip(memo["ts"], ts)) and memo["key"] == self._packed_key):
                    if i:
                        memos.insert(0, memos.pop(i))
                    return memo["cond"]
        cond = self.prepare_conditioning([{"byt5": byt5, "clip": clip, "clip_image": clip_image}], hw, share_uniform=False)
        if vers is not None:
            memos.insert(0, {"hw": tuple(hw), "vers": vers, "ts": ts, "cond": cond, "key": self._packed_key})
            del memos[4:]
            self._cond_single = memos
        return cond

    def add_noise(self, x, t, mask=None, random_x=None):
        """ref/src/modules.py:277-283 on torch's random stream."""
        if mask is None:
            return ops.add_noise(x, t, random_x, self.num_labels)
        if random_x is None:
            random_x = ops.randint(self.num_labels, x.shape, x.device)
        return torch.where(mask.bool(), random_x, x), mask

    def get_loss_weight(self, t, mask, min_val=0.3):    # ref/utils/modules.py:290-291 (training helper)
        return 1 - (1 - mask) * ((1 - t) * (1 - min_val))[:, None, None]
