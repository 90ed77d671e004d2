"""Python mirror of the reference's f4 VQGAN codec (ref/src/vqgan.py:6-112) and of the third-party
``torchtools.nn.VectorQuantize`` it instantiates (restated: see oracle/vqgan_oracle.py, PARITY UNPINNED).

Same class names, constructor kwargs, attribute names and state-dict keys as the reference; the ``torch.nn``
layers are parameter holders only — ``encode`` / ``decode`` / ``decode_indices`` run the CUDA library
(include/paella_b200.h, pb200_vqgan_*).  No CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch
from torch import nn

from . import _lib, ops
from ._lib import PaellaB200Error, check, current_stream, lib, ptr


class VectorQuantize(nn.Module):
    """Nearest-codebook quantiser with the call surface the reference uses:
    ``VectorQuantize(c_latent, k=codebook_size)``, ``.codebook.weight [k, C]``,
    ``forward(x, dim) -> (z_q, (vq_loss, commit_loss), indices)``, ``idx2vq(idx, dim)``."""

    def __init__(self, embedding_size, k, ema_decay=0.99, ema_loss=False):
        super().__init__()
        self.codebook = nn.Embedding(k, embedding_size)
        self.codebook.weight.data.uniform_(-1. / k, 1. / k)

    def forward(self, x, get_losses=True, dim=-1):
        if dim != -1:
            x = x.movedim(dim, -1)
        x = x.contiguous().float()
        idx = ops.vq_nearest(x, self.codebook.weight.data)
        zq = ops.vq_gather(idx, self.codebook.weight.data)
        vq_loss = commit = None
        if get_losses:
            vq_loss = torch.mean((zq - x) ** 2)
            commit = vq_loss.clone()
        if dim != -1:
            zq = zq.movedim(-1, dim)
        return zq, (vq_loss, commit), idx

    def idx2vq(self, idx, dim=-1):
        q = ops.vq_gather(idx, self.codebook.weight.data)
        if dim != -1:
            q = q.movedim(-1, dim)
        return q


class ResBlock(nn.Module):
    """ref/src/vqgan.py:6-42 (parameter holder)."""

    def __init__(self, c, c_hidden):
        super().__init__()
        self.norm1 = nn.LayerNorm(c, elementwise_affine=False, eps=1e-6)
        self.depthwise = nn.Sequential(nn.ReplicationPad2d(1), nn.Conv2d(c, c, kernel_size=3, groups=c))
        self.norm2 = nn.LayerNorm(c, elementwise_affine=False, eps=1e-6)
        self.channelwise = nn.Sequential(nn.Linear(c, c_hidden), nn.GELU(), nn.Linear(c_hidden, c))
        self.gammas = nn.Parameter(torch.zeros(6), requires_grad=True)
        for mod in self.modules():
            if isinstance(mod, (nn.Linear, nn.Conv2d)):
                nn.init.xavier_uniform_(mod.weight)
                if mod.bias is not None:
                    nn.init.constant_(mod.bias, 0)

    def forward(self, x):
        """ref/src/vqgan.py:36-42 on its own: NCHW fp32 in/out, the same kernels VQModel's plan runs (pb200_vqgan_resblock)."""
        from .modules import _cached, _f32, _to_nchw, _to_rows, _w16
        if x.dim() != 4 or x.shape[1] != self.norm1.normalized_shape[0]:
            raise PaellaB200Error(f"vqgan.ResBlock({self.norm1.normalized_shape[0]}) got shape {tuple(x.shape)}")
        B, c, H, W = x.shape
        rows = _to_rows(x)
        dw, l1, l2 = self.depthwise[1], self.channelwise[0], self.channelwise[2]
        w9 = _cached(dw, "w9", dw.weight, lambda t: t.float().reshape(c, 9).t().contiguous())
        gam = (ctypes.c_float * 6)(*[float(v) for v in self.gammas.detach().float().cpu()])
        L = lib()
        ws = torch.empty(L.pb200_vqgan_resblock_workspace_bytes(B, H, W, c), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            check(L.pb200_vqgan_resblock(ptr(rows), B, H, W, c, ptr(w9), ptr(_f32(dw.bias)), ptr(_w16(l1, "w16", l1.weight)),
                                         ptr(_f32(l1.bias)), ptr(_w16(l2, "w16", l2.weight)), ptr(_f32(l2.bias)), gam, ptr(ws),
                                         ws.numel(), current_stream()), "pb200_vqgan_resblock")
        return _to_nchw(rows, x.shape)


class VQModel(nn.Module):
    """Drop-in for ``VQModel`` (ref/src/vqgan.py:45-112)."""

    def __init__(self, levels=2, bottleneck_blocks=12, c_hidden=384, c_latent=4, codebook_size=8192, scale_factor=0.3764):
        super().__init__()
        self.c_latent = c_latent
        self.scale_factor = scale_factor
        self._cfg = dict(levels=levels, bottleneck_blocks=bottleneck_blocks, c_hidden=c_hidden, c_latent=c_latent,
                         codebook_size=codebook_size, scale_factor=scale_factor)
        c_levels = [c_hidden // (2 ** i) for i in reversed(range(levels))]
        self.in_block = nn.Sequential(nn.PixelUnshuffle(2), nn.Conv2d(3 * 4, c_levels[0], kernel_size=1))
        down = []
        for i in range(levels):
            if i > 0:
                down.append(nn.Conv2d(c_levels[i - 1], c_levels[i], kernel_size=4, stride=2, padding=1))
            down.append(ResBlock(c_levels[i], c_levels[i] * 4))
        down.append(nn.Sequential(nn.Conv2d(c_levels[-1], c_latent, kernel_size=1, bias=False), nn.BatchNorm2d(c_latent)))
        self.down_blocks = nn.Sequential(*down)
        self.codebook_size = codebook_size
        self.vquantizer = VectorQuantize(c_latent, k=codebook_size)
        up = [nn.Sequential(nn.Conv2d(c_latent, c_levels[-1], kernel_size=1))]
        for i in range(levels):
            for _ in range(bottleneck_blocks if i == 0 else 1):
                up.append(ResBlock(c_levels[levels - 1 - i], c_levels[levels - 1 - i] * 4))
            if i < levels - 1:
                up.append(nn.ConvTranspose2d(c_levels[levels - 1 - i], c_levels[levels - 2 - i], kernel_size=4, stride=2, padding=1))
        self.up_blocks = nn.Sequential(*up)
        self.out_block = nn.Sequential(nn.Conv2d(c_levels[0], 3 * 4, kernel_size=1), nn.PixelShuffle(2))
        self._handle = None
        self._blob = None
        self._packed_key = None
        self._workspace = None

    # -------------------------------------------------------------- native handle + packed weights
    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                lib().pb200_vqgan_destroy(self._handle)
        except Exception:
            pass

    def _device(self):
        po = getattr(self, "_packed_only", None)
        return po if po is not None else self.vquantizer.codebook.weight.device

    def _weights_key(self):
        return (str(self._device()),) + tuple((t.data_ptr(), t._version) for t in self.state_dict().values())

    def load_state_dict(self, state_dict, strict=True, **kw):
        # the real vqgan_f4.pt may carry extra vquantizer.* buffers (EMA statistics) from the unpinned torchtools
        own = set(self.state_dict().keys())
        extra = [k for k in state_dict if k not in own and k.startswith("vquantizer.")]
        if extra:
            state_dict = {k: v for k, v in state_dict.items() if k not in extra}
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def pack_weights(self, broadcast_src: Optional[int] = None):
        dev = self._device()
        if dev.type != "cuda":
            raise PaellaB200Error("VQModel runs on CUDA only: move the model with .to('cuda') (no CPU fallback)")
        L = lib()
        if self._handle is None:
            cfg = _lib.VqganConfig()
            for k in ("levels", "bottleneck_blocks", "c_hidden", "c_latent", "codebook_size"):
                setattr(cfg, k, int(self._cfg[k]))
            cfg.scale_factor = float(self.scale_factor)
            h = ctypes.c_void_p()
            check(L.pb200_vqgan_create(ctypes.byref(cfg), ctypes.byref(h)), "pb200_vqgan_create")
            self._handle = h
        with torch.cuda.device(dev):
            nbytes = L.pb200_vqgan_weight_bytes(self._handle)
            if self._blob is None or self._blob.numel() != nbytes or self._blob.device != dev:
                self._blob = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
            check(L.pb200_vqgan_bind_weights(self._handle, ptr(self._blob)), "pb200_vqgan_bind_weights")
            import torch.distributed as dist
            distributed = broadcast_src is not None and dist.is_available() and dist.is_initialized()
            if not distributed or dist.get_rank() == broadcast_src:
                sd = self.state_dict()
                for i in range(L.pb200_vqgan_num_params(self._handle)):
                    name = L.pb200_vqgan_param_name(self._handle, i)
                    t = sd[name.decode()].detach().to(dtype=torch.float32).contiguous()
                    check(L.pb200_vqgan_load_param(self._handle, name, ptr(t), t.numel(), current_stream()),
                          f"pb200_vqgan_load_param({name.decode()})")
                torch.cuda.current_stream().synchronize()
            if distributed:
                from .parallel import broadcast_blob
                broadcast_blob(self._blob, src=broadcast_src)      # + checksum agreement across ranks (raises on mismatch)
            # the library mirrors the six ResBlock gammas on the host (kernel arguments): refresh them from the blob now that
            # it is complete on every rank (a rank that only received the broadcast never ran load_param)
            check(L.pb200_vqgan_sync_params(self._handle, current_stream()), "pb200_vqgan_sync_params")
        self._packed_key = self._weights_key()
        return self

    def _ensure_packed(self):
        if getattr(self, "_packed_only", None) is not None:
            return
        if self._handle is None or self._packed_key != self._weights_key():
            self.pack_weights()

    def _apply(self, fn, *a, **k):
        if getattr(self, "_packed_only", None) is not None:
            return self
        self._packed_key = None
        return super()._apply(fn, *a, **k)

    # -------------------------------------------------------------- on-disk packed form (SURVEY.md §8 f3)
    def save_packed(self, path: str):
        """Packed blob + config of this codec -> ``path`` (tools/pack_checkpoint.py does this for ``vqgan_f4.pt``, nb:157)."""
        from .packed import save_blob
        self._ensure_packed()
        save_blob(path, "vqgan", dict(self._cfg), self._blob)

    @classmethod
    def from_packed(cls, path: str, device="cuda"):
        from .packed import load_blob
        cfg, blob = load_blob(path, "vqgan", device)
        with torch.device("meta"):
            m = cls(**cfg)
        m.eval().requires_grad_(False)
        L = lib()
        m._packed_only = blob.device
        ccfg = _lib.VqganConfig()
        for k in ("levels", "bottleneck_blocks", "c_hidden", "c_latent", "codebook_size"):
            setattr(ccfg, k, int(cfg[k]))
        ccfg.scale_factor = float(cfg["scale_factor"])
        h = ctypes.c_void_p()
        check(L.pb200_vqgan_create(ctypes.byref(ccfg), ctypes.byref(h)), "pb200_vqgan_create")
        m._handle = h
        if L.pb200_vqgan_weight_bytes(h) != blob.numel():
            raise PaellaB200Error(f"{path}: packed blob has {blob.numel()} bytes, this build's plan needs {L.pb200_vqgan_weight_bytes(h)}")
        m._blob = blob
        with torch.cuda.device(blob.device):
            check(L.pb200_vqgan_bind_weights(h, ptr(blob)), "pb200_vqgan_bind_weights")      # gammas are re-read lazily
        return m

    def _ws(self, nbytes):
        if self._workspace is None or self._workspace.numel() < nbytes or self._workspace.device != self._device():
            self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=self._device())
        return self._workspace

    # -------------------------------------------------------------- reference API
    def encode(self, x, quantize=False):
        """ref/src/vqgan.py:91-95 -> (qe/sf, x/sf, indices, vq_loss + 0.25*commit_loss).  ``quantize`` is accepted
        and ignored: the notebook passes it although the reference signature does not take it (SURVEY.md §3.3)."""
        self._ensure_packed()
        L, dev = lib(), self._device()
        B, C, H, W = x.shape
        assert C == 3, "VQModel.encode expects [B,3,H,W]"
        with torch.cuda.device(dev):
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            h, w = H // 4, W // 4
            lat = torch.empty(B, self.c_latent, h, w, dtype=torch.float32, device=dev)
            qe = torch.empty_like(lat)
            idx = torch.empty(B, h, w, dtype=torch.int64, device=dev)
            ws = self._ws(L.pb200_vqgan_workspace_bytes(self._handle, B, H, W))
            check(L.pb200_vqgan_encode(self._handle, ptr(x), B, H, W, ptr(lat), ptr(qe), ptr(idx), ptr(ws), ws.numel(),
                                       current_stream()), "pb200_vqgan_encode")
        mse = torch.mean((qe - lat) ** 2)
        return qe / self.scale_factor, lat / self.scale_factor, idx, mse + mse * 0.25

    def _decode(self, idx, lat, mode=_lib.IMG_F32_NCHW):
        self._ensure_packed()
        L, dev = lib(), self._device()
        with torch.cuda.device(dev):
            if idx is not None:
                idx = idx.to(device=dev, dtype=torch.int64).contiguous()
                B, h, w = idx.shape
            else:
                lat = lat.to(device=dev, dtype=torch.float32).contiguous()
                B, _, h, w = lat.shape
            if mode == _lib.IMG_U8_NHWC:
                img = torch.empty(B, 4 * h, 4 * w, 3, dtype=torch.uint8, device=dev)
            else:
                img = torch.empty(B, 3, 4 * h, 4 * w, dtype=torch.float32, device=dev)
            ws = self._ws(L.pb200_vqgan_workspace_bytes(self._handle, B, 4 * h, 4 * w))
            check(L.pb200_vqgan_decode_ex(self._handle, ptr(idx), ptr(lat), B, h, w, ptr(img), mode, ptr(ws), ws.numel(),
                                          current_stream()), "pb200_vqgan_decode_ex")
        return img

    def decode(self, x):
        """ref/src/vqgan.py:97-101."""
        return self._decode(None, x * self.scale_factor)

    def decode_indices(self, x):
        """ref/src/vqgan.py:103-107 (no scale_factor on this path, as in the reference)."""
        return self._decode(x, None)

    def decode_indices_clamped(self, x):
        """``decode_indices(x).clamp(0, 1)`` (ref/src_distributed/train.py:168-171) with the clamp fused into the decoder's last kernel."""
        return self._decode(x, None, _lib.IMG_F32_NCHW_CLAMP01)

    def decode_indices_u8(self, x):
        """uint8 NHWC images [B,4h,4w,3]: ``decode_indices(x).clamp(0,1)`` followed by torchvision save_image's byte conversion
        (``mul(255).add_(0.5).clamp_(0,255).to(uint8)`` on the HWC view), fused into the decoder's last kernel."""
        return self._decode(x, None, _lib.IMG_U8_NHWC)

    def decode_composite(self, x, orig, pixel_mask, output="uint8"):
        """Decode indices x [B,h,w] and paste the original image back: pixels where ``pixel_mask`` ([B,4h,4w] or [4h,4w],
        1 = decoded) is 0 come from ``orig`` (fp32 NCHW [B,3,4h,4w]) through the same conversion as the decoded ones.
        ``output``: 'uint8' (NHWC, as ``decode_indices_u8``), 'clamp' or 'raw' (fp32 NCHW).  One fused last kernel."""
        mode = {"uint8": _lib.IMG_U8_NHWC, "clamp": _lib.IMG_F32_NCHW_CLAMP01, "raw": _lib.IMG_F32_NCHW}.get(output)
        if mode is None:
            raise ValueError(f"output={output!r}: expected 'uint8', 'clamp' or 'raw'")
        self._ensure_packed()
        L, dev = lib(), self._device()
        with torch.cuda.device(dev):
            idx = x.to(device=dev, dtype=torch.int64).contiguous()
            B, h, w = idx.shape
            if tuple(orig.shape) != (B, 3, 4 * h, 4 * w):
                raise PaellaB200Error(f"decode_composite: orig has shape {tuple(orig.shape)}, expected {(B, 3, 4 * h, 4 * w)}")
            if tuple(pixel_mask.shape) not in ((B, 4 * h, 4 * w), (4 * h, 4 * w)):
                raise PaellaB200Error(f"decode_composite: pixel_mask has shape {tuple(pixel_mask.shape)}, expected "
                                      f"{(B, 4 * h, 4 * w)} or {(4 * h, 4 * w)}")
            orig = orig.to(device=dev, dtype=torch.float32).contiguous()
            pm = pixel_mask.to(device=dev).bool().expand(B, 4 * h, 4 * w).to(torch.uint8).contiguous()
            if mode == _lib.IMG_U8_NHWC:
                img = torch.empty(B, 4 * h, 4 * w, 3, dtype=torch.uint8, device=dev)
            else:
                img = torch.empty(B, 3, 4 * h, 4 * w, dtype=torch.float32, device=dev)
            ws = self._ws(L.pb200_vqgan_workspace_bytes(self._handle, B, 4 * h, 4 * w))
            check(L.pb200_vqgan_decode_composite(self._handle, ptr(idx), B, h, w, ptr(orig), ptr(pm), ptr(img), mode, ptr(ws),
                                                 ws.numel(), current_stream()), "pb200_vqgan_decode_composite")
        return img

    def forward(self, x, quantize=False):
        qe, x, _, vq_loss = self.encode(x, quantize)
        return self.decode(qe), vq_loss
