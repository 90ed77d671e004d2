"""Masked sampling (inpainting / outpainting) on the GPU: the sparse fused sampler against the dense one, the masked loop's
identities, per-step parity with the oracle's masked loop, outpainting geometries, the compositing decoder tail and the
editing wrappers."""
import json

import pytest
import torch

from helpers import load_golden, t
from masked_oracle import token_masks

pytestmark = pytest.mark.gpu
DEV = "cuda"
MAX_ABS_D = 2.5e-3          # asserted logits tolerance of the default model (tests/test_gpu_model.py)


def _log(name, payload):
    """Measured agreement figures, one JSON line on stdout (shown with `pytest -s`)."""
    print(json.dumps({"test": name, **payload}))


def _gen():
    return torch.cuda.default_generators[torch.cuda.current_device()]


# ---------------------------------------------------------------------------------------------- sparse sampler
@pytest.mark.parametrize("NL,B,H", [(8192, 8, 32), (8192, 3, 8), (8200, 2, 16), (64, 2, 8), (8192, 64, 32), (8192, 128, 32)])
def test_masked_sampler_equals_dense_sampler(NL, B, H):
    """sample_tokens_masked(known, mask) == where(mask, sample_tokens(...), known) bit for bit, and the generator ends at the
    same offset.  Shapes: shared-Philox kernel with a full and a partial last block, the small-grid policies, the generic
    8200-label kernel, exactly 2^29 elements (bs 64) and a split draw (bs 128, two kernels)."""
    from paella_b200.modules import Paella
    cfg, sd, g = load_golden("paella_tiny.npz")
    big = dict(cfg)
    big.update(c_in=256, c_out=256, num_labels=NL)
    torch.manual_seed(0)
    m = Paella(**big).to(DEV).eval()
    gen = torch.Generator(device=DEV).manual_seed(3)
    feats = torch.randn(2 * B * H * H, 256, device=DEV, generator=gen)
    W = m.out_mapper[1].weight.detach().view(NL, 256) * 30.0        # spread the logits
    with torch.no_grad():
        m.out_mapper[1].weight.copy_(W.view(NL, 256, 1, 1))
    m.pack_weights()
    n = B * H * H
    known = torch.randint(0, NL, (B, H, H), device=DEV, generator=gen)
    masks = token_masks(B, H, H, seed=NL + B)
    for cfg_s, f in ((8.0, feats), (None, feats[:n].contiguous())):
        torch.manual_seed(42)
        dense = m.sample_tokens(f, B, H, H, cfg_s, 0.7)
        off = _gen().get_offset()
        for name, mk in masks.items():
            mk = mk.to(DEV)
            torch.manual_seed(42)
            got = m.sample_tokens_masked(f, B, H, H, cfg_s, 0.7, known, mk)
            assert _gen().get_offset() == off, (name, cfg_s)
            assert torch.equal(got, torch.where(mk, dense, known)), (NL, B, H, name, cfg_s)
    # a [H,W] mask given as uint8 broadcasts over the batch
    torch.manual_seed(42)
    got = m.sample_tokens_masked(feats, B, H, H, 8.0, 0.7, known, masks["rect"][0].to(DEV).to(torch.uint8).expand(B, H, H))
    torch.manual_seed(42)
    assert torch.equal(got, torch.where(masks["rect"].to(DEV), m.sample_tokens(feats, B, H, H, 8.0, 0.7), known))


# ---------------------------------------------------------------------------------------------- loop identities
@pytest.fixture(scope="module")
def tiny():
    from paella_b200.modules import Paella
    cfg, sd, g = load_golden("paella_tiny.npz")
    m = Paella(**cfg).to(DEV).eval()
    m.load_state_dict(sd)
    return m, cfg, sd, g


@pytest.fixture(scope="module")
def default_model():
    from paella_b200.modules import Paella
    from paella_b200.synth import rerandomize_
    torch.manual_seed(0)
    m = Paella(byt5_embd=2560).eval()
    rerandomize_(m.state_dict(), seed=0)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    return m.to(DEV), sd


def _check_identities(m, K, cond, uncond, B, H, W, steps, vq=None):
    from paella_b200 import utils as U
    known = torch.randint(0, K, (B, H, W), device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    kw = dict(steps=steps, temperature=(1.0, 0.3), cfg=(6.0, 4.0))
    # mask == 1: the notebook loop, bit for bit, tokens and every intermediate
    for exact in (False, True):
        torch.manual_seed(11)
        a, ia = U.sample_notebook(m, cond, (B, H, W), uncond, exact=exact, **kw)
        off = _gen().get_offset()
        torch.manual_seed(11)
        b, ib = U.sample_masked(m, cond, known, torch.ones(H, W, dtype=torch.bool), uncond, exact=exact, **kw)
        assert _gen().get_offset() == off
        assert torch.equal(a, b) and len(ia) == len(ib) and all(torch.equal(x, y) for x, y in zip(ia, ib)), exact
    # mask == 0: known throughout, same generator consumption
    torch.manual_seed(12)
    c, ic = U.sample_masked(m, cond, known, torch.zeros(B, H, W, dtype=torch.bool), uncond, **kw)
    assert _gen().get_offset() == off
    assert torch.equal(c, known) and all(torch.equal(x, known) for x in ic)
    # a partial mask: kept tokens never change, in every mode
    mk = token_masks(B, H, W, seed=5)["random30"].to(DEV)
    modes = [("multinomial", False), ("multinomial", True), ("argmax", False)] + ([("quant", False)] if vq is not None else [])
    for mode, exact in modes:
        torch.manual_seed(13)
        d, idd = U.sample_masked(m, cond, known, mk, uncond, mode=mode, exact=exact, vqmodel=vq, **kw)
        for x in [d] + idd:
            assert torch.equal(x[~mk], known[~mk]), (mode, exact)
        assert bool((d[mk] != known[mk]).any()), (mode, exact)         # and the masked ones were resampled


def test_masked_loop_identities_tiny(tiny):
    from paella_b200.vqgan import VQModel
    m, cfg, sd, g = tiny
    byt5, clip = t(g["byt5"]).to(DEV), t(g["clip"]).to(DEV)
    cond = {"byt5": byt5, "clip": clip}
    uncond = {"byt5": torch.zeros_like(byt5), "clip": torch.zeros_like(clip)}
    vq = VQModel(levels=2, bottleneck_blocks=1, c_hidden=32, c_latent=4, codebook_size=cfg["num_labels"]).to(DEV)
    _check_identities(m, cfg["num_labels"], cond, uncond, 2, 8, 8, 4, vq)


def test_masked_loop_identities_default_32(default_model):
    from paella_b200.synth import synthetic_conditioning
    m, _ = default_model
    cond, uncond = synthetic_conditioning(1, 32, device=DEV)
    _check_identities(m, 8192, cond, uncond, 1, 32, 32, 3)


# ---------------------------------------------------------------------------------------------- parity with the oracle
def _oracle_step(po, sd, oc, tokens, t_, cond, uncond, cfg, temp, q):
    B = tokens.shape[0]
    r = torch.full((B,), t_)
    lc = po.paella_forward(sd, oc, tokens, r, **cond)
    lg = lc * cfg + po.paella_forward(sd, oc, tokens, r, **uncond) * (1 - cfg)
    K = lg.shape[1]
    flat = lg.permute(0, 2, 3, 1).reshape(-1, K)
    p = flat.div(temp).softmax(dim=-1)
    return torch.argmax(p / q, dim=-1).view(tokens.shape), flat


def test_masked_default_vs_oracle_per_step_with_margin_audit(default_model):
    """Reference-default 1.008 B model, bs 1, 32x32, 8-step CFG, a 16x16 centre mask: every step run on the GPU from the
    oracle's masked state (teacher forcing) with the generator where the loop has it.  Masked positions agree >= 99 % over
    the 8 x 256 masked draws, every mismatch is a Gumbel-score near-tie within what the logits tolerance allows, and kept
    positions equal `known` at every step.  The oracle side is the masked loop of tests/masked_oracle.py applied step by
    step (start state, merge after the draw, renoise).  Measured on B200: 2 near-ties (score gap 0.004) at the T = 0.31 step, 100 %
    elsewhere; the agreement floor is on the total because 256 draws per step leave no room for a third tie in one step."""
    from oracle import paella_oracle as po
    from paella_b200.synth import synthetic_conditioning
    m, sd = default_model
    oc = po.PaellaConfig(byt5_embd=2560)
    B, H, K, steps, renoise, cfg = 1, 32, 8192, 8, 7, 8.0
    cond, uncond = synthetic_conditioning(B, 128)
    cache = m.prepare_conditioning([{k: v.to(DEV) for k, v in cond.items()}, {k: v.to(DEV) for k, v in uncond.items()}], (H, H))
    t_list = torch.linspace(1.0, 0.0, steps + 1)
    temps = torch.linspace(1.0, 0.2, steps)
    known = torch.randint(0, K, (B, H, H), generator=torch.Generator().manual_seed(4))
    mask = torch.zeros(H, H, dtype=torch.bool)
    mask[8:24, 8:24] = True
    mb = mask.expand(B, H, H)
    torch.manual_seed(20261017)
    gen = _gen()
    init = torch.randint(0, K, (B, H, H), device=DEV).cpu()
    offs_q, qs, us = [], [], []
    for i in range(steps):
        offs_q.append(gen.get_offset())
        qs.append(torch.empty(B * H * H, K, device=DEV).exponential_(1).cpu())
        if i < renoise:
            us.append(torch.rand(B, H, H, device=DEV).cpu())
    init_noise = torch.where(mb, init, known)
    state = init_noise.clone()
    per_step, n_agree, n_masked = [], 0, 0
    with torch.inference_mode():
        for i in range(steps):
            tt, temp = float(t_list[i]), float(temps[i])
            want, flat = _oracle_step(po, sd, oc, state, tt, cond, uncond, cfg, temp, qs[i])
            want = torch.where(mb, want, known)
            gen.set_offset(offs_q[i])
            feats = m.features(state.to(DEV), torch.full((B,), tt, device=DEV), cache, cfg_pairs=True)
            got = m.sample_tokens_masked(feats, B, H, H, cfg, temp, known.to(DEV), mb.to(DEV)).cpu()
            assert torch.equal(got[~mb], known[~mb])
            agree = float((got[mb] == want[mb]).float().mean())
            n_agree, n_masked = n_agree + int((got[mb] == want[mb]).sum()), n_masked + int(mb.sum())
            bad = (got != want).view(-1).nonzero().flatten()
            gap = 0.0
            if bad.numel():
                score = flat[bad].double() / temp - torch.log(qs[i][bad].double())
                gap = float((score.gather(1, want.view(-1)[bad][:, None]) - score.gather(1, got.view(-1)[bad][:, None])).max())
            bound = 2 * (abs(cfg) + abs(1 - cfg)) * MAX_ABS_D / temp
            per_step.append({"step": i, "T": temp, "agree_masked": agree, "mismatches": int(bad.numel()), "worst_gap": gap,
                             "gap_bound": bound})
            assert gap <= bound, per_step[-1]
            state = want
            if i < renoise:
                state, _ = po.add_noise(state, torch.full((B,), float(t_list[i + 1])), init_noise, us[i])
    _log("masked_default_vs_oracle", {"per_step": per_step, "agree_masked_total": n_agree / n_masked})
    assert n_agree / n_masked >= 0.99, per_step


# ---------------------------------------------------------------------------------------------- outpainting geometry
@pytest.mark.parametrize("canvas", [(48, 48), (32, 64)])
def test_outpaint_geometry_fused_vs_exact_per_step(default_model, canvas):
    """A 32x32-token image in a 48x48 and a 32x64 token canvas (shapes off the square attention fast path).  Each step from
    the same state: the fused masked draw vs the exact path (materialised logits, torch-op draw, then the merge) -- >= 99 %
    agreement on the regenerated tokens; the image's tokens stay intact in the free-running loop."""
    from paella_b200 import ops
    from paella_b200 import utils as U
    from paella_b200.synth import synthetic_conditioning
    m, _ = default_model
    CH, CW = canvas
    B, K, cfg, temp = 1, 8192, 6.0, 0.7
    cond, uncond = synthetic_conditioning(B, 32, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(21)
    known = torch.randint(0, K, (B, CH, CW), device=DEV, generator=g)
    mask = torch.ones(CH, CW, dtype=torch.bool, device=DEV)
    oy, ox = (CH - 32) // 2, (CW - 32) // 2
    mask[oy:oy + 32, ox:ox + 32] = False
    mb = mask.expand(B, CH, CW)
    cache = m.prepare_conditioning([cond, uncond], (CH, CW))
    state = known.clone()
    agrees = []
    with torch.inference_mode():
        for i, tt in enumerate((1.0, 0.6, 0.2)):
            state = torch.where(mb, torch.randint(0, K, (B, CH, CW), device=DEV, generator=g), known) if i == 0 else state
            feats = m.features(state, torch.full((B,), tt, device=DEV), cache, cfg_pairs=True)
            off = _gen().get_offset()
            fused = m.sample_tokens_masked(feats, B, CH, CW, cfg, temp, known, mb)
            _gen().set_offset(off)
            n = B * CH * CW
            lc = m.logits_from_features(feats[:n], B, CH, CW)
            lu = m.logits_from_features(feats[n:], B, CH, CW)
            exact = torch.where(mb, ops.resample_logits(lc, lu, cfg, temp), known)
            assert torch.equal(fused[~mb], known[~mb])
            agrees.append(float((fused[mb] == exact[mb]).float().mean()))
            assert agrees[-1] >= 0.99, (canvas, i, agrees)
            state = exact
    torch.manual_seed(3)
    toks, inter = U.sample_masked(m, cond, known, mask, uncond, steps=4, temperature=(1.0, 0.3))
    assert toks.shape == (B, CH, CW)
    assert all(torch.equal(x[:, oy:oy + 32, ox:ox + 32], known[:, oy:oy + 32, ox:ox + 32]) for x in [toks] + inter)
    _log("outpaint_geometry", {"canvas": list(canvas), "agree": agrees})


# ---------------------------------------------------------------------------------------------- compositing decoder
def _u8(img):
    """torchvision save_image's byte conversion of fp32 NCHW -> uint8 NHWC (after the decoder's clamp)."""
    return img.clamp(0, 1).mul(255).add_(0.5).clamp_(0, 255).permute(0, 2, 3, 1).to(torch.uint8)


@pytest.mark.parametrize("which,h,w", [("default", 32, 32), ("tiny", 6, 9)])
def test_decode_composite_matches_torch_composition(which, h, w):
    """decode_composite == where(pixel_mask, decode, orig) through the same conversion, bit for bit: 128x128 px on the
    reference codec (thread-per-position writer) and 24x36 px on the tiny golden codec (warp-per-position writer)."""
    from paella_b200.synth import rerandomize_
    from paella_b200.vqgan import VQModel
    if which == "default":
        torch.manual_seed(0)
        vq = VQModel().eval()
        rerandomize_(vq.state_dict(), seed=4)
        vq = vq.to(DEV)
    else:
        cfg, sd, _ = load_golden("vqgan_tiny.npz")
        vq = VQModel(**cfg).to(DEV).eval()
        vq.load_state_dict(sd)
    K = vq.vquantizer.codebook.weight.shape[0]
    g = torch.Generator(device=DEV).manual_seed(6)
    B = 2
    idx = torch.randint(0, K, (B, h, w), device=DEV, generator=g)
    orig = torch.rand(B, 3, 4 * h, 4 * w, device=DEV, generator=g) * 1.4 - 0.2          # outside [0,1] too: the clamp matters
    pm = torch.rand(B, 4 * h, 4 * w, device=DEV, generator=g) < 0.5
    raw = vq.decode_indices(idx)
    m3 = pm[:, None]
    assert torch.equal(vq.decode_composite(idx, orig, pm, "raw"), torch.where(m3, raw, orig))
    assert torch.equal(vq.decode_composite(idx, orig, pm, "clamp"), torch.where(m3, raw.clamp(0, 1), orig.clamp(0, 1)))
    u8 = vq.decode_composite(idx, orig, pm, "uint8")
    assert u8.dtype == torch.uint8 and u8.shape == (B, 4 * h, 4 * w, 3)
    assert torch.equal(u8, torch.where(pm[..., None], vq.decode_indices_u8(idx), _u8(orig)))
    # a [H,W] mask broadcasts over the batch
    assert torch.equal(vq.decode_composite(idx, orig, pm[0], "uint8"),
                       torch.where(pm[0][None, ..., None], vq.decode_indices_u8(idx), _u8(orig)))


# ---------------------------------------------------------------------------------------------- editing wrappers
def test_inpaint_and_outpaint_end_to_end(tiny):
    from paella_b200 import editing
    from paella_b200.vqgan import VQModel
    m, cfg, sd, g = tiny
    vcfg, vsd, _ = load_golden("vqgan_tiny.npz")
    vq = VQModel(**vcfg).to(DEV).eval()
    vq.load_state_dict(vsd)
    byt5, clip = t(g["byt5"]).to(DEV), t(g["clip"]).to(DEV)
    cond = {"byt5": byt5, "clip": clip}
    B = byt5.shape[0]
    gi = torch.Generator(device=DEV).manual_seed(8)
    img = torch.rand(B, 3, 32, 32, device=DEV, generator=gi)
    pm = torch.zeros(32, 32, dtype=torch.bool, device=DEV)
    pm[9:21, 5:30] = True
    kw = dict(steps=3, temperature=(1.0, 0.3))
    out = editing.inpaint(m, vq, img, pm, cond, **kw)
    assert out.shape == (B, 32, 32, 3) and out.dtype == torch.uint8
    assert torch.equal(out[:, ~pm], _u8(img)[:, ~pm])
    assert editing.inpaint(m, vq, img, pm, cond, output="clamp", **kw).shape == (B, 3, 32, 32)
    assert editing.inpaint(m, vq, img, pm, cond, output="raw", paste_back=False, **kw).dtype == torch.float32
    toks = editing.inpaint(m, vq, img, pm, cond, output="tokens", **kw)
    known = vq.encode(img)[2]
    tm = editing.token_mask(pm)
    assert toks.shape == (B, 8, 8) and toks.dtype == torch.int64 and torch.equal(toks[:, ~tm], known[:, ~tm])
    # outpaint: a 32x32 px image at (0, 16) on a 32x64 px canvas
    out = editing.outpaint(m, vq, img, (32, 64), (0, 16), cond, **kw)
    assert out.shape == (B, 32, 64, 3) and out.dtype == torch.uint8
    assert torch.equal(out[:, :, 16:48], _u8(img))
    toks = editing.outpaint(m, vq, img, (32, 64), (0, 16), cond, output="tokens", **kw)
    assert toks.shape == (B, 8, 16) and torch.equal(toks[:, :, 4:12], known)
