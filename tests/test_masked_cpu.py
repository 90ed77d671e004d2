"""Masked sampling without a GPU: the masked oracle loop, the editing wrappers' geometry checks and the pixel -> token
mask rule."""
import pytest
import torch
import torch.nn.functional as F

import masked_oracle as mo
from helpers import load_golden, oracle_cfg, t
from masked_oracle import token_masks


@pytest.fixture(scope="module")
def tiny_oracle():
    cfg, sd, g = load_golden("paella_tiny.npz")
    oc = oracle_cfg(cfg)
    B, H, K, steps = 2, 8, cfg["num_labels"], 3
    gen = torch.Generator().manual_seed(7)
    draws = {"init": torch.randint(0, K, (B, H, H), generator=gen),
             "q": [torch.empty(B * H * H, K).exponential_(1, generator=gen) for _ in range(steps)],
             "u": [torch.rand(B, H, H, generator=gen) for _ in range(steps - 1)]}
    byt5, clip = t(g["byt5"]), t(g["clip"])
    args = (sd, oc, {"byt5": byt5, "clip": clip}, (B, H, H), {"byt5": torch.zeros_like(byt5), "clip": torch.zeros_like(clip)})
    kw = dict(steps=steps, renoise_steps=steps - 1, temperature=(1.0, 0.3), cfg_scale=4.0, draws=draws)
    known = torch.randint(0, K, (B, H, H), generator=gen)
    return args, kw, known


def test_masked_oracle_all_ones_mask_is_the_unmasked_loop(tiny_oracle):
    from oracle import paella_oracle as po
    args, kw, known = tiny_oracle
    want = po.sample(*args, **kw)
    assert torch.equal(mo.sample(*args, known, torch.ones(known.shape, dtype=torch.bool), **kw), want)
    assert torch.equal(mo.sample(*args, known, torch.ones(known.shape[1:], dtype=torch.uint8), **kw), want)


def test_masked_oracle_all_zeros_mask_returns_known(tiny_oracle):
    args, kw, known = tiny_oracle
    assert torch.equal(mo.sample(*args, known, torch.zeros(known.shape, dtype=torch.bool), **kw), known)


def test_masked_oracle_partial_mask_keeps_known(tiny_oracle):
    args, kw, known = tiny_oracle
    mk = token_masks(*known.shape, seed=1)["rect"]
    out = mo.sample(*args, known, mk, **kw)
    assert torch.equal(out[~mk], known[~mk])
    assert bool((out[mk] != known[mk]).any())


@pytest.fixture(scope="module")
def tiny_model():
    from paella_b200.modules import Paella
    cfg, _, _ = load_golden("paella_tiny.npz")
    return Paella(**cfg).eval()          # only its configuration is read: every check runs before a launch


def test_latent_multiple_of_the_tiny_model(tiny_model):
    from paella_b200 import editing
    assert editing.latent_multiple(tiny_model) == 8          # patch_size 2, three levels: 2 << 2


@pytest.mark.parametrize("case", ["latent_not_multiple", "image_not_multiple_of_4", "mask_shape", "not_nchw", "output"])
def test_inpaint_rejects_bad_geometry(tiny_model, case):
    from paella_b200 import editing
    from paella_b200._lib import PaellaB200Error
    img, pm, kw = torch.rand(2, 3, 32, 32), torch.ones(32, 32, dtype=torch.bool), {}
    if case == "latent_not_multiple":
        img, pm = torch.rand(2, 3, 40, 40), torch.ones(40, 40, dtype=torch.bool)       # 10x10 tokens, needs a multiple of 8
    elif case == "image_not_multiple_of_4":
        img, pm = torch.rand(2, 3, 30, 32), torch.ones(30, 32, dtype=torch.bool)
    elif case == "mask_shape":
        pm = torch.ones(3, 32, 32, dtype=torch.bool)
    elif case == "not_nchw":
        img = torch.rand(2, 32, 32, 3)
    else:
        kw = {"output": "png"}
    with pytest.raises(PaellaB200Error):
        editing.inpaint(tiny_model, None, img, pm, {}, **kw)


@pytest.mark.parametrize("case,img_hw,canvas,offset", [
    ("canvas_latent_not_multiple", (32, 32), (40, 64), (0, 0)),
    ("canvas_not_multiple_of_4", (32, 32), (32, 66), (0, 0)),
    ("offset_not_multiple_of_4", (32, 32), (32, 64), (0, 2)),
    ("image_not_multiple_of_4", (30, 32), (32, 64), (0, 0)),
    ("does_not_fit", (32, 32), (32, 64), (0, 40)),
    ("negative_offset", (32, 32), (32, 64), (-4, 0)),
])
def test_outpaint_rejects_bad_geometry(tiny_model, case, img_hw, canvas, offset):
    from paella_b200 import editing
    from paella_b200._lib import PaellaB200Error
    with pytest.raises(PaellaB200Error):
        editing.outpaint(tiny_model, None, torch.rand(1, 3, *img_hw), canvas, offset, {})


def test_sample_masked_rejects_mask_shape(tiny_model):
    from paella_b200 import utils as U
    from paella_b200._lib import PaellaB200Error
    with pytest.raises(PaellaB200Error):
        U.sample_masked(tiny_model, {}, torch.zeros(2, 8, 8, dtype=torch.int64), torch.ones(8, 16, dtype=torch.bool))
    with pytest.raises(PaellaB200Error):
        U.sample_masked(tiny_model, {}, torch.zeros(8, 8, dtype=torch.int64), torch.ones(8, 8, dtype=torch.bool))


@pytest.mark.parametrize("shape", [(2, 32, 48), (64, 16)])
def test_token_mask_is_any_pixel_of_the_4x4_block(shape):
    from paella_b200 import editing
    g = torch.Generator().manual_seed(3)
    pm = torch.rand(shape, generator=g) < 0.02                  # sparse: many blocks empty, many with a single pixel
    want = F.max_pool2d(pm.float().reshape(-1, 1, *shape[-2:]), 4).reshape(*shape[:-2], shape[-2] // 4, shape[-1] // 4) > 0
    got = editing.token_mask(pm)
    assert got.dtype == torch.bool and torch.equal(got, want)
    assert bool(got.any()) and not bool(got.all())
