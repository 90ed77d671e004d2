"""Pin the oracle to the reference at the reference-default size (1.008 B denoiser, f4 VQGAN).

tests/golden/reference_default.npz holds what the unmodified reference computed (tests/golden/make_golden.py). The weights
(this package's CPU parameter holders share the reference's constructors and initialisation) and the float inputs are
re-created here from the same seeds and checked against the fingerprints stored with the outputs; the denoiser's 8.4 M
logits are compared on a seeded sample and through their per-channel and per-position means."""
import numpy as np
import pytest
import torch

from helpers import load_golden, t

TOL = dict(rtol=1e-3, atol=2e-5)


@pytest.fixture(scope="module")
def golden():
    return load_golden("reference_default.npz")[2]


def _check_fingerprint(g, prefix, tensors):
    assert [str(k) for k in g[prefix + "keys"]] == list(tensors), f"{prefix}: names differ from the fixture's"
    ts = [v.detach().double() for v in tensors.values()]
    np.testing.assert_allclose([float(v.sum()) for v in ts], g[prefix + "sum"], rtol=1e-7, atol=1e-6, err_msg=prefix)
    np.testing.assert_allclose([float(v.pow(2).sum()) for v in ts], g[prefix + "sumsq"], rtol=1e-7, err_msg=prefix)


def test_default_denoiser_forward(golden):
    from oracle import paella_oracle as po
    from paella_b200.modules import Paella
    from paella_b200.synth import rerandomize_, synthetic_conditioning
    g = golden
    torch.manual_seed(0)
    with torch.no_grad():
        m = Paella(byt5_embd=2560).eval()
        rerandomize_(m.state_dict(), seed=0)
        assert sum(p.numel() for p in m.parameters()) == 1008350592
        sd = m.state_dict()
        _check_fingerprint(g, "denoiser_sd_", sd)
        cond, _ = synthetic_conditioning(1, 16, with_clip_image=True)
        _check_fingerprint(g, "cond_", cond)
        x, r = t(g["x"]).long(), t(g["r"])
        got = po.paella_forward(sd, po.PaellaConfig(byt5_embd=2560), x, r, cond["byt5"], cond["clip"], cond["clip_image"])
    assert tuple(got.shape) == tuple(int(s) for s in g["logits_shape"])
    assert float(g["logits_std"]) > 0.05          # re-randomised: logits are not identically zero (SURVEY F3)
    assert abs(float(got.std()) - float(g["logits_std"])) <= 1e-3 * float(g["logits_std"])
    torch.testing.assert_close(got.reshape(-1)[t(g["logits_idx"]).long()], t(g["logits_sample"]), **TOL)
    torch.testing.assert_close(got.mean((0, 2, 3)), t(g["logits_channel_mean"]), **TOL)
    torch.testing.assert_close(got.mean(1).reshape(-1), t(g["logits_position_mean"]), **TOL)


def test_default_vqgan_conv_stacks(golden):
    from oracle import vqgan_oracle as vo
    from paella_b200.synth import rerandomize_
    from paella_b200.vqgan import VQModel
    g = golden
    torch.manual_seed(0)
    with torch.no_grad():
        vq = VQModel().eval()
        rerandomize_(vq.state_dict(), seed=4)
        sd = vq.state_dict()
        _check_fingerprint(g, "vqgan_sd_", sd)
        img = torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(7))
        _check_fingerprint(g, "vq_img_", {"img": img})
        torch.testing.assert_close(vo.encode_latents(sd, img).permute(0, 3, 1, 2), t(g["vq_latents"]), **TOL)
        torch.testing.assert_close(vo.decode_indices(sd, t(g["vq_idx"]).long()), t(g["vq_dec_indices"]), **TOL)
