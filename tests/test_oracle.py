"""CPU tests that pin the oracle (spec ③): reference DPT class output, scheduler collapse,
published parameter counts, text-embed fixture, committed end-to-end goldens."""
import os

import numpy as np
import pytest
import torch

from genpercept_b200 import weights as W


def test_param_counts_match_published_sizes():
    assert abs(W.param_count(W.unet_spec()) / 1e6 - 865.9) < 0.05      # SD-2.1 UNet
    assert abs(W.param_count(W.vae_spec()) / 1e6 - 83.65) < 0.01       # SD VAE
    assert abs(W.param_count(W.dpt_spec()) / 1e6 - 18.47) < 0.01       # dpt_head.py head


def test_oracle_state_dict_keys_equal_spec():
    from oracle.dpt import DPTNeckHeadIdentity
    from oracle.unet import UNet2DConditionModel
    from oracle.vae import AutoencoderKL
    for mod, spec in ((UNet2DConditionModel(), W.unet_spec()), (AutoencoderKL(), W.vae_spec()),
                      (DPTNeckHeadIdentity(), W.dpt_spec())):
        sd = mod.state_dict()
        assert set(sd.keys()) == set(spec.keys())
        for k, (shape, _) in spec.items():
            assert tuple(sd[k].shape) == tuple(shape), k


def test_scheduler_collapses_to_minus_v():
    """SURVEY.md F7: beta=1 => alphas_cumprod = 0 => x0 = -v, timesteps == [1]."""
    from oracle.scheduler import DDIMOneStep
    s = DDIMOneStep()
    assert float(s.alphas_cumprod.max()) == 0.0
    ts = s.set_timesteps(1)
    assert ts.tolist() == [1]
    g = torch.Generator().manual_seed(0)
    v = torch.randn((2, 4, 8, 8), generator=g)
    x = torch.randn((2, 4, 8, 8), generator=g)
    _, x0 = s.step(v, ts[0], x)
    assert torch.equal(x0, -v)


def test_text_embed_fixture(golden_dir):
    e = np.load(os.path.join(golden_dir, "empty_text_embed_2x1024.npy"))
    assert e.shape == (2, 1024) and e.dtype == np.float16
    assert np.isfinite(e.astype(np.float32)).all()


def test_dpt_oracle_equals_reference_class(synth_state, golden_dir):
    """The golden was produced by the reference's own DPTNeckHeadForUnetAfterUpsampleIdentity
    (tests/golden/make_golden.py) on the same seeded weights and features."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk", os.path.join(golden_dir, "make_golden.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    from oracle.dpt import DPTNeckHeadIdentity
    m = DPTNeckHeadIdentity().eval()
    m.load_state_dict(synth_state["dpt"], strict=True)
    with torch.no_grad():
        out = m(mk.dpt_features(8)).numpy()
    ref = np.load(os.path.join(golden_dir, "dpt_ref_h8.npz"))["out"]
    assert out.shape == ref.shape
    np.testing.assert_allclose(out, ref, rtol=0, atol=2e-5)


def test_oracle_e2e_matches_committed_golden(synth_state, text_embed, golden_dir):
    from oracle.pipeline import OraclePipeline
    g = np.load(os.path.join(golden_dir, "oracle_e2e_64.npz"))
    x = torch.from_numpy(g["rgb"]).float() / 255.0 * 2.0 - 1.0
    p = OraclePipeline(synth_state, text_embed, use_dpt=False)
    y, inter = p.single_infer(x, mode="depth", return_intermediates=True)
    np.testing.assert_allclose(inter["rgb_latent"].numpy(), g["rgb_latent"], atol=1e-4)
    np.testing.assert_allclose(inter["unet_out"].numpy(), g["unet_out"], atol=5e-4)
    np.testing.assert_allclose(y.numpy(), g["depth"], atol=5e-4)
    assert 0.1 < float(y.std()) and float(y.min()) >= 0 and float(y.max()) <= 1   # not degenerate
    p = OraclePipeline(synth_state, text_embed, use_dpt=True)
    np.testing.assert_allclose(p.single_infer(x, mode="depth").numpy(), g["dpt"], atol=5e-4)


def test_cross_attention_two_token_closed_form(synth_state, text_embed):
    """SURVEY.md F6: attn2 over a 2-token context == c0 + sigmoid(x.U) M (what the engine runs)."""
    from oracle.blocks import Attention
    c, heads = 320, 5
    a = Attention(c, heads, 64, cross_attention_dim=1024).eval()
    p = "down_blocks.0.attentions.0.transformer_blocks.0.attn2."
    a.load_state_dict({k[len(p):]: v for k, v in synth_state["unet"].items() if k.startswith(p)})
    g = torch.Generator().manual_seed(3)
    x = torch.randn((2, 50, c), generator=g)
    with torch.no_grad():
        ref = a(x, text_embed.repeat(2, 1, 1))
        e = text_embed[0]
        K, V = e @ a.to_k.weight.T, e @ a.to_v.weight.T            # [2, C]
        Wq, Wo, bo = a.to_q.weight, a.to_out[0].weight, a.to_out[0].bias
        dK = (K[0] - K[1]).view(heads, 64)
        U = torch.einsum("hdc,hd->ch", Wq.view(heads, 64, c), dK) / 8.0      # [C, heads]
        dV = torch.zeros(heads, c)
        for h in range(heads):
            dV[h] = (V[0] - V[1])[h * 64:(h + 1) * 64] @ Wo[:, h * 64:(h + 1) * 64].T
        c0 = V[1] @ Wo.T + bo
        out = c0 + torch.sigmoid(x @ U) @ dV
    torch.testing.assert_close(out, ref, atol=2e-5, rtol=1e-4)


def test_upsample2d_matches_the_reference_vendored_class(golden_dir):
    """genpercept/models/dpt_head.py:92-210 in the reference vendors diffusers' ``Upsample2D`` — the one block of the
    UNet / VAE graphs whose source IS in the reference tree.  oracle.blocks.Upsample2D (used by every up block of both
    graphs) must match it bit for bit, including the explicit-size path diffusers takes when a level has an odd extent.
    The reference's results are stored as digests (tests/golden/make_golden_reference.py); input and weights are
    integer-valued, so the float32 result is exact on any machine."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mkref", os.path.join(golden_dir, "make_golden_reference.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    ref = np.load(os.path.join(golden_dir, "reference_glue.npz"))
    from oracle.blocks import Upsample2D
    x, w, b = mk.upsample_case()
    mine = Upsample2D(24).eval()
    mine.conv.load_state_dict({"weight": w, "bias": b})
    with torch.no_grad():
        for size in mk.UPSAMPLE_SIZES:
            y = mine(x) if size is None else mine(x, size)
            key = "none" if size is None else f"{size[0]}x{size[1]}"
            assert tuple(y.shape) == tuple(ref[f"upsample_{key}_shape"]), key
            assert mk.digest(y) == str(ref[f"upsample_{key}_sha256"]), key
