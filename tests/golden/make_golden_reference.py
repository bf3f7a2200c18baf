"""Regenerates tests/golden/reference_glue.npz: what the reference's own code computes around this repository's oracle
modules, so that tests/test_oracle_vs_reference_pipeline.py and tests/test_oracle.py can pin the oracle against it
without a checkout of the reference.

  python tests/golden/make_golden_reference.py <path to a GenPercept checkout>

The reference modules are imported through a minimal ``diffusers`` / ``matplotlib`` shim (base classes and type names
only: diffusers itself is not needed) and driven with the oracle's VAE / UNet / scheduler behind thin adapters, plus the
reference's own DPT head class.  Everything between those modules — latent scaling, the mean half of the moments, the
scheduler call and ``pred_original_sample``, ``/ scale`` + post_quant_conv + decoder, the channel mean, clip and shift,
the DPT feature order and min-max, the UNet's skip stack and ``upsample_size`` forwarding — is the reference's code.

The pipeline and UNet cases run in float64: the tests compare at 1e-6, and float32 CPU convolutions and GEMMs change
their summation order with the thread count and instruction set by more than that.  The Upsample2D case uses
integer-valued inputs and weights, so its float32 output is exact on any machine and the test can compare bit for bit.
"""
import hashlib
import importlib
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

UNET_SIZES = ((8, 8), (9, 11), (12, 10))       # multiples of 8, odd extents, 8 does not divide
FEATURE_SAMPLE = 512                           # seeded sample of each UNet feature map (the maps are up to 0.6 MB each)
UPSAMPLE_SIZES = (None, (13, 17), (14, 18), (13, 18))
RESIZE_EDGES = (64, 128, 200)


def digest(t):
    """sha256 of a tensor's or array's bytes: a bitwise comparison against the stored reference result."""
    a = t.numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def glue_input(seed=21):
    """32 x 32: the glue does not depend on the image size, and the stored maps stay small."""
    g = torch.Generator().manual_seed(seed)
    return torch.rand((1, 3, 32, 32), generator=g) * 2 - 1


def unet_inputs():
    g = torch.Generator().manual_seed(4)
    return [torch.randn((1, 4, h, w), generator=g) for h, w in UNET_SIZES]


def upsample_case():
    """Integer-valued input and conv weights: every product and partial sum is an exact float32 integer."""
    g = torch.Generator().manual_seed(3)
    x = torch.randint(-4, 5, (2, 24, 7, 9), generator=g).float()
    w = torch.randint(-2, 3, (24, 24, 3, 3), generator=g).float()
    b = torch.randint(-8, 9, (24,), generator=g).float()
    return x, w, b


def resize_case():
    g = torch.Generator().manual_seed(8)
    x = torch.randint(0, 256, (1, 3, 90, 160), generator=g, dtype=torch.uint8)
    c = torch.rand((3, 4, 5), generator=g)
    return x, c


def _install_shims(ref):
    import torch.nn as nn
    d = types.ModuleType("diffusers")

    class DiffusionPipeline:
        def __init__(self):
            self._cfg = {}

        def register_modules(self, **kw):
            for k, v in kw.items():
                setattr(self, k, v)

        def register_to_config(self, **kw):
            self._cfg.update(kw)

        @property
        def device(self):
            return torch.device("cpu")

        @property
        def dtype(self):
            return torch.float64

    for name in ("AutoencoderKL", "DDIMScheduler", "LCMScheduler", "DDPMScheduler"):
        setattr(d, name, type(name, (), {}))
    d.UNet2DConditionModel = type("UNet2DConditionModel", (nn.Module,), {})
    d.DiffusionPipeline = DiffusionPipeline
    du = types.ModuleType("diffusers.utils")
    du.BaseOutput = type("BaseOutput", (), {})
    du.USE_PEFT_BACKEND = True
    du.deprecate = lambda *a, **k: None
    du.logging = types.SimpleNamespace(get_logger=lambda *a, **k: None)
    du.scale_lora_layers = lambda *a, **k: None
    du.unscale_lora_layers = lambda *a, **k: None
    dm = types.ModuleType("diffusers.models")
    dl = types.ModuleType("diffusers.models.lora")
    dl.LoRACompatibleConv = nn.Conv2d
    unets = types.ModuleType("diffusers.models.unets")
    u2d = types.ModuleType("diffusers.models.unets.unet_2d_condition")
    u2d.UNet2DConditionOutput = type("UNet2DConditionOutput", (), {})
    cu = types.ModuleType("diffusers.configuration_utils")
    cu.ConfigMixin = type("ConfigMixin", (), {})
    cu.register_to_config = lambda f: f
    d.utils, d.models, dm.lora = du, dm, dl
    m = types.ModuleType("matplotlib")
    mp = types.ModuleType("matplotlib.pyplot")
    m.pyplot = mp
    sys.modules.update({"diffusers": d, "diffusers.utils": du, "diffusers.models": dm, "diffusers.models.lora": dl,
                        "diffusers.models.unets": unets, "diffusers.models.unets.unet_2d_condition": u2d,
                        "diffusers.configuration_utils": cu, "matplotlib": m, "matplotlib.pyplot": mp})
    sys.path.insert(0, ref)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


class _UNetAdapter:
    def __init__(self, unet):
        self.unet = unet

    def __call__(self, x, t, encoder_hidden_states=None, return_feature=False):
        t = torch.as_tensor(t).reshape(-1)[:1]
        out = self.unet(x, t, encoder_hidden_states, return_feature=return_feature)
        return types.SimpleNamespace(multi_level_feats=out) if return_feature else types.SimpleNamespace(sample=out)


class _SchedulerAdapter:
    beta_start = 1
    beta_end = 1

    def __init__(self, s):
        self.s = s

    def set_timesteps(self, n, device=None):
        self.timesteps = self.s.set_timesteps(n)

    def step(self, model_output, t, sample, generator=None):
        prev, x0 = self.s.step(model_output, int(t), sample)
        return types.SimpleNamespace(prev_sample=prev, pred_original_sample=x0)


def pipeline_glue(ref, state, te, res):
    """genpercept/genpercept_pipeline.py: single_infer / encode_rgb / decode_pred around the oracle's modules."""
    from oracle.pipeline import OraclePipeline
    mod = importlib.import_module("genpercept.genpercept_pipeline")
    rgb = glue_input().double()
    op = OraclePipeline(state, te, dtype=torch.float64)
    rp = mod.GenPerceptPipeline(unet=_UNetAdapter(op.unet), vae=op.vae, scheduler=_SchedulerAdapter(op.scheduler),
                                text_encoder=None, tokenizer=None, genpercept_pipeline=True)
    rp.text_embed = op.text_embed
    with torch.no_grad():
        for mode in ("depth", "normal"):
            rp.mode = mode
            res[f"glue_{mode}"] = rp.single_infer(rgb, 1, None, False).numpy()
        res["glue_encode_rgb"] = rp.encode_rgb(rgb).numpy()
        res["glue_normal_fix_timesteps_7"] = rp.single_infer(rgb, 1, None, False, fix_timesteps=7).numpy()
    # the UNet's own forward (genpercept/models/custom_unet.py) around the oracle's blocks
    unet_dataflow(ref, op.unet, te, res)
    del op, rp
    od = OraclePipeline(state, te, use_dpt=True, dtype=torch.float64)
    head_mod = sys.modules["genpercept.models.dpt_head"]
    # transformers >= 4.4x refuses ModelOutput subclasses that are not dataclasses; the reference's output container
    # (dpt_head.py:24-49, written for an older transformers) is replaced by a plain attribute bag — no arithmetic involved
    head_mod.DepthEstimatorOutput = lambda **kw: types.SimpleNamespace(**kw)
    from transformers import DPTConfig
    head = head_mod.DPTNeckHeadForUnetAfterUpsampleIdentity(
        DPTConfig.from_pretrained(f"{ref}/hf_configs/dpt-sd2.1-unet-after-upsample-general")).eval()
    head.load_state_dict(state["dpt"], strict=True)
    head.double()
    rd = mod.GenPerceptPipeline(unet=_UNetAdapter(od.unet), vae=od.vae, scheduler=_SchedulerAdapter(od.scheduler),
                                text_encoder=None, tokenizer=None, customized_head=head, genpercept_pipeline=True)
    rd.text_embed = od.text_embed
    rd.mode = "depth"
    with torch.no_grad():
        res["glue_dpt"] = rd.single_infer(rgb, 1, None, False).numpy()


def unet_dataflow(ref, ou, te, res):
    import torch.nn as nn
    mod = _load("ref_custom_unet", f"{ref}/genpercept/models/custom_unet.py")

    class Down(nn.Module):
        def __init__(self, blk, cross):
            super().__init__()
            self.blk, self.has_cross_attention = blk, cross

        def forward(self, hidden_states, temb, encoder_hidden_states=None, **kw):
            return self.blk(hidden_states, temb, encoder_hidden_states)

    class Mid(nn.Module):
        has_cross_attention = True

        def __init__(self, blk):
            super().__init__()
            self.blk = blk

        def forward(self, sample, emb, encoder_hidden_states=None, **kw):
            return self.blk(sample, emb, encoder_hidden_states)

    class Up(nn.Module):
        def __init__(self, blk):
            super().__init__()
            self.blk, self.has_cross_attention, self.resnets = blk, blk.attentions is not None, blk.resnets

        def forward(self, hidden_states, temb, res_hidden_states_tuple, encoder_hidden_states=None, upsample_size=None, **kw):
            return self.blk(hidden_states, res_hidden_states_tuple, temb, encoder_hidden_states, upsample_size)

    class TimeEmb(nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, t_emb, cond=None):
            return self.m(t_emb)

    ru = mod.CustomUNet2DConditionModel()
    ru.num_upsamplers = 3
    ru.config = types.SimpleNamespace(center_input_sample=False, class_embed_type=None, addition_embed_type=None,
                                      class_embeddings_concat=False, encoder_hid_dim_type=None)
    ru.class_embedding = ru.time_embed_act = ru.encoder_hid_proj = None
    ru.time_proj, ru.time_embedding = ou.time_proj, TimeEmb(ou.time_embedding)
    ru.conv_in, ru.conv_norm_out, ru.conv_act, ru.conv_out = ou.conv_in, ou.conv_norm_out, nn.SiLU(), ou.conv_out
    ru.down_blocks = nn.ModuleList([Down(b, i < 3) for i, b in enumerate(ou.down_blocks)])
    ru.mid_block = Mid(ou.mid_block)
    ru.up_blocks = nn.ModuleList([Up(b) for b in ou.up_blocks])
    ru.eval()
    ctx = te.double().reshape(1, -1, 1024)
    g = torch.Generator().manual_seed(5)
    for (h, w), x in zip(UNET_SIZES, unet_inputs()):
        with torch.no_grad():
            res[f"unet_{h}x{w}_sample"] = ru(x.double(), 1, ctx).sample.numpy()
            feats = ru(x.double(), torch.tensor([1]), ctx, return_feature=True).multi_level_feats
        assert len(feats) == 4
        for i, f in enumerate(feats):
            idx = torch.randperm(f.numel(), generator=g)[:FEATURE_SAMPLE]
            res[f"unet_{h}x{w}_feat{i}_shape"] = np.array(f.shape)
            res[f"unet_{h}x{w}_feat{i}_idx"] = idx.numpy().astype(np.int32)
            res[f"unet_{h}x{w}_feat{i}_val"] = f.reshape(-1)[idx].numpy()


def scheduler_constants(ref, res):
    """src/customized_modules/ddim.py (DDIMSchedulerCustomized.__init__) from hf_configs/scheduler_beta_1.0_1.0."""
    import json
    mod = _load("ref_ddim", f"{ref}/src/customized_modules/ddim.py")
    cfg = json.load(open(f"{ref}/hf_configs/scheduler_beta_1.0_1.0/scheduler_config.json"))
    s = mod.DDIMSchedulerCustomized(**{k: v for k, v in cfg.items() if not k.startswith("_") and k != "skip_prk_steps"})
    res["sched_betas"] = s.betas.numpy()
    res["sched_alphas_cumprod"] = s.alphas_cumprod.numpy()
    res["sched_final_alpha_cumprod"] = s.final_alpha_cumprod.numpy()
    res["sched_init_noise_sigma"] = np.array(float(s.init_noise_sigma))


def image_helpers(res):
    """genpercept/util/image_util.py: resize_max_res, get_tv_resample_method, chw2hwc."""
    r = importlib.import_module("genpercept.util.image_util")
    x, c = resize_case()
    for edge in RESIZE_EDGES:
        y = r.resize_max_res(x, edge)
        res[f"resize_{edge}_shape"] = np.array(y.shape)
        res[f"resize_{edge}_sha256"] = np.array(digest(y))
    for m in ("bilinear", "bicubic", "nearest"):
        res[f"resample_{m}"] = np.array(r.get_tv_resample_method(m).value)
    try:
        r.get_tv_resample_method("lanczos")
        raise AssertionError("the reference accepted 'lanczos'")
    except ValueError:
        pass
    res["chw2hwc_tensor"] = r.chw2hwc(c).numpy()
    res["chw2hwc_array"] = r.chw2hwc(c.numpy())


def upsample2d(ref, res):
    """genpercept/models/dpt_head.py vendors diffusers' Upsample2D (the scale-factor and explicit-size paths)."""
    sys.path.insert(0, HERE)
    import make_golden
    make_golden.REF = ref
    make_golden.load_reference_dpt()
    m = sys.modules["ref_dpt_head"].Upsample2D(24, use_conv=True).eval()
    x, w, b = upsample_case()
    with torch.no_grad():
        m.conv.weight.copy_(w)
        m.conv.bias.copy_(b)
        for size in UPSAMPLE_SIZES:
            y = m(x) if size is None else m(x, output_size=size)
            assert torch.equal(y, y.round())
            key = "none" if size is None else f"{size[0]}x{size[1]}"
            res[f"upsample_{key}_shape"] = np.array(y.shape)
            res[f"upsample_{key}_sha256"] = np.array(digest(y))


def legacy_v1(ref, state, res):
    """GenPercept_v1/genpercept/pipeline_genpercept.py single_infer (t = 1, pred_latent = -unet_pred, range [-1, 1]) with
    its 77-token padded empty-prompt embedding."""
    from oracle.pipeline import OraclePipeline
    v1_root = f"{ref}/GenPercept_v1"
    spec = importlib.util.spec_from_file_location("genpercept_v1", f"{v1_root}/genpercept/__init__.py",
                                                  submodule_search_locations=[f"{v1_root}/genpercept"])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules["genpercept_v1"] = pkg
    spec.loader.exec_module(pkg)
    mod = importlib.import_module("genpercept_v1.pipeline_genpercept")
    e = np.load(f"{v1_root}/empty_text_embed.npy")
    res["v1_empty_text_embed"] = e
    te = torch.from_numpy(e.astype(np.float32))[None]
    op = OraclePipeline(state, te, dtype=torch.float64)
    p1 = mod.GenPerceptPipeline(unet=_UNetAdapter(op.unet), vae=op.vae, empty_text_embed=op.text_embed)
    with torch.no_grad():
        res["v1_depth"] = p1.single_infer(glue_input(31).double(), mode="depth").numpy()


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "genpercept")):
        sys.exit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    _install_shims(ref)
    from genpercept_b200 import weights as W
    state = W.synth_state(1234)
    te = torch.from_numpy(np.load(os.path.join(HERE, "empty_text_embed_2x1024.npy")).astype(np.float32))[None]
    res = {}
    scheduler_constants(ref, res)
    image_helpers(res)
    upsample2d(ref, res)
    pipeline_glue(ref, state, te, res)
    legacy_v1(ref, state, res)
    # float32 storage: rounding costs <= 6e-8 on the [0, 1] maps and ~1e-6 on UNet features of magnitude <= 17
    res = {k: v.astype(np.float32) if v.dtype == np.float64 else v for k, v in res.items()}
    out = os.path.join(HERE, "reference_glue.npz")
    np.savez_compressed(out, **res)
    print(out, os.path.getsize(out), "bytes")
    for k, v in res.items():
        print(k, v.shape, v.dtype)


if __name__ == "__main__":
    main()
