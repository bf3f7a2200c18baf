"""Pins the oracle's orchestration (oracle/pipeline.py) and the oracle's UNet dataflow against the REFERENCE'S OWN code:
``GenPerceptPipeline.single_infer`` / ``encode_rgb`` / ``decode_pred`` (genpercept/genpercept_pipeline.py:375-526),
``CustomUNet2DConditionModel.forward`` (genpercept/models/custom_unet.py:34-427), ``DDIMSchedulerCustomized``, the host
image helpers and the first release's pipeline.

tests/golden/make_golden_reference.py ran the reference's code around THIS package's modules (the oracle's VAE / UNet /
scheduler behind thin adapters, the reference's own DPT head class) and stored what it computed in
tests/golden/reference_glue.npz.  Everything between those modules — latent scaling, the mean half of the moments, the
scheduler call and ``pred_original_sample``, ``/ scale`` + post_quant_conv + decoder, the channel mean, clip and shift,
the DPT feature order and min-max, the skip stack and ``upsample_size`` forwarding — was the reference's code; here the
oracle runs the same modules on the same weights and inputs and must land on the stored results.  Both sides run in
float64 so that the tolerances below do not depend on this machine's float32 summation order.
(What stays unpinned is the inside of the diffusers blocks; see oracle/__init__.py.)"""
import importlib.util
import os

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def mk(golden_dir):
    spec = importlib.util.spec_from_file_location("make_golden_reference", os.path.join(golden_dir, "make_golden_reference.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_glue.npz"))


def _close(mine, want, atol):
    mine = mine.double()
    want = torch.from_numpy(want).double()
    assert mine.shape == want.shape, (tuple(mine.shape), tuple(want.shape))
    assert torch.allclose(mine, want, atol=atol, rtol=0), float((mine - want).abs().max())


def test_single_infer_glue_matches_the_reference(mk, ref, synth_state, text_embed):
    from oracle.pipeline import OraclePipeline
    rgb = mk.glue_input().double()
    # VAE readout, 1- and 3-channel modes
    op = OraclePipeline(synth_state, text_embed, dtype=torch.float64)
    for mode in ("depth", "normal"):
        _close(op.single_infer(rgb, mode=mode), ref[f"glue_{mode}"], 1e-6)
    _close(op.encode_rgb(rgb), ref["glue_encode_rgb"], 1e-7)
    # --fix_timesteps: the reference feeds that timestep to the UNet instead of the scheduler's
    _close(op.single_infer(rgb, mode="normal", fix_timesteps=7), ref["glue_normal_fix_timesteps_7"], 1e-6)
    del op
    # DPT readout (the reference ran its own head class on the same weights)
    od = OraclePipeline(synth_state, text_embed, use_dpt=True, dtype=torch.float64)
    _close(od.single_infer(rgb, mode="depth"), ref["glue_dpt"], 2e-6)


def test_unet_dataflow_matches_the_reference_forward(mk, ref, synth_state, text_embed):
    """The reference's own UNet forward (skip stack, the `upsample_size` forwarding for odd extents, the DPT feature taps,
    conv_norm_out / conv_out) was executed around the ORACLE's blocks, attached to an instance of the reference class;
    oracle.unet's forward must give its output and (a fixed, seeded sample of) its feature maps."""
    from oracle.pipeline import OraclePipeline
    ou = OraclePipeline(synth_state, text_embed, dtype=torch.float64).unet
    ctx = text_embed.double().reshape(1, -1, 1024)
    for (h, w), x in zip(mk.UNET_SIZES, mk.unet_inputs()):
        key = f"unet_{h}x{w}"
        with torch.no_grad():
            _close(ou(x.double(), torch.tensor([1]), ctx), ref[f"{key}_sample"], 1e-6)
            mf = ou(x.double(), torch.tensor([1]), ctx, return_feature=True)
        assert len(mf) == 4
        for i, f in enumerate(mf):
            assert tuple(f.shape) == tuple(ref[f"{key}_feat{i}_shape"]), (key, i)
            idx = torch.from_numpy(ref[f"{key}_feat{i}_idx"].astype(np.int64))
            _close(f.reshape(-1)[idx], ref[f"{key}_feat{i}_val"], 1e-5)


def test_scheduler_constants_match_the_reference_class(ref):
    """src/customized_modules/ddim.py:144-217 (DDIMSchedulerCustomized.__init__ — the part of the scheduler that IS in
    the reference tree; set_timesteps / step are diffusers') instantiated from the reference's own
    hf_configs/scheduler_beta_1.0_1.0/scheduler_config.json, against oracle.scheduler.DDIMOneStep."""
    from oracle.scheduler import DDIMOneStep
    mine = DDIMOneStep()
    assert torch.equal(torch.from_numpy(ref["sched_betas"]), mine.betas)
    assert torch.equal(torch.from_numpy(ref["sched_alphas_cumprod"]), mine.alphas_cumprod)
    assert torch.equal(torch.from_numpy(ref["sched_final_alpha_cumprod"]), mine.final_alpha_cumprod)
    assert float(ref["sched_alphas_cumprod"][1]) == 0.0 and float(ref["sched_init_noise_sigma"]) == 1.0  # beta = 1
    # one DDIM step at the single timestep the pipeline uses (t = 1, leading spacing + offset 1): x0 = -v
    ts = mine.set_timesteps(1)
    assert ts.tolist() == [1]
    g = torch.Generator().manual_seed(0)
    v, x = torch.randn((1, 4, 8, 8), generator=g), torch.randn((1, 4, 8, 8), generator=g)
    prev, x0 = mine.step(v, 1, x)
    assert torch.equal(x0, -v)


def test_host_image_helpers_match_the_reference_functions(mk, ref):
    """genpercept_b200.image_util (host mirror) and oracle.imgproc against the reference's own
    genpercept/util/image_util.py: resize_max_res (:75-105, bit for bit), get_tv_resample_method (:108-119), chw2hwc
    (:66-72)."""
    from genpercept_b200 import image_util as mine
    from oracle import imgproc as IP
    x, c = mk.resize_case()
    for edge in mk.RESIZE_EDGES:
        r = mine.resize_max_res(x, edge)
        assert tuple(r.shape) == tuple(ref[f"resize_{edge}_shape"])
        assert mk.digest(r) == str(ref[f"resize_{edge}_sha256"]), edge
        assert tuple(r.shape[-2:]) == IP.resize_max_res_shape(90, 160, edge)
        d = np.abs(IP.resize_aa(x.numpy(), *r.shape[-2:]).astype(np.int32) - r.numpy().astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() <= 1e-3
    for m in ("bilinear", "bicubic", "nearest"):
        assert mine.get_tv_resample_method(m).value == str(ref[f"resample_{m}"])
    with pytest.raises(ValueError):                           # the reference raises too
        mine.get_tv_resample_method("lanczos")
    assert torch.equal(mine.chw2hwc(c), torch.from_numpy(ref["chw2hwc_tensor"]))
    assert np.array_equal(mine.chw2hwc(c.numpy()), ref["chw2hwc_array"])


def test_legacy_v1_pipeline_closed_form_matches(mk, ref, synth_state):
    """GenPercept_v1/genpercept/pipeline_genpercept.py:263-354 — the first release hard-codes what the v2 scheduler
    collapses to (t = 1, pred_latent = -unet_pred, no scheduler object) and feeds the full 77-token padded empty-prompt
    embedding (GenPercept_v1/empty_text_embed.npy, stored with the result).  Its single_infer around the oracle's modules
    must equal the oracle run with that 77-token context (range [-1,1] there, [0,1] in v2)."""
    from oracle.pipeline import OraclePipeline
    te = torch.from_numpy(ref["v1_empty_text_embed"].astype(np.float32))[None]       # [1, 77, 1024]
    op = OraclePipeline(synth_state, te, dtype=torch.float64)
    mine = op.single_infer(mk.glue_input(31).double(), mode="depth") * 2.0 - 1.0
    # (x + 1) / 2 * 2 - 1 and the different place of the channel mean cost a few ulps of values up to 1
    _close(mine, ref["v1_depth"], 2e-5)
