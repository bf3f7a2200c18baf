"""CPU tests of the host layer: C-ABI symbols, loud failure without a GPU, image helpers."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from genpercept_b200 import build, engine
    build.build()
    lib = engine.lib()
    hdr = open(os.path.join(ROOT, "include", "genpercept_b200.h")).read()
    syms = sorted(set(re.findall(r"\b(gp_[a-z0-9_]+)\s*\(", hdr)))
    assert len(syms) >= 20
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_path_fails_loudly_without_gpu():
    from genpercept_b200 import engine
    cfg = engine._Config(0, engine.GP_F16, 0, 1, 0)
    h = ctypes.c_void_p()
    assert engine.lib().gp_create(ctypes.byref(cfg), ctypes.byref(h)) == 4      # GP_ERR_CUDA, no fallback
    with pytest.raises(RuntimeError):
        engine.Engine()


def test_product_package_never_imports_oracle():
    for dp, _, fs in os.walk(os.path.join(ROOT, "genpercept_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f


def test_resize_max_res_matches_reference_semantics():
    from genpercept_b200.image_util import get_tv_resample_method, resize_max_res
    x = torch.randint(0, 256, (1, 3, 450, 675), dtype=torch.uint8)
    y = resize_max_res(x, 768, get_tv_resample_method("bilinear"))
    assert tuple(y.shape) == (1, 3, 512, 768) and y.dtype == torch.uint8      # int() truncation (image_util.py:101)
    with pytest.raises(ValueError):
        get_tv_resample_method("lanczos")


def test_spectral_colormap_endpoints():
    from genpercept_b200.image_util import colorize_depth_maps
    c = colorize_depth_maps(np.array([[0.0, 1.0], [0.5, 0.25]]), 0, 1)
    np.testing.assert_allclose(c[0, :, 0, 0], [158 / 255, 1 / 255, 66 / 255], atol=1e-6)
    np.testing.assert_allclose(c[0, :, 0, 1], [94 / 255, 79 / 255, 162 / 255], atol=1e-6)


def test_legacy_vae_key_remap():
    from genpercept_b200.weights import remap_legacy_vae_keys
    sd = {"encoder.mid_block.attentions.0.query.weight": torch.zeros(512, 512, 1, 1),
          "encoder.mid_block.attentions.0.proj_attn.bias": torch.zeros(512), "encoder.conv_in.weight": torch.zeros(1)}
    out = remap_legacy_vae_keys(sd)
    assert out["encoder.mid_block.attentions.0.to_q.weight"].shape == (512, 512)
    assert "encoder.mid_block.attentions.0.to_out.0.bias" in out and "encoder.conv_in.weight" in out


def test_dropin_seeds_the_reference_import_path(tmp_path):
    """run.py:33 does `from genpercept import GenPerceptPipeline`; genpercept/__init__.py:18 resolves it through
    `.genpercept_pipeline`.  With genpercept_b200.dropin installed, an UNMODIFIED reference-style package hands out this
    repo's classes (its own genpercept_pipeline.py — which needs diffusers — is never executed) while its other
    submodules still resolve on disk."""
    import subprocess
    import sys
    pkg = tmp_path / "genpercept"
    (pkg / "util").mkdir(parents=True)
    (pkg / "__init__.py").write_text("from .genpercept_pipeline import GenPerceptPipeline, GenPerceptOutput\n")
    (pkg / "genpercept_pipeline.py").write_text("import diffusers_that_is_not_installed\n")
    (pkg / "util" / "__init__.py").write_text("")
    (pkg / "util" / "image_util.py").write_text("MARK = 'reference util'\n")
    (tmp_path / "run.py").write_text(
        "import sys\nfrom genpercept import GenPerceptPipeline, GenPerceptOutput\nfrom genpercept.util.image_util import MARK\n"
        "print(GenPerceptPipeline.__module__, GenPerceptOutput.__module__, MARK, sys.argv[1:])\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-m", "genpercept_b200.dropin", "run.py", "--mode", "depth"], cwd=tmp_path,
                       env=dict(os.environ, PYTHONPATH=root), capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    assert "genpercept_b200.pipeline genpercept_b200.pipeline reference util ['--mode', 'depth']" in p.stdout
    # the in-process route (dropin.install()) resolves the same package from the working directory
    code = ("import genpercept_b200.dropin as d; d.install(); from genpercept import GenPerceptPipeline as P; "
            "import genpercept; print(P.__module__, genpercept.__file__)")
    q = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, env=dict(os.environ, PYTHONPATH=root), capture_output=True,
                       text=True, timeout=300)
    assert q.returncode == 0, q.stderr[-2000:]
    assert f"genpercept_b200.pipeline {pkg / '__init__.py'}" in q.stdout


def test_tile_shape_policy():
    """The planner's (BN, MT) table (DESIGN.md section 4): many-wave layers keep the wide default, layers that do not fill the
    GPU get narrower N tiles only where the L2 operand traffic allows (host-only C-ABI entry, no device needed)."""
    from genpercept_b200 import engine as E
    # big VAE layers: untouched by the model
    assert E.tile_shape(128, 128, 3, 8, 768, 768) == (128, 2)
    assert E.tile_shape(256, 256, 3, 8, 384, 384) == (256, 1)
    assert E.tile_shape(512, 512, 3, 8, 192, 192) == (256, 1)
    # Cout = 320 / 640: multiples of 64 (staged epilogue), never the divisor 160
    assert E.tile_shape(320, 960, 3, 8, 96, 96)[0] in (192, 128)
    assert E.tile_shape(640, 640, 3, 8, 48, 48) == (128, 2)            # 48 x 48 level at batch 8: two M tiles (fewer weight re-reads)
    # batch 8, 12 x 12 level, 2560 -> 1280: stays at BN = 256 (narrower tiles would move more bytes through L2: measured 152 vs 210 us)
    assert E.tile_shape(1280, 2560, 3, 8, 12, 12) == (256, 1)
    # batch 1, same level: 10 of 148 SMs busy with BN = 256 -> narrow N tiles
    assert E.tile_shape(1280, 2560, 3, 1, 12, 12) == (64, 1)
    assert E.tile_shape(1280, 1280, 1, 1, 12, 12, tokens_mode=True)[0] == 64
    # layers the model never touches: Cout < 128 or not a multiple of 64
    assert E.tile_shape(64, 256, 3, 1, 96, 96) == (64, 1)
    assert E.tile_shape(4, 320, 3, 8, 96, 96) == (16, 2)
