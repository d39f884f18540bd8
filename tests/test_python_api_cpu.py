"""Drop-in surface: names, field order and error behaviour of the reference's Python API."""
import ast
import os
import re

import pytest
import torch
from reference_data import Reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SGB_REFERENCE_TREE", "")     # the original project's source tree: read by recording runs only
CHN_FIELDS = ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
              "projmatrix", "sh_degree", "campos", "prefiltered", "debug", "num_channels")


def _ref_settings_fields(path):
    tree = ast.parse(open(path).read())
    for node in ast.walk(tree):
        if isinstance(node, ast.ClassDef) and node.name == "GaussianRasterizationSettings":
            return tuple(s.target.id for s in node.body if isinstance(s, ast.AnnAssign))
    raise AssertionError("class not found")


def test_settings_fields_match_reference():
    from semantic_gaussians_b200 import channel_rasterization as chn
    from semantic_gaussians_b200 import rgbd_rasterization as rgbd
    assert chn.GaussianRasterizationSettings._fields == CHN_FIELDS
    assert rgbd.GaussianRasterizationSettings._fields == CHN_FIELDS[:-1]
    ref = Reference("python_api")
    if ref.recording:
        ref.put("channel_settings_fields", _ref_settings_fields(
            f"{REF}/submodules/channel-rasterization/channel_rasterization/__init__.py"))
        ref.put("rgbd_settings_fields", _ref_settings_fields(
            f"{REF}/submodules/rgbd-rasterization/rgbd_rasterization/__init__.py"))
    assert ref.equal("channel_settings_fields", chn.GaussianRasterizationSettings._fields)
    assert ref.equal("rgbd_settings_fields", rgbd.GaussianRasterizationSettings._fields)


def test_module_surface():
    from semantic_gaussians_b200 import channel_rasterization as chn
    from semantic_gaussians_b200 import renderer
    for name in ("GaussianRasterizationSettings", "GaussianRasterizer", "rasterize_gaussians", "_C"):
        assert hasattr(chn, name)
    for name in ("rasterize_gaussians", "rasterize_gaussians_backward", "mark_visible"):   # ext.cpp:16-18
        assert callable(getattr(chn._C, name))
    import inspect
    sig = inspect.signature(renderer.render)
    assert list(sig.parameters) == ["viewpoint_camera", "pc", "pipe", "bg_color", "scaling_modifier", "override_color",
                                    "override_shape", "foreground", "world_rotate"]
    sig = inspect.signature(renderer.render_chn)
    assert list(sig.parameters) == ["viewpoint_camera", "pc", "pipe", "bg_color", "scaling_modifier", "num_channels",
                                    "override_color", "override_shape", "foreground", "world_rotate"]
    fsig = inspect.signature(chn.GaussianRasterizer.forward)
    assert list(fsig.parameters) == ["self", "means3D", "means2D", "opacities", "shs", "colors_precomp", "scales",
                                     "rotations", "cov3D_precomp"]


def test_rasterizer_argument_errors_match_reference():
    from semantic_gaussians_b200 import channel_rasterization as chn
    rs = chn.GaussianRasterizationSettings(8, 8, 1.0, 1.0, torch.zeros(3), 1.0, torch.eye(4), torch.eye(4), 0,
                                           torch.zeros(3), False, False, 3)
    r = chn.GaussianRasterizer(rs)
    z = torch.zeros
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(means3D=z(1, 3), means2D=z(1, 3), opacities=z(1, 1), scales=z(1, 3), rotations=z(1, 4))
    with pytest.raises(Exception, match="Please provide exactly one of either scale/rotation pair"):
        r(means3D=z(1, 3), means2D=z(1, 3), opacities=z(1, 1), colors_precomp=z(1, 3), scales=z(1, 3))
    with pytest.raises(RuntimeError, match="no CPU path"):    # CPU tensors are rejected, never silently computed
        r(means3D=z(1, 3), means2D=z(1, 3), opacities=z(1, 1), colors_precomp=z(1, 3), scales=z(1, 3), rotations=z(1, 4))
    with pytest.raises(RuntimeError, match="means3D must have dimensions"):
        chn._C.rasterize_gaussians(z(3), z(4, 4), z(4, 3), z(4), z(4, 3), z(4, 4), 1.0, torch.Tensor([]), torch.eye(4),
                                   torch.eye(4), 1.0, 1.0, 8, 8, torch.Tensor([]), 0, z(3), False, False, 3)


def test_eval_sh_matches_reference_python():
    from semantic_gaussians_b200.sh_utils import eval_sh
    torch.manual_seed(0)
    sh = torch.randn(50, 3, 16)
    d = torch.nn.functional.normalize(torch.randn(50, 3), dim=1)
    ref = Reference("eval_sh")
    if ref.recording:
        import importlib.util
        spec = importlib.util.spec_from_file_location("ref_sh_utils", f"{REF}/utils/sh_utils.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        for deg in range(4):
            ref.put(f"degree_{deg}", mod.eval_sh(deg, sh, d))
    for deg in range(4):
        ours, want, _ = ref.pair(f"degree_{deg}", eval_sh(deg, sh, d))    # all 150 values are stored
        assert torch.allclose(ours, want, rtol=1e-6, atol=1e-6)
    assert eval_sh(0, sh, d).shape == (50, 3)


def test_gaussian_model_getters_follow_reference_activations():
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.scene_synth import make_scene
    s = make_scene(100, 1, sh=True)
    m = GaussianModel.from_activated(s.xyz, s.scales, s.rotations, s.opacity, s.shs, device="cpu")
    assert torch.allclose(m.get_scaling, torch.as_tensor(s.scales), rtol=1e-5)
    assert torch.allclose(m.get_opacity, torch.as_tensor(s.opacity), rtol=1e-4, atol=1e-6)
    assert m.get_features.shape == (100, 16, 3)
    cov = m.get_covariance(1.0)
    L = torch.diag_embed(torch.as_tensor(s.scales))
    from semantic_gaussians_b200.gaussian_model import build_rotation
    R = build_rotation(torch.as_tensor(s.rotations))
    full = R @ L @ L.transpose(1, 2) @ R.transpose(1, 2)
    assert torch.allclose(cov[:, 0], full[:, 0, 0], rtol=1e-4, atol=1e-7)
    assert torch.allclose(cov[:, 4], full[:, 1, 2], rtol=1e-4, atol=1e-7)
    m.create_semantic(12)
    assert m._features_semantic.shape == (100, 12) and m._times.shape == (100, 1)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "semantic-gaussians_b200")
    bad = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M) or "liboracle" in txt or "libref_" in txt:
                    bad.append(f)
    assert not bad, f"product files reference the test oracle: {bad}"


def test_next_row_modules_reject_cpu_tensors_loudly():
    """semantic head / distCUDA2 / label rendering have no CPU path: CPU tensors raise, nothing falls back."""
    import pytest
    import torch
    from semantic_gaussians_b200 import semantic
    from semantic_gaussians_b200.simple_knn import distCUDA2
    with pytest.raises(ValueError):
        semantic.semantic_head(torch.zeros(4, 2, 2), torch.zeros(3, 4))
    with pytest.raises(ValueError):
        semantic.feature_logits(torch.zeros(5, 4), torch.zeros(3, 4))
    with pytest.raises(ValueError):
        semantic.label_argmax(torch.zeros(3, 2, 2))
    with pytest.raises(ValueError):
        semantic.distill_loss_and_grad(torch.zeros(4, 2, 2), torch.zeros(3, 4), torch.zeros(2, 2, dtype=torch.int64))
    with pytest.raises(ValueError):
        distCUDA2(torch.zeros(10, 3))


def test_nccl_overlap_options_request_a_high_priority_stream(monkeypatch):
    import torch.distributed as dist
    if not hasattr(dist, "ProcessGroupNCCL"):
        return
    from semantic_gaussians_b200.distributed import nccl_overlap_options
    monkeypatch.delenv("SGB_NCCL_MAX_CTAS", raising=False)
    assert nccl_overlap_options().is_high_priority_stream
    monkeypatch.setenv("SGB_NCCL_MAX_CTAS", "8")
    assert nccl_overlap_options().config.max_ctas == 8
