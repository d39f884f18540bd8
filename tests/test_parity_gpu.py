"""Parity of the CUDA path (through the drop-in Python API over the C-ABI) against
  (a) the UNMODIFIED compiled reference (oracle/_ref) on the same inputs, its outputs stored in
      tests/golden/reference_outputs.npz (tests/reference_data.py) — bit-exact for the integer stage and, on the
      RGB-D path, for the pixels too; 1e-4 relative for floats;
  (b) golden fixtures produced by that reference (tests/golden/raster_golden_k1.npz);
  (c) the CPU oracle (oracle/raster_oracle.c)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from reference_data import Reference  # noqa: E402
from util import dev_cam, dev_scene, frac_bad, ours_state, run_ours  # noqa: E402

from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "raster_golden_k1.npz")
RTOL = 1e-4   # north_star: "within 1e-4 rel fp32"


def _ref(name):
    """The live reference library: only recording runs (SGB_RECORD_REFERENCE) call it."""
    from oracle import ref as refmod
    return refmod.RefRasterizer(name)


def _ref_forward(r, sc, cm, C, use_features, bg):
    return r.forward(bg=bg, means3D=sc["means3D"], opacities=sc["opacities"], viewmatrix=cm["viewmatrix"],
                     projmatrix=cm["projmatrix"], campos=cm["campos"], tanfovx=cm["tanfovx"], tanfovy=cm["tanfovy"],
                     W=cm["W"], H=cm["H"], shs=None if use_features else sc["shs"],
                     colors_precomp=sc["features"] if use_features else None, scales=sc["scales"],
                     rotations=sc["rotations"], num_channels=C)


@pytest.mark.parametrize("P,W,H,view", [(10000, 256, 256, 0), (200000, 640, 480, 2), (1000000, 1920, 1080, 1),
                                        (30000, 333, 211, 3),
                                        (3000, 4112, 4112, 0)])   # 257 x 257 = 66 049 tiles: the 32-bit tile-key path
def test_rgbd_forward_bit_exact_vs_reference(P, W, H, view):
    """K1 / K2: every integer stage, the state floats and the RGB-D pixels equal the reference's bits."""
    dev = torch.device("cuda:0")
    scene = make_scene(P, seed=0, sh=True)
    cam = orbit_cameras(4, W, H)[view]
    sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
    st = ours_state(sc, cm, 3, use_features=False, want_depth=True)
    ref = Reference(f"rgbd_forward[{P}-{W}-{H}-{view}]")
    if ref.recording:
        r = _ref("rgbd")
        out = _ref_forward(r, sc, cm, 3, False, torch.zeros(3, device=dev))
        rvis = out["radii"] > 0
        for name in ("R", "radii", "color", "depth"):
            ref.put(name, out[name])
        for name in ("depths", "means2D", "conic_opacity", "cov3D", "rgb", "tiles_touched", "clamped"):
            ref.put(name, r.field(name)[rvis])
        for name in ("point_list", "ranges", "n_contrib", "accum_alpha"):
            ref.put(name, r.field(name))
        del out, r
    assert ref.equal("R", st["R"])
    assert ref.equal("radii", st["radii"])
    vis = st["radii"] > 0                                              # == the reference's mask (radii equal)
    for name in ("depths", "means2D", "conic_opacity", "cov3D", "rgb", "tiles_touched", "clamped"):
        assert ref.equal(name, st[name][vis]), name                     # bits of the floats
    assert ref.equal("point_list", st["point_list"])                  # sort order incl. tie-breaks
    assert ref.equal("ranges", st["ranges"])
    assert ref.equal("n_contrib", st["n_contrib"])
    assert ref.equal("accum_alpha", st["final_T"])
    assert ref.equal("color", st["color"])
    assert ref.equal("depth", st["depth"])


@pytest.mark.parametrize("P,W,H,C", [(100000, 640, 480, 32), (100000, 640, 480, 100), (50000, 320, 240, 5),
                                     (300000, 1296, 968, 256), (20000, 200, 120, 768)])
def test_channel_forward_vs_reference(P, W, H, C):
    """K3/K4-style feature raster: integer stage bit-exact, pixels within 1e-4 relative."""
    dev = torch.device("cuda:0")
    scene = make_scene(P, seed=1, channels=C)
    cam = orbit_cameras(4, W, H)[1]
    sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
    st = ours_state(sc, cm, C, use_features=True)
    ref = Reference(f"channel_forward[{P}-{W}-{H}-{C}]")
    if ref.recording:
        r = _ref("chn")
        out = _ref_forward(r, sc, cm, C, True, torch.zeros(C, device=dev))
        for name in ("R", "radii", "color"):
            ref.put(name, out[name])
        for name in ("point_list", "ranges", "n_contrib", "accum_alpha"):
            ref.put(name, r.field(name))
        del out, r
    assert ref.equal("R", st["R"])
    assert ref.equal("radii", st["radii"])
    assert ref.equal("point_list", st["point_list"])
    assert ref.equal("ranges", st["ranges"])
    assert ref.equal("n_contrib", st["n_contrib"])
    assert ref.equal("accum_alpha", st["final_T"])
    assert ref.frac_bad("color", st["color"], rtol=RTOL, atol_scale=1e-6) == 0.0
    assert ref.rel_err("color", st["color"]) < 1e-5


@pytest.mark.parametrize("refname,P,W,H,C,use_features", [
    ("chn", 10000, 256, 256, 3, False),        # SH path, the shipped 3-channel backward
    ("rgbd", 20000, 320, 240, 3, False),
    ("chn", 50000, 320, 240, 3, True),
    ("chn_c100", 50000, 320, 240, 100, True),  # reference rebuilt with NUM_CHANNELS=100
    ("chn_c100", 30000, 333, 211, 100, True),  # ragged image (W % 4 = 1, partial tiles): scalar row paths of the GEMM kernels
    ("chn_c256", 100000, 640, 480, 256, True)])
def test_backward_vs_reference(refname, P, W, H, C, use_features):
    dev = torch.device("cuda:0")
    scene = make_scene(P, seed=2, sh=not use_features, channels=C if use_features else 0)
    cam = orbit_cameras(4, W, H)[1]
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    bg = torch.linspace(0.0, 0.5, C, device=dev)
    o = run_ours("rgbd" if refname == "rgbd" else "chn", sc, cm, bg, use_features=use_features)
    dL = torch.as_tensor(np.random.default_rng(5).standard_normal((C, H, W)).astype(np.float32), device=dev)
    (o["color"] * dL).sum().backward()
    pairs = [("dL_dmeans2D", o["means2D"].grad), ("dL_dopacity", sc["opacities"].grad.view(-1)),
             ("dL_dmeans3D", sc["means3D"].grad), ("dL_dscales", sc["scales"].grad),
             ("dL_drotations", sc["rotations"].grad)]
    pairs.append(("dL_dcolors", sc["features"].grad) if use_features else ("dL_dsh", sc["shs"].grad))
    ref = Reference(f"backward[{refname}-{P}-{W}-{H}-{C}-{use_features}]")
    if ref.recording:
        r = _ref(refname)
        sd = {k: (v.detach() if v is not None else None) for k, v in sc.items()}
        _ref_forward(r, sd, cm, C, use_features, bg)
        g = r.backward(dL)
        for name, _ in pairs:
            ref.put(name, g[name])
        del r, g
    for name, got in pairs:
        # the reference itself sums with fp32 atomics in arbitrary order: compare at 1e-4 relative
        # plus 1e-4 of the tensor's scale, and require every stored entry to pass
        assert ref.frac_bad(name, got, rtol=RTOL, atol_scale=1e-4) == 0.0, name
        assert ref.rel_err(name, got) < 1e-4, name


def test_cov3d_precomp_and_scale_modifier_vs_reference():
    dev = torch.device("cuda:0")
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    scene = make_scene(20000, seed=4, sh=True)
    cam = orbit_cameras(4, 320, 240)[0]
    sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
    pc = GaussianModel.from_activated(scene.xyz, scene.scales, scene.rotations, scene.opacity, scene.shs, device=dev)
    cov = pc.get_covariance(1.7).contiguous()
    o = run_ours("rgbd", sc, cm, torch.zeros(3, device=dev), use_features=False, cov3D_precomp=cov)
    o2 = run_ours("rgbd", sc, cm, torch.zeros(3, device=dev), use_features=False, scale_modifier=0.6)
    ref = Reference("cov3d_precomp_and_scale_modifier")
    if ref.recording:
        r = _ref("rgbd")
        out = r.forward(bg=torch.zeros(3, device=dev), means3D=sc["means3D"], opacities=sc["opacities"],
                        viewmatrix=cm["viewmatrix"], projmatrix=cm["projmatrix"], campos=cm["campos"],
                        tanfovx=cm["tanfovx"], tanfovy=cm["tanfovy"], W=320, H=240, shs=sc["shs"], cov3D_precomp=cov)
        ref.put("cov3D_precomp.radii", out["radii"])
        ref.put("cov3D_precomp.color", out["color"])
        out2 = r.forward(bg=torch.zeros(3, device=dev), means3D=sc["means3D"], opacities=sc["opacities"],
                         viewmatrix=cm["viewmatrix"], projmatrix=cm["projmatrix"], campos=cm["campos"],
                         tanfovx=cm["tanfovx"], tanfovy=cm["tanfovy"], W=320, H=240, shs=sc["shs"], scales=sc["scales"],
                         rotations=sc["rotations"], scale_modifier=0.6)
        ref.put("scale_modifier.color", out2["color"])
        ref.put("scale_modifier.depth", out2["depth"])
        del out, out2, r
    assert ref.equal("cov3D_precomp.radii", o["radii"])
    assert ref.equal("cov3D_precomp.color", o["color"])
    assert ref.equal("scale_modifier.color", o2["color"])
    assert ref.equal("scale_modifier.depth", o2["depth"])


def test_mark_visible_vs_reference_and_oracle():
    from oracle import oracle as orc
    from semantic_gaussians_b200 import channel_rasterization as chn
    dev = torch.device("cuda:0")
    scene = make_scene(50000, seed=9, kind="room")
    from semantic_gaussians_b200.scene_synth import room_cameras
    cam = room_cameras(3, 320, 240)[1]
    sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
    rs = chn.GaussianRasterizationSettings(240, 320, cm["tanfovx"], cm["tanfovy"], torch.zeros(3, device=dev), 1.0,
                                           cm["viewmatrix"], cm["projmatrix"], 0, cm["campos"], False, False, 3)
    got = chn.GaussianRasterizer(rs).markVisible(sc["means3D"]).cpu().numpy()
    want = orc.mark_visible(scene.xyz, cam.world_view_transform)
    assert got.dtype == np.bool_ and 0 < got.sum() < got.size
    assert np.array_equal(got, want)


# ------------------------------------------------------------------ golden fixtures + CPU oracle
@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden fixture not generated yet")
def test_matches_golden_fixture_k1():
    from make_raster_golden import golden_inputs
    dev = torch.device("cuda:0")
    gold = np.load(GOLD)
    scene, cam, dL, bg = golden_inputs("k1")
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    o = run_ours("rgbd", sc, cm, torch.as_tensor(bg, device=dev), use_features=False)
    assert np.array_equal(o["radii"].cpu().numpy(), gold["k1_radii"])
    assert np.array_equal(o["color"].detach().cpu().numpy().view(np.int32), gold["k1_color"].view(np.int32))
    assert np.array_equal(o["depth"].cpu().numpy().view(np.int32), gold["k1_depth"].view(np.int32))
    o["color"].backward(torch.as_tensor(dL, device=dev))
    for name, got in (("dL_dmeans3D", sc["means3D"].grad), ("dL_dsh", sc["shs"].grad),
                      ("dL_dscales", sc["scales"].grad), ("dL_drotations", sc["rotations"].grad),
                      ("dL_dopacity", sc["opacities"].grad.view(-1)), ("dL_dmeans2D", o["means2D"].grad)):
        assert frac_bad(got, gold["k1_" + name], rtol=RTOL, atol_scale=1e-4) == 0.0, name


@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden fixture not generated yet")
def test_matches_golden_fixture_features():
    from make_raster_golden import KF, golden_inputs
    dev = torch.device("cuda:0")
    gold = np.load(GOLD)
    scene, cam, dL, bg = golden_inputs("kf")
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    o = run_ours("chn", sc, cm, torch.as_tensor(bg, device=dev), use_features=True)
    assert np.array_equal(o["radii"].cpu().numpy(), gold["kf_radii"])
    assert frac_bad(o["color"], gold["kf_color"], rtol=RTOL, atol_scale=1e-6) == 0.0
    o["color"].backward(torch.as_tensor(dL, device=dev))
    assert frac_bad(sc["features"].grad, gold["kf_dL_dcolors"], rtol=RTOL, atol_scale=1e-4) == 0.0
    assert frac_bad(sc["means3D"].grad, gold["kf_dL_dmeans3D"], rtol=RTOL, atol_scale=1e-4) == 0.0
    assert KF["C"] == o["color"].shape[0]


@pytest.mark.parametrize("C,use_features", [(3, False), (40, True)])
def test_cuda_vs_cpu_oracle(C, use_features):
    """The CPU restatement is not bit-identical to a GPU (no FMA contraction, libm expf), so pixels
    whose decisions sit within a few ulp of a threshold are exempt (the oracle flags them)."""
    from oracle import oracle as orc
    dev = torch.device("cuda:0")
    P, W, H = 8000, 192, 128
    scene = make_scene(P, seed=12, sh=not use_features, channels=C if use_features else 0, scale_mean=0.04)
    cam = orbit_cameras(5, W, H)[3]
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    bg = torch.full((C,), 0.25, device=dev)
    o = run_ours("chn", sc, cm, bg, use_features=use_features)
    ref = orc.forward(orc.scene_dict(scene), orc.cam_dict(cam), W, H, bg.cpu().numpy(),
                      features=scene.features if use_features else None)
    ok = ~ref["fragile"]
    assert ok.mean() > 0.99
    rad = o["radii"].cpu().numpy()
    mism = rad != ref["pre"]["radii"]
    # a radius may differ only where 3*sqrt(lambda) is within a few ulp of an integer
    rr = ref["pre"]["raw_radius"][mism]
    assert np.all(np.abs(rr - np.round(rr)) < 1e-4 * np.maximum(rr, 1)), "unexplained radius mismatch"
    assert mism.mean() < 1e-3
    col = o["color"].detach().cpu().numpy()
    err = np.abs(col - ref["color"])[:, ok]
    assert err.max() <= RTOL * np.abs(ref["color"]).max() + 1e-6
    dL = np.random.default_rng(3).standard_normal((C, H, W)).astype(np.float32)
    o["color"].backward(torch.as_tensor(dL, device=dev))
    g = orc.backward(ref, orc.scene_dict(scene), orc.cam_dict(cam), W, H, bg.cpu().numpy(), dL,
                     features=scene.features if use_features else None)
    checks = [("dL_dopacity", sc["opacities"].grad.view(-1)), ("dL_dmeans3D", sc["means3D"].grad),
              ("dL_dscales", sc["scales"].grad), ("dL_drotations", sc["rotations"].grad)]
    checks.append(("dL_dcolors", sc["features"].grad) if use_features else ("dL_dsh", sc["shs"].grad))
    for name, got in checks:
        # threshold flips at fragile pixels perturb a handful of Gaussians: allow 0.5 % outliers
        assert frac_bad(got, g[name], rtol=1e-3, atol_scale=1e-3) < 5e-3, name


def test_empty_and_degenerate_inputs():
    from semantic_gaussians_b200 import channel_rasterization as chn
    dev = torch.device("cuda:0")
    cam = orbit_cameras(1, 64, 48)[0]
    cm = dev_cam(cam, dev)

    def rs(C):
        return chn.GaussianRasterizationSettings(48, 64, cm["tanfovx"], cm["tanfovy"], torch.full((C,), 0.5, device=dev),
                                                 1.0, cm["viewmatrix"], cm["projmatrix"], 0, cm["campos"], False, False, C)
    # P = 0: the reference skips the native call and returns its zero-filled image (rasterize_points.cu:73,84)
    z = lambda *s: torch.zeros(s, device=dev)
    color, radii = chn.GaussianRasterizer(rs(8))(means3D=z(0, 3), means2D=z(0, 3), opacities=z(0, 1),
                                                 colors_precomp=z(0, 8), scales=z(0, 3), rotations=z(0, 4))
    assert color.shape == (8, 48, 64) and radii.numel() == 0 and torch.all(color == 0.0)
    # everything behind the camera: nothing rendered, R = 0
    xyz = torch.tensor([[0.0, 0.0, 0.0]], device=dev) + torch.as_tensor(cam.camera_center, device=dev) * 2
    color, radii = chn.GaussianRasterizer(rs(4))(means3D=xyz, means2D=z(1, 3), opacities=torch.ones(1, 1, device=dev),
                                                 colors_precomp=torch.ones(1, 4, device=dev),
                                                 scales=torch.full((1, 3), 0.1, device=dev),
                                                 rotations=torch.tensor([[1.0, 0, 0, 0]], device=dev))
    assert int(radii[0]) == 0 and torch.all(color == 0.5)
    # argument validation mirrors the reference's messages
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        chn.GaussianRasterizer(rs(3))(means3D=xyz, means2D=z(1, 3), opacities=z(1, 1), scales=z(1, 3), rotations=z(1, 4))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        chn.GaussianRasterizer(rs(3))(means3D=xyz, means2D=z(1, 3), opacities=z(1, 1), colors_precomp=z(1, 3))
    with pytest.raises(RuntimeError, match="non-RGB"):
        chn.GaussianRasterizer(rs(5))(means3D=xyz, means2D=z(1, 3), opacities=z(1, 1), shs=z(1, 16, 3),
                                      scales=z(1, 3), rotations=z(1, 4))


def test_sh_degrees_and_ragged_image_sizes():
    dev = torch.device("cuda:0")
    scene = make_scene(20000, seed=21, sh=True)
    ref = Reference("sh_degrees_and_ragged_image_sizes")
    for deg, (W, H) in zip((0, 1, 2, 3), ((17, 33), (250, 100), (641, 479), (16, 16))):
        cam = orbit_cameras(2, W, H)[1]
        sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
        o = run_ours("rgbd", sc, cm, torch.zeros(3, device=dev), use_features=False, sh_degree=deg)
        if ref.recording:
            out = _ref("rgbd").forward(
                bg=torch.zeros(3, device=dev), means3D=sc["means3D"], opacities=sc["opacities"],
                viewmatrix=cm["viewmatrix"], projmatrix=cm["projmatrix"], campos=cm["campos"], tanfovx=cm["tanfovx"],
                tanfovy=cm["tanfovy"], W=W, H=H, shs=sc["shs"], scales=sc["scales"], rotations=sc["rotations"],
                sh_degree=deg)
            ref.put(f"color.{deg}", out["color"])
            ref.put(f"depth.{deg}", out["depth"])
        assert ref.equal(f"color.{deg}", o["color"]), (deg, W, H)
        assert ref.equal(f"depth.{deg}", o["depth"])


def test_channel_forward_and_backward_above_65535_tiles():
    """C > 4 path (alpha pass, directory, GEMM kernels) on a 66 049-tile image: tile ids no longer fit 16 bits."""
    dev = torch.device("cuda:0")
    C, W, H = 8, 4112, 4112
    scene = make_scene(3000, seed=6, sh=False, channels=C)
    cam = orbit_cameras(4, W, H)[2]
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    bg = torch.linspace(0.0, 0.3, C, device=dev)
    o = run_ours("chn", sc, cm, bg, use_features=True)
    sd = {k: (v.detach() if v is not None else None) for k, v in sc.items()}
    ref = Reference("channel_forward_above_65535_tiles")
    if ref.recording:
        out = _ref_forward(_ref("chn"), sd, cm, C, True, bg)
        ref.put("radii", out["radii"])
        ref.put("color", out["color"])
        del out
    assert ref.equal("radii", o["radii"])
    assert ref.rel_err("color", o["color"]) < 1e-5
    dL = torch.zeros((C, H, W), device=dev)
    dL[:, ::7, ::5] = 1.0
    (o["color"] * dL).sum().backward()
    g = sc["features"].grad
    assert torch.isfinite(g).all() and float(g.abs().sum()) > 0
    # linearity in the features pins the C-channel backward without a NUM_CHANNELS=8 reference build:
    # d/df <render(f), dL> = render-weights, so <grad, f> == <render(f) - T*bg, dL>
    with torch.no_grad():
        o0 = run_ours("chn", {**sd, "features": torch.zeros_like(sd["features"])}, cm, bg, use_features=True)["color"]
        lhs = float((g.double() * sd["features"].double()).sum())
        rhs = float(((o["color"].detach() - o0).double() * dL.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * abs(rhs) + 1e-6


@pytest.mark.parametrize("C,W,H", [(6, 250, 100), (5, 333, 211), (36, 641, 479)])
def test_channel_counts_not_multiple_of_four_and_ragged_images(C, W, H):
    """C % 4 != 0 takes the direct-load forward and the scalar feature loads of the chain backward; W % 4 != 0 the
    scalar image-row paths.  Forward against the reference (any C), backward through linearity in the features."""
    dev = torch.device("cuda:0")
    scene = make_scene(20000, seed=8, sh=False, channels=C)
    cam = orbit_cameras(4, W, H)[3]
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    bg = torch.linspace(0.1, 0.4, C, device=dev)
    o = run_ours("chn", sc, cm, bg, use_features=True)
    sd = {k: (v.detach() if v is not None else None) for k, v in sc.items()}
    ref = Reference(f"channel_counts[{C}-{W}-{H}]")
    if ref.recording:
        out = _ref_forward(_ref("chn"), sd, cm, C, True, bg)
        ref.put("radii", out["radii"])
        ref.put("color", out["color"])
        del out
    assert ref.equal("radii", o["radii"])
    assert ref.frac_bad("color", o["color"], rtol=RTOL, atol_scale=1e-6) == 0.0
    dL = torch.as_tensor(np.random.default_rng(C).standard_normal((C, H, W)).astype(np.float32), device=dev)
    (o["color"] * dL).sum().backward()
    g = sc["features"].grad
    with torch.no_grad():
        o0 = run_ours("chn", {**sd, "features": torch.zeros_like(sd["features"])}, cm, bg, use_features=True)["color"]
        lhs = float((g.double() * sd["features"].double()).sum())
        rhs = float(((o["color"].detach() - o0).double() * dL.double()).sum())
        assert abs(lhs - rhs) <= 1e-4 * abs(rhs) + 1e-5
    # every gradient must equal the one of the same problem zero-padded to a multiple of 4 channels (the vector
    # paths, pinned against the reference's NUM_CHANNELS rebuilds above)
    Cp = (C + 3) // 4 * 4 + 4
    pad = lambda t, dim: torch.cat([t, torch.zeros(*[(Cp - C) if i == dim else n for i, n in enumerate(t.shape)], device=dev)], dim=dim)
    sp = {k: (v.detach().clone().requires_grad_(True) if v is not None else None) for k, v in sc.items()}
    sp["features"] = pad(sd["features"], 1).requires_grad_(True)
    op_ = run_ours("chn", sp, cm, pad(bg, 0), use_features=True)
    (op_["color"] * pad(dL, 0)).sum().backward()
    assert frac_bad(op_["color"][:C], o["color"], rtol=RTOL, atol_scale=1e-6) == 0.0
    for name in ("means3D", "scales", "rotations", "opacities"):
        assert frac_bad(sc[name].grad, sp[name].grad, rtol=RTOL, atol_scale=1e-4) == 0.0, name
    assert frac_bad(o["means2D"].grad, op_["means2D"].grad, rtol=RTOL, atol_scale=1e-4) == 0.0
    assert frac_bad(g, sp["features"].grad[:, :C], rtol=RTOL, atol_scale=1e-4) == 0.0
    assert float(sp["features"].grad[:, C:].abs().max()) == 0.0      # zero dL/dout on the padding channels
