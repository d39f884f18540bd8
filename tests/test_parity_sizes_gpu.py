"""Parity at the sizes BASELINE.json states (VERDICT r01 "next" #1): the CUDA path through the drop-in API against
the UNMODIFIED compiled reference (oracle/_ref), at full size; the reference's outputs are stored in
tests/golden/reference_outputs.npz (tests/reference_data.py: digests of the bit-exact outputs, seeded samples of the
others).

  K3  1 M Gaussians x 256 ch, 1920x1080: forward AND backward (reference backward = NUM_CHANNELS=256 rebuild)
  K4  3 M Gaussians x 512 ch, 1296x968 : forward AND backward (NUM_CHANNELS=512 rebuild), one view
  K5  fusion of 2 M Gaussians x 512 ch fp16 maps at 640x480, 3 views, against the numpy oracle on a row sample
  non-finite feature rows: poisoned pixels are exactly the reference's (forward.cu:340-356 skips before it accumulates)

Tolerances: integer outputs bit-exact; floats 1e-4 relative (north_star)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from reference_data import Reference  # noqa: E402
from util import dev_cam, dev_scene, ours_state, run_ours  # noqa: E402

from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras, room_cameras  # noqa: E402

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _ref(name):
    """The live reference library: only recording runs (SGB_RECORD_REFERENCE) call it."""
    from oracle import ref as refmod
    return refmod.RefRasterizer(name)


def _ref_forward(r, sc, cm, C, bg):
    return r.forward(bg=bg, means3D=sc["means3D"], opacities=sc["opacities"], viewmatrix=cm["viewmatrix"],
                     projmatrix=cm["projmatrix"], campos=cm["campos"], tanfovx=cm["tanfovx"], tanfovy=cm["tanfovy"],
                     W=cm["W"], H=cm["H"], colors_precomp=sc["features"], scales=sc["scales"],
                     rotations=sc["rotations"], num_channels=C)


def _free():
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def _full_size_case(P, W, H, C, kind, view, refname_bwd):
    dev = torch.device("cuda:0")
    scene = make_scene(P, seed=0, kind=kind, channels=C)
    cam = (orbit_cameras if kind == "blob" else room_cameras)(8, W, H)[view]
    sc, cm = dev_scene(scene, dev, requires_grad=True), dev_cam(cam, dev)
    del scene
    bg = torch.zeros(C, device=dev)
    sd = {k: (v.detach() if v is not None else None) for k, v in sc.items()}

    ref = Reference(f"full_size[{P}-{W}-{H}-{C}]")
    # ---- forward: integer stage bit-exact, pixels 1e-4
    if ref.recording:
        r = _ref("chn")
        out = _ref_forward(r, sd, cm, C, bg)
        for name in ("R", "radii", "color"):
            ref.put(name, out[name])
        for name in ("point_list", "ranges", "n_contrib", "accum_alpha"):
            ref.put(name, r.field(name))
        del out, r
        _free()
    st = ours_state(sd, cm, C, use_features=True)
    assert ref.equal("R", st["R"])
    assert ref.equal("radii", st["radii"])
    assert ref.equal("point_list", st["point_list"])
    assert ref.equal("ranges", st["ranges"])
    assert ref.equal("n_contrib", st["n_contrib"])
    assert ref.equal("accum_alpha", st["final_T"])
    assert ref.frac_bad("color", st["color"], rtol=RTOL, atol_scale=1e-6) == 0.0
    fwd_err = ref.rel_err("color", st["color"])
    assert fwd_err < 1e-5
    del st
    _free()

    # ---- backward through autograd against the NUM_CHANNELS=C rebuild of the reference
    o = run_ours("chn", sc, cm, bg, use_features=True)
    g = torch.Generator(device=dev).manual_seed(5)
    dL = torch.randn((C, H, W), device=dev, generator=g) / (H * W)
    o["color"].backward(dL)
    pairs = [("dL_dmeans2D", o["means2D"].grad), ("dL_dopacity", sc["opacities"].grad.view(-1)),
             ("dL_dmeans3D", sc["means3D"].grad), ("dL_dscales", sc["scales"].grad),
             ("dL_drotations", sc["rotations"].grad), ("dL_dcolors", sc["features"].grad)]
    if ref.recording:
        r2 = _ref(refname_bwd)
        _ref_forward(r2, sd, cm, C, bg)
        gr = r2.backward(dL)
        for name, _ in pairs:
            ref.put(name, gr[name])
        del gr, r2
    errs = {}
    for name, got in pairs:
        # the reference sums with fp32 atomics in arbitrary order: 1e-4 relative + 1e-4 of the tensor's scale
        assert ref.frac_bad(name, got, rtol=RTOL, atol_scale=1e-4) == 0.0, name
        errs[name] = ref.rel_err(name, got)
        assert errs[name] < 1e-4, name
    print(f"P={P} C={C} {W}x{H}: forward max rel err {fwd_err:.2e}; gradient max rel err "
          + ", ".join(f"{k}={v:.1e}" for k, v in errs.items()) + " (on the stored sample)")
    del o, dL, sc, sd
    _free()


def test_k3_full_size_forward_and_backward_vs_reference():
    """BASELINE.json configs[2]: 1 M Gaussians, 256 channels, 1920x1080, fwd + bwd."""
    _full_size_case(1_000_000, 1920, 1080, 256, "blob", 1, "chn_c256")


def test_k4_full_size_forward_and_backward_vs_reference():
    """BASELINE.json configs[3], one of its views: 3 M Gaussians, 512 channels, 1296x968 (W x H), fwd + bwd."""
    _full_size_case(3_000_000, 1296, 968, 512, "room", 2, "chn_c512")


def test_k5_full_size_fusion_vs_oracle_rows():
    """BASELINE.json configs[4] at size: 2 M Gaussians, 512-channel fp16 maps at 640x480, 3 fused views.  The numpy
    oracle (pinned to the reference's own fusion_utils.py by tests/golden/fusion_golden.npz) treats every Gaussian
    independently, so it is evaluated on a 100 k row sample; the sampled rows of the full-size device result must
    equal it bit for bit (pixel indices, fp32 sums in view order, counts)."""
    from oracle import fusion_oracle as fo
    from semantic_gaussians_b200.fusion import PointCloudToImageMapper, normalize_fused
    dev = torch.device("cuda:0")
    P, C, w, h, nviews = 2_000_000, 512, 640, 480, 3
    scene = make_scene(P, 0, kind="room")
    cams = room_cameras(nviews, w, h)
    rng = np.random.default_rng(7)
    xyz = torch.as_tensor(scene.xyz, device=dev)
    fs = torch.zeros((P, C), device=dev)
    cnt = torch.zeros(P, device=dev)
    rows = np.sort(rng.choice(P, 100_000, replace=False))
    xs = scene.xyz[rows]
    want_sum = np.zeros((rows.size, C), np.float32)
    want_cnt = np.zeros(rows.size, np.float32)
    nvis_total = 0
    for i in range(nviews):
        fm_np = rng.standard_normal((C, h, w)).astype(np.float16)
        depth_np = (2.5 + 0.5 * rng.random((h, w))).astype(np.float32)
        fm = torch.from_numpy(fm_np).to(dev)
        depth = torch.from_numpy(depth_np).to(dev)
        mapper = PointCloudToImageMapper([w, h], 0.25, 10, cams[i].intrinsics(), device=dev)
        nvis = mapper.accumulate(cams[i].world_view_transform, xyz, fm, fs, cnt, depth)
        nvis_total += int(nvis)
        # device mapping of the sampled rows == numpy mapping (bit-exact int64)
        got_map = mapper.compute_mapping_device(cams[i].world_view_transform, xyz, depth)[torch.as_tensor(rows, device=dev)]
        K = fo.rescale_intrinsics(cams[i].intrinsics(), [w, h])
        m = fo.compute_mapping(cams[i].world_view_transform, xs, [w, h], K, 0.25, 10, depth_np)
        assert np.array_equal(got_map.cpu().numpy(), m)
        mk = m[:, 2] != 0
        want_sum[mk] += fm_np[:, m[mk, 0], m[mk, 1]].T.astype(np.float32)
        want_cnt[mk] += 1
        del fm, depth
    assert nvis_total > 0 and want_cnt.sum() > 0
    idx = torch.as_tensor(rows, device=dev)
    assert np.array_equal(cnt[idx].cpu().numpy(), want_cnt)
    assert np.array_equal(fs[idx].cpu().numpy().view(np.int32), want_sum.view(np.int32))   # fp32 sums, bit for bit
    normalize_fused(fs, cnt)
    wc = want_cnt.copy()
    wc[wc == 0] = 1e-5
    assert np.array_equal(fs[idx].cpu().numpy().view(np.int32), (want_sum / wc[:, None]).view(np.int32))
    print(f"K5 at size: {nviews} views, mean visible per view {nvis_total / nviews:.0f} of {P}")


@pytest.mark.parametrize("C,W,H", [(64, 320, 240), (37, 250, 100)])   # TMA ring kernel / direct-load kernel
def test_nonfinite_feature_rows_poison_only_the_pixels_that_blend_them(C, W, H):
    """forward.cu:340-356 skips a Gaussian before it touches the accumulators, so a non-finite feature row only
    reaches the pixels that blend it.  The GEMM-shaped forward multiplies zero weights too (0 * inf = NaN) and
    must repair that: every pixel is non-finite exactly where the reference's is, and equal elsewhere."""
    dev = torch.device("cuda:0")
    scene = make_scene(20000, seed=11, channels=C, scale_mean=0.03)
    cam = orbit_cameras(4, W, H)[0]
    feats = scene.features.copy()
    bad = np.random.default_rng(0).choice(20000, 40, replace=False)
    feats[bad[:15], :] = np.inf
    feats[bad[15:25], ::3] = -np.inf
    feats[bad[25:], 1::2] = np.nan
    scene.features = feats
    sc, cm = dev_scene(scene, dev), dev_cam(cam, dev)
    bg = torch.linspace(0.0, 0.2, C, device=dev)
    o = run_ours("chn", sc, cm, bg, use_features=True)["color"]
    ref = Reference(f"nonfinite_feature_rows[{C}-{W}-{H}]")
    if ref.recording:
        out = _ref_forward(_ref("chn"), sc, cm, C, bg)["color"]
        ref.put("finite", torch.isfinite(out))
        ref.put("nan", torch.isnan(out))
        ref.put("inf_sign", torch.sign(out[torch.isinf(out)]))
        ref.put("finite_values", out[torch.isfinite(out)])
        del out
    fin_o = torch.isfinite(o)
    assert 0 < int((~fin_o).sum()) < fin_o.numel() // 2, "the test scene must poison some pixels, not most"
    assert ref.equal("finite", fin_o)
    assert ref.equal("nan", torch.isnan(o))
    assert ref.equal("inf_sign", torch.sign(o[torch.isinf(o)]))       # inf where the reference has inf (masks equal)
    a, b, scale = ref.pair("finite_values", o[fin_o])
    assert float((a - b).abs().max()) <= RTOL * scale + 1e-6
