"""Fusion oracle (oracle/fusion_oracle.py) pinned against golden vectors produced by the
REFERENCE's own PointCloudToImageMapper + fusion.py accumulate statements
(tests/golden/make_fusion_golden.py)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_fusion_golden import fusion_inputs  # noqa: E402

from oracle import fusion_oracle as fo  # noqa: E402
from reference_data import Reference  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fusion_golden.npz")


@pytest.fixture(scope="module")
def data():
    return fusion_inputs(), np.load(GOLD)


@pytest.mark.parametrize("mode", ["none", "surface", "depth"])
def test_mapping_and_fusion_match_reference(data, mode):
    (scene, cams, feats, depths), gold = data
    w, h = cams[0].image_width, cams[0].image_height
    P, C = scene.P, feats[0].shape[0]
    feat_sum = np.zeros((P, C), np.float32)
    count = np.zeros(P, np.float32)
    for i, cam in enumerate(cams):
        K = fo.rescale_intrinsics(cam.intrinsics(), [w, h])
        depth = {"none": None, "surface": "surface", "depth": depths[i]}[mode]
        m = fo.compute_mapping(cam.world_view_transform, scene.xyz, [w, h], K, 0.05, 4, depth)
        g = gold[f"{mode}_mapping_{i}"]
        assert m.dtype == np.int64 and m.shape == g.shape
        assert np.array_equal(m, g), f"view {i}: {(m != g).any(axis=1).sum()} rows differ"   # bit-exact indices
        fo.accumulate(feats[i], m, feat_sum, count)
    fo.normalize(feat_sum, count)
    assert np.array_equal(count.reshape(-1, 1), gold[f"{mode}_times"])
    assert np.array_equal(feat_sum, gold[f"{mode}_fused"])          # same fp32 sums, same order


def test_some_points_visible_and_some_not(data):
    _, gold = data
    for mode in ("none", "surface", "depth"):
        vis = gold[f"{mode}_mapping_0"][:, 2]
        assert 0 < vis.sum() < vis.size


def test_oracle_matches_live_reference_on_other_seed():
    """Other seed, sizes and thresholds than fusion_golden.npz; the reference mapper's output is stored in
    tests/golden/reference_outputs.npz (recorded with SGB_RECORD_REFERENCE, see tests/reference_data.py)."""
    ref = Reference("fusion_mapping_seed7")
    if ref.recording:
        from make_fusion_golden import import_reference_mapper
        Mapper = import_reference_mapper()
    scene, cams, feats, depths = fusion_inputs(seed=7, P=5000, w=96, h=64, C=4, nviews=2)
    for i, cam in enumerate(cams):
        for mode, depth in zip(("none", "surface", "depth"), (None, "surface", depths[i])):
            if ref.recording:
                want, _ = Mapper([96, 64], 0.1, 2, cam.intrinsics()).compute_mapping(cam.world_view_transform,
                                                                                     scene.xyz, depth)
                ref.put(f"{mode}_mapping_{i}", want)
            K = fo.rescale_intrinsics(cam.intrinsics(), [96, 64])
            got = fo.compute_mapping(cam.world_view_transform, scene.xyz, [96, 64], K, 0.1, 2, depth)
            assert ref.equal(f"{mode}_mapping_{i}", got), (mode, i)
