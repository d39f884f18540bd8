"""Generates tests/golden/fusion_golden.npz by running the REFERENCE's own
PointCloudToImageMapper.compute_mapping (imported from dataset/fusion_utils.py of the original project's
source tree, with the collections.Sequence/Iterable aliases it needs on Python >= 3.10) and the
accumulate/normalise statements of fusion.py:136-147 on seeded synthetic inputs:

    SGB_REFERENCE_TREE=<original project> python tests/golden/make_fusion_golden.py

Inputs are regenerated from the seed by the tests; only outputs are stored."""
import collections
import collections.abc
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = os.environ.get("SGB_REFERENCE_TREE", "")


def import_reference_mapper():
    collections.Sequence = collections.abc.Sequence      # fusion_utils.py:8 uses the pre-3.10 names
    collections.Iterable = collections.abc.Iterable
    # fusion_utils.py:9 imports utils.graphics_utils (torch + numpy only) from the reference tree
    sys.path.insert(0, REF)
    try:
        import importlib
        mod = importlib.import_module("dataset.fusion_utils")
    finally:
        sys.path.remove(REF)
    return mod.PointCloudToImageMapper


def fusion_inputs(seed=0, P=20000, w=160, h=120, C=16, nviews=3):
    """Seeded scene/cameras/feature maps/depths shared by the generator and the tests."""
    from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras
    rng = np.random.default_rng(seed + 100)
    scene = make_scene(P, seed, kind="blob")
    cams = orbit_cameras(nviews, w, h, radius=3.0)
    feats = [rng.standard_normal((C, h, w)).astype(np.float16) for _ in range(nviews)]
    depths = []
    for i, cam in enumerate(cams):
        # synthetic depth: distance-like field with noise, float32 (as render()["depth"]) for even
        # views and float64 (as imageio / depth_scale) for odd ones
        yy, xx = np.mgrid[0:h, 0:w]
        d = 2.2 + 0.8 * np.sin(xx / 17.0 + i) * np.cos(yy / 13.0) + 0.05 * rng.standard_normal((h, w))
        depths.append(d.astype(np.float32) if i % 2 == 0 else d.astype(np.float64))
    return scene, cams, feats, depths


def main():
    import torch
    Mapper = import_reference_mapper()
    scene, cams, feats, depths = fusion_inputs()
    out = {}
    w, h = cams[0].image_width, cams[0].image_height
    P, C = scene.P, feats[0].shape[0]
    modes = {"none": None, "surface": "surface", "depth": "per-view"}
    for mode, dsel in modes.items():
        feat_sum = torch.zeros((P, C), dtype=torch.float32)
        times = torch.zeros((P, 1), dtype=torch.float32)
        for i, cam in enumerate(cams):
            mapper = Mapper([w, h], 0.05, 4, cam.intrinsics())
            depth = depths[i] if dsel == "per-view" else dsel
            mapping = np.ones([P, 4], dtype=int)
            mapping[:, 1:4], weight = mapper.compute_mapping(cam.world_view_transform, scene.xyz, depth)
            out[f"{mode}_mapping_{i}"] = mapping[:, 1:4].astype(np.int64)
            if mapping[:, 3].sum() == 0:
                continue
            mp = torch.from_numpy(mapping)
            mask = mp[:, 3]
            features = torch.from_numpy(feats[i])
            fm = features[:, mp[:, 1], mp[:, 2]].permute(1, 0)     # fusion.py:139-140
            mask_k = mask != 0
            times[mask_k] += 1                                        # fusion.py:143
            feat_sum[mask_k] += fm[mask_k]                            # fusion.py:144
        times[times == 0] = 1e-5                                      # fusion.py:146
        feat_sum /= times                                             # fusion.py:147
        out[f"{mode}_fused"] = feat_sum.numpy()
        out[f"{mode}_times"] = times.numpy()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fusion_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
