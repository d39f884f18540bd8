"""distCUDA2 (SURVEY §8 n4): csrc/knn.cu against the compiled unmodified reference simple-knn (bit-exact; its outputs
are stored in tests/golden/reference_outputs.npz, see tests/reference_data.py) and against the numpy brute-force
oracle."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from reference_data import Reference  # noqa: E402

pytestmark = pytest.mark.gpu
REF = os.path.join(ROOT, "oracle", "_ref", "libref_knn.so")


def _clouds(n, seed):
    rng = np.random.default_rng(seed)
    uniform = rng.uniform(-1.3, 1.3, (n, 3)).astype(np.float32)
    centres = rng.uniform(-4, 4, (12, 3))
    clustered = (centres[rng.integers(0, 12, n)] + rng.standard_normal((n, 3)) * rng.uniform(0.01, 0.6, (n, 1))).astype(np.float32)
    planar = uniform.copy()
    planar[:, 2] = 0.25                                      # degenerate extent on one axis
    dup = uniform.copy()
    dup[n // 2:] = dup[: n - n // 2]                          # every point has an exact duplicate
    return {"uniform": uniform, "clustered": clustered, "planar": planar, "duplicates": dup}


def _ref(points_dev):
    """The live reference library: only recording runs (SGB_RECORD_REFERENCE) call it."""
    lib = C.CDLL(REF)
    lib.ref_knn.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    out = torch.zeros(points_dev.shape[0], device=points_dev.device)
    assert lib.ref_knn(points_dev.shape[0], points_dev.data_ptr(), out.data_ptr()) == 0
    return out


@pytest.mark.parametrize("n", [5, 300, 20000, 200001])
def test_bit_exact_vs_compiled_reference(n):
    from semantic_gaussians_b200.simple_knn._C import distCUDA2
    dev = torch.device("cuda:0")
    ref = Reference(f"knn[{n}]")
    for name, pts in _clouds(n, n).items():
        p = torch.from_numpy(pts).to(dev)
        if ref.recording:
            ref.put(name, _ref(p))
        ours = distCUDA2(p)
        assert ref.equal(name, ours), (name, n)


@pytest.mark.parametrize("n", [4, 7, 257, 1500])
def test_matches_bruteforce_oracle(n):
    from oracle.knn_oracle import mean_dist2_3nn
    from semantic_gaussians_b200.simple_knn._C import distCUDA2
    dev = torch.device("cuda:0")
    for name, pts in _clouds(n, 100 + n).items():
        ours = distCUDA2(torch.from_numpy(pts).to(dev)).cpu().numpy()
        o = mean_dist2_3nn(pts)
        assert np.allclose(ours, o, rtol=2e-6, atol=1e-12), (name, n)


def test_edge_cases_and_create_from_pcd():
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.simple_knn import distCUDA2
    dev = torch.device("cuda:0")
    assert distCUDA2(torch.zeros((0, 3), device=dev)).shape == (0,)
    fmax = torch.finfo(torch.float32).max
    one = distCUDA2(torch.zeros((1, 3), device=dev))                       # no neighbour: 3 x FLT_MAX / 3 overflows
    assert torch.isinf(one).all()
    three = distCUDA2(torch.tensor([[0., 0, 0], [1, 0, 0], [0, 2, 0]], device=dev))
    assert torch.isinf(three).all() or bool((three > fmax / 4).all())    # two neighbours + one FLT_MAX term
    with pytest.raises(ValueError):
        distCUDA2(torch.zeros((4, 2), device=dev))
    with pytest.raises(ValueError):
        distCUDA2(torch.zeros((4, 3)))
    rng = np.random.default_rng(0)
    pts, col = rng.uniform(-1, 1, (5000, 3)), rng.uniform(0, 1, (5000, 3))
    m = GaussianModel(3).create_from_pcd(pts, col, spatial_lr_scale=1.0, device=dev)
    d2 = torch.clamp_min(distCUDA2(torch.from_numpy(pts).float().to(dev)), 1e-7)
    assert torch.equal(m._scaling, torch.log(torch.sqrt(d2))[..., None].repeat(1, 3))
    assert m._features_dc.shape == (5000, 1, 3) and m._features_rest.shape == (5000, 15, 3)
    assert torch.allclose(m.get_opacity, torch.full((5000, 1), 0.1, device=dev)) and bool((m._rotation[:, 0] == 1).all())
