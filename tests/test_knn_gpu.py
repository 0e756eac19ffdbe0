"""GPU: sagars_knn (csrc/knn.cu) through its Python wrapper and the two import stand-ins (SURVEY.md section 8(f) rank 1)
against the brute-force oracle, and against golden outputs of the unmodified reference extension (fp32 rounding level:
rtol 1e-6)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import knn_oracle
from tests import common, knn_cases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", list(knn_cases.clouds()))
@pytest.mark.parametrize("K", [1, 3, 8, 16, 32])
def test_knn_matches_bruteforce(name, K):
    from seganygaussians_b200.knn import knn
    pts = knn_cases.clouds()[name]
    for excl in (False, True):
        idx, d2, mean = knn(torch.from_numpy(pts).cuda(), None, K=K, exclude_self=excl, want_mean=True)
        idx, d2, mean = idx.cpu().numpy(), d2.cpu().numpy(), mean.cpu().numpy()
        oi, od = knn_oracle.knn_bruteforce(pts, None, K=K, exclude_self=excl)
        valid = oi >= 0
        assert np.array_equal(idx >= 0, valid)
        assert np.allclose(d2[valid], od[valid], rtol=2e-6, atol=1e-12)           # ascending squared distances
        # every returned index really is at the returned distance, and never the query itself when excluded
        rows, cols = np.nonzero(valid)
        diff = pts[idx[rows, cols]] - pts[rows]
        assert np.allclose((diff * diff).sum(1), d2[rows, cols], rtol=1e-5, atol=1e-12)
        if excl:
            assert not (idx == np.arange(len(pts))[:, None]).any()
        else:
            assert np.all(d2[:, 0] == 0)
        full = valid.all(axis=1)
        assert np.allclose(mean[full], d2[full].sum(1) / K, rtol=1e-5)


def test_separate_query_set():
    from seganygaussians_b200.knn import knn
    rng = np.random.default_rng(5)
    pts = rng.standard_normal((4000, 3)).astype(np.float32)
    qs = (rng.standard_normal((1500, 3)) * 2).astype(np.float32)      # some queries outside the cloud's bounding box
    idx, d2, _ = knn(torch.from_numpy(pts).cuda(), torch.from_numpy(qs).cuda(), K=5)
    oi, od = knn_oracle.knn_bruteforce(pts, qs, K=5)
    assert np.allclose(d2.cpu().numpy(), od, rtol=2e-6, atol=1e-12)


def test_distcuda2_shim_matches_live_reference():
    """distCUDA2 against the reference's simple_knn._C.distCUDA2 on a B200: its whole output on the small clouds, a sampled
    golden vector (plus max and sum of the whole output) on a 300k-point scene cloud."""
    sys.path.append(os.path.join(ROOT, "seganygaussians_b200", "shims"))
    from simple_knn._C import distCUDA2
    golden = os.path.join(ROOT, "tests", "golden", "knn")
    small = np.load(os.path.join(golden, "simple_knn_small.npz"))
    for name, pts in knn_cases.clouds().items():
        if len(pts) < 4:
            continue
        ours, theirs = distCUDA2(torch.from_numpy(pts).cuda()).cpu().numpy(), small[name]
        # both are exact 3-NN searches in fp32; the mean differs by a few ulps at most (FMA contraction of the distances)
        assert np.allclose(ours, theirs, rtol=1e-6, atol=0), (name, float((np.abs(ours - theirs) / theirs).max()))
    ours = distCUDA2(torch.from_numpy(knn_cases.scene_cloud()).cuda()).cpu().numpy()
    ok, line = common.check_summary(np.load(os.path.join(golden, "simple_knn_scene_300k.npz")), "scene_300k", ours, rtol=1e-6, atol_scale=0)
    assert ok, line


def test_knn_points_shim():
    sys.path.append(os.path.join(ROOT, "seganygaussians_b200", "shims"))
    from pytorch3d.ops import knn_points
    pts = torch.from_numpy(knn_cases.clouds()["clustered_3000"]).cuda()
    out = knn_points(pts.unsqueeze(0), pts.unsqueeze(0), K=16)       # the reference's call (gaussian_model_ff.py:326-331)
    idx = out.idx.squeeze()
    assert idx.shape == (3000, 16) and idx.dtype == torch.int64 and out.dists.shape == (1, 3000, 16)
    oi, od = knn_oracle.knn_bruteforce(pts.cpu().numpy(), None, K=16)
    assert np.allclose(out.dists[0].cpu().numpy(), od, rtol=2e-6, atol=1e-12)
    assert torch.equal(idx[:, 0].cpu(), torch.arange(3000))
    # the smoothing gather the map feeds (gaussian_model_ff.py:355-362) works on it
    feats = torch.nn.functional.normalize(torch.randn(3000, 32, device="cuda"), dim=-1)
    assert feats[idx[:, torch.randperm(16)[:8]], :].mean(dim=1).shape == (3000, 32)
