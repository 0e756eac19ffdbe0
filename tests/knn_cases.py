"""Seeded point clouds shared by the neighbour-search tests and the golden-vector generator."""
import numpy as np


def clouds():
    out = {}
    rng = np.random.default_rng(11)
    out["uniform_2000"] = rng.random((2000, 3), dtype=np.float32) * 4 - 2
    # clustered + far outliers (what a trained scene looks like: dense surfaces, sparse floaters)
    c = rng.standard_normal((8, 3)).astype(np.float32) * 3
    pts = (c[rng.integers(0, 8, 3000)] + 0.05 * rng.standard_normal((3000, 3))).astype(np.float32)
    pts[:20] = (rng.standard_normal((20, 3)) * 80).astype(np.float32)
    out["clustered_3000"] = pts
    # exact duplicates and a flat (z = const) sheet
    d = rng.random((500, 3), dtype=np.float32)
    out["duplicates_1000"] = np.concatenate([d, d]).astype(np.float32)
    flat = rng.random((1500, 3), dtype=np.float32)
    flat[:, 2] = 0.25
    out["flat_1500"] = flat
    out["tiny_5"] = rng.random((5, 3), dtype=np.float32)
    return out


def scene_cloud():
    """300k points shaped like a scene's initial point cloud, with floaters far away from the bulk."""
    rng = np.random.default_rng(2)
    big = (rng.standard_normal((300000, 3)) * np.array([5, 1, 3])).astype(np.float32)
    big[:1000] *= 40
    return big
