"""The fp32 tile-per-CTA forward kernel (seganygaussians_b200/csrc/render_forward_kernels.cuh) executed on the CPU under the
CUDA execution shim.  Keeps the kernel's control flow (cp.async staging of double-buffered batches, sentinel padding, early
exit, ragged edges) under test in the CPU-only suite; the shim lets every asynchronous copy land as late, or as early, as the
programming model allows, so a read before the wait or a buffer refilled while still in use computes on the wrong data.

Compared with the CPU oracle: n_contrib exact, final_T / colours / mask / depth to fp32 rounding (the host compiler does not
contract a*b+c the way nvcc does, so the last bit of `power` may differ; 5e-6 relative is ample)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import common
from seganygaussians_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# "late": asynchronous copies land as late as the programming model allows (a missing wait reads stale bytes); "eager": the moment
# they are issued (a buffer refilled while it is still being read computes on the wrong data)
@pytest.fixture(scope="module", params=["late", "eager"])
def emu(request):
    d = tempfile.mkdtemp(prefix="sagars_emu_")
    so = os.path.join(d, "libemu_render_forward.so")
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-ffp-contract=off", "-shared", "-fPIC"] +
                          (["-DSAGARS_EMU_ASYNC_EAGER"] if request.param == "eager" else []) + [
                           "-I", os.path.join(ROOT, "tests", "cuda_emu"), "-I", os.path.join(ROOT, "seganygaussians_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cuda_emu", "emu_render_forward.cpp"), "-o", so])
    L = C.CDLL(so)
    L.emu_render_forward.restype = C.c_int
    L.emu_render_forward.argtypes = [C.c_int] * 4 + [C.c_void_p] * 12
    L.emu_make_geo.argtypes = [C.c_int] + [C.c_void_p] * 3
    return L


def _render(emu, o, sc, K, depth, bg):
    P, H, W = sc.P, sc.H, sc.W
    geo = np.zeros((P, 8), np.float32)
    m2 = np.ascontiguousarray(o.means2D.astype(np.float32))
    co = np.ascontiguousarray(o.conic_opacity.astype(np.float32))
    p = lambda a: None if a is None else a.ctypes.data
    emu.emu_make_geo(P, p(m2), p(co), p(geo))
    feats = np.ascontiguousarray(sc.gauss.colors.numpy()[:, :K].astype(np.float32))
    ranges = np.ascontiguousarray(o.ranges.astype(np.uint32))
    pl = np.ascontiguousarray(np.concatenate([o.point_list, np.zeros(64, np.uint32)]))
    depths = np.ascontiguousarray(o.depths.astype(np.float32))
    mask = None
    if depth:
        import torch
        mask = np.ascontiguousarray((torch.rand(P, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).numpy().reshape(-1))
    out = dict(final_T=np.zeros((H, W), np.float32), n_contrib=np.zeros((H, W), np.uint32), color=np.zeros((K, H, W), np.float32),
               out_mask=np.zeros((1, H, W), np.float32), out_depth=np.zeros((1, H, W), np.float32))
    bg = np.ascontiguousarray(bg.astype(np.float32))
    rc = emu.emu_render_forward(int(depth), W, H, K, p(ranges), p(pl), p(geo), p(feats), p(mask), p(depths), p(bg),
                                p(out["final_T"]), p(out["n_contrib"]), p(out["color"]), p(out["out_mask"]), p(out["out_depth"]))
    assert rc == 0
    return out


CASES = [
    # name, P, H, W, K, depth, sigma: more than 64 instances per tile -> several batches through both pipeline stages
    ("base_k3", 700, 40, 56, 3, False, 5.0),
    ("depth_k3", 500, 33, 47, 3, True, 5.0),
    ("vec_k8", 600, 32, 48, 8, False, 6.0),
    ("vec_k32", 400, 32, 32, 32, False, 6.0),
    ("short_lists", 60, 48, 48, 3, False, 2.0),          # fewer than 64 instances: one padded batch, empty tiles
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_emulated_forward_matches_oracle(emu, case):
    name, P, H, W, K, depth, sigma = case
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    import torch
    bg = np.linspace(0.1, 0.9, max(K, 3)).astype(np.float32)
    o = common.run_oracle(sc, K, depth=depth, backward=False, bg=torch.tensor(bg))
    if name != "short_lists":
        assert (o.ranges[:, 1].astype(np.int64) - o.ranges[:, 0]).max() > 130     # at least three batches somewhere
    out = _render(emu, o, sc, K, depth, bg)
    assert np.array_equal(out["n_contrib"], o.n_contrib)
    np.testing.assert_allclose(out["final_T"], o.final_T, rtol=5e-6, atol=1e-9)
    np.testing.assert_allclose(out["color"], o.color, rtol=5e-6, atol=2e-7)
    if depth:
        np.testing.assert_allclose(out["out_mask"], o.out_mask, rtol=5e-6, atol=2e-7)
        np.testing.assert_allclose(out["out_depth"], o.out_depth, rtol=5e-6, atol=2e-6)
