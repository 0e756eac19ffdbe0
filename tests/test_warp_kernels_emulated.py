"""The DEFAULT blend kernels of the K = 32 path -- one warp per 8x4 pixel block, channel contraction on mma.sync
(seganygaussians_b200/csrc/render_{forward,backward}_warp_kernels.cuh) -- executed on the CPU under the CUDA execution shim
(tests/cuda_emu/: threads, warp shuffles / votes, a collective restatement of mma.m16n8k8 with tf32 operand truncation, float
reductions as atomic adds) and compared with the CPU oracle.

These kernels are GPU-validated (tests/test_parity_gpu.py); having the same source under test here means a change to the
candidate tables, the carry-over of partial groups or the fragment index arithmetic can be checked for correctness before a
GPU minute is spent on it.  Tolerances: n_contrib exact; final_T / colours 5e-6 relative (3xTF32 + host rounding);
gradients the suite's 1e-4 relative (tests/common.py)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from tests import common
from seganygaussians_b200 import synthetic
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# (a candidate's list position rides in the unused 8th float of its record in the warp kernels' candidate tables: measured on
# B200 in round 2, forward 1.009 -> 0.931 ms at c2, and made the only code path)
def _build_emu(extra):
    d = tempfile.mkdtemp(prefix="sagars_emu_")
    so = os.path.join(d, "libemu_warp.so")
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-ffp-contract=off", "-shared", "-fPIC"] + extra +
                          ["-I", os.path.join(ROOT, "tests", "cuda_emu"), "-I", os.path.join(ROOT, "seganygaussians_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cuda_emu", "emu_warp_kernels.cpp"), "-o", so])
    return so


# "eager": asynchronous copies land the moment they are issued (the other extreme of what the programming model allows): a buffer
# refilled while it is still being read shows up as wrong results
@pytest.fixture(scope="module", params=["default", "eager"])
def emu(request):
    so = _build_emu(["-DSAGARS_EMU_ASYNC_EAGER"] if request.param == "eager" else [])
    L = C.CDLL(so)
    L.variant = request.param
    L.emu_forward_warp.restype = C.c_int
    L.emu_forward_warp.argtypes = [C.c_int] * 3 + [C.c_void_p] * 8
    L.emu_backward_warp.restype = C.c_int
    L.emu_backward_warp.argtypes = [C.c_int] * 4 + [C.c_void_p] * 11
    L.emu_backward_tile.restype = C.c_int
    L.emu_backward_tile.argtypes = [C.c_int] * 5 + [C.c_void_p] * 11
    L.emu_backward_tc.restype = C.c_int
    L.emu_backward_tc.argtypes = [C.c_int] * 2 + [C.c_void_p] * 10
    L.emu_forward_tc.restype = C.c_int
    L.emu_forward_tc.argtypes = [C.c_int] * 2 + [C.c_void_p] * 8
    L.emu_make_geo.argtypes = [C.c_int] + [C.c_void_p] * 3
    return L


def _p(a):
    return None if a is None else a.ctypes.data


def _oracle_forward(sc, K, depth, bg):
    g, c = sc.gauss, sc.cam
    mask = None
    if depth:
        mask = (torch.rand(sc.P, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).numpy().reshape(-1)
    return orc.forward(means3D=g.means3D.numpy(), opacities=g.opacities.numpy(), bg=bg, viewmatrix=c.world_view_transform.numpy(),
                       projmatrix=c.full_proj_transform.numpy(), campos=c.camera_center.numpy(), image_height=sc.H, image_width=sc.W,
                       tanfovx=c.tanfovx, tanfovy=c.tanfovy, colors_precomp=g.colors.numpy()[:, :K], scales=g.scales.numpy(),
                       rotations=g.rotations.numpy(), mask=mask, num_channels=K)


def _inputs(emu, fw, sc, K):
    P = sc.P
    geo = np.zeros((P, 8), np.float32)
    m2 = np.ascontiguousarray(fw.means2D.astype(np.float32))
    co = np.ascontiguousarray(fw.conic_opacity.astype(np.float32))
    emu.emu_make_geo(P, _p(m2), _p(co), _p(geo))
    feats = np.ascontiguousarray(sc.gauss.colors.numpy()[:, :K].astype(np.float32))
    ranges = np.ascontiguousarray(fw.ranges.astype(np.uint32))
    pl = np.ascontiguousarray(np.concatenate([fw.point_list, np.zeros(64, np.uint32)]))
    return geo, feats, ranges, pl


@pytest.mark.parametrize("case", [("k32", 260, 32, 32, 32, 5.0), ("k32_ragged", 200, 27, 41, 32, 4.0), ("k32_opaque", 260, 32, 32, 32, 5.0),
                                  ("k16", 300, 32, 32, 16, 5.0), ("k64", 200, 24, 32, 64, 4.0), ("k12", 260, 32, 32, 12, 5.0),
                                  ("k5", 260, 32, 32, 5, 5.0),
                                  ("k3_warp_any", 300, 32, 32, 3, 5.0)], ids=lambda c: c[0])
def test_forward_warp_kernel(emu, case):
    name, P, H, W, K, sigma = case
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    if name == "k32_opaque":
        sc.gauss.opacities = torch.full_like(sc.gauss.opacities, 0.9995)     # 0.99 clamp, pixels saturate (early block exit)
    bg = np.linspace(0.2, 0.8, max(K, 3)).astype(np.float32)
    fw = _oracle_forward(sc, K, False, bg)
    if name == "k32_opaque":
        assert fw.final_T.max() < 1e-3 or (fw.n_contrib.max() < (fw.ranges[:, 1].astype(np.int64) - fw.ranges[:, 0]).max())
    assert (fw.ranges[:, 1].astype(np.int64) - fw.ranges[:, 0]).max() > 70          # several 32-entry chunks, carried leftovers
    geo, feats, ranges, pl = _inputs(emu, fw, sc, K)
    final_T = np.zeros((H, W), np.float32)
    n_contrib = np.zeros((H, W), np.uint32)
    color = np.zeros((K, H, W), np.float32)
    rc = emu.emu_forward_warp(W, H, K, _p(ranges), _p(pl), _p(geo), _p(feats), _p(bg), _p(final_T), _p(n_contrib), _p(color))
    assert rc == 0
    assert np.array_equal(n_contrib, fw.n_contrib)
    np.testing.assert_allclose(final_T, fw.final_T, rtol=5e-6, atol=1e-9)
    np.testing.assert_allclose(color, fw.color, rtol=5e-6, atol=5e-7)


@pytest.mark.parametrize("case", [("k32", 300, 32, 48, 5.0), ("k32_ragged", 220, 27, 41, 4.0), ("k32_opaque", 260, 32, 32, 5.0), ("k32_sparse", 30, 48, 48, 2.0)],
                         ids=lambda c: c[0])
def test_forward_tcgen05_tile_kernel(emu, case):
    """The opt-in tile-per-CTA forward on tcgen05 (SAGARS_FLAG_FWD_TILE; csrc/render_forward_tc_kernels.cuh): operand tiles in the
    canonical K-major layout, asynchronous MMAs committed to mbarriers (executed by the shim as late as the model allows), TMEM
    accumulators read back with tcgen05.ld."""
    name, P, H, W, sigma = case
    K = 32
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    if name == "k32_opaque":
        sc.gauss.opacities = torch.full_like(sc.gauss.opacities, 0.9995)
    bg = np.linspace(0.2, 0.8, K).astype(np.float32)
    fw = _oracle_forward(sc, K, False, bg)
    geo, feats, ranges, pl = _inputs(emu, fw, sc, K)
    final_T = np.zeros((H, W), np.float32)
    n_contrib = np.zeros((H, W), np.uint32)
    color = np.zeros((K, H, W), np.float32)
    rc = emu.emu_forward_tc(W, H, _p(ranges), _p(pl), _p(geo), _p(feats), _p(bg), _p(final_T), _p(n_contrib), _p(color))
    assert rc == 0
    assert np.array_equal(n_contrib, fw.n_contrib)
    np.testing.assert_allclose(final_T, fw.final_T, rtol=5e-6, atol=1e-9)
    np.testing.assert_allclose(color, fw.color, rtol=5e-6, atol=5e-7)


@pytest.mark.parametrize("case", [("k32", 220, 32, 32, 32, False, 5.0, False), ("k32_bg", 160, 24, 32, 32, False, 4.0, True),
                                  ("k32_opaque", 160, 24, 32, 32, False, 4.0, True),       # alpha hits the 0.99 clamp, pixels saturate early
                                  ("k3", 300, 32, 32, 3, False, 5.0, False), ("depth_mask", 300, 32, 32, 3, True, 5.0, True)],
                         ids=lambda c: c[0])
@pytest.mark.parametrize("kind", ["warp", "simt_tile", "mma_tile", "tcgen05"])
def test_backward_kernels(emu, case, kind):
    _backward_case(emu, case, kind)


@pytest.mark.parametrize("case", [("k64", 160, 24, 32, 64, False, 4.0, True),       # two 32-channel blocks of the S product, 4 m-tiles
                                  ("k16", 200, 32, 32, 16, False, 5.0, False),      # ROW = 16
                                  ("k5", 200, 32, 32, 5, False, 5.0, True),         # K % 4 != 0: scalar feature loads, bounds-checked emits
                                  ("k32_mask", 160, 24, 32, 32, True, 4.0, True)],  # mask gradient as channel K: ROW = 64 with K = 32
                         ids=lambda c: c[0])
def test_backward_warp_kernel_other_channel_counts(emu, case):
    """The default backward at the other template instances (gradient / feature tiles in fragment order for ROW = 8, 16, 64, the
    channel-block loop, the generic reduction path)."""
    _backward_case(emu, case, "warp")


def _backward_case(emu, case, kind):
    """kind: the default warp-per-block kernel, and the two CTA-per-tile alternates (fp32 SIMT behind
    SAGARS_FLAG_NO_TENSOR_CORES -- csrc/render_backward_kernels.cuh; mma.sync behind SAGARS_FLAG_BWD_TILE --
    csrc/render_backward_mma_kernels.cuh)."""
    name, P, H, W, K, depth, sigma, with_bg = case
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    if name == "k32_opaque":
        sc.gauss.opacities = torch.full_like(sc.gauss.opacities, 0.9995)
    bg = (np.linspace(0.2, 0.8, max(K, 3)) if with_bg else np.zeros(max(K, 3))).astype(np.float32)
    fw = _oracle_forward(sc, K, depth, bg)
    dpix = np.ascontiguousarray(sc.dL_dout[:K].numpy())
    dmask = np.ascontiguousarray(sc.dL_dmask.numpy()) if depth else None
    bw = orc.backward(fw, dpix, dmask)
    geo, feats, ranges, pl = _inputs(emu, fw, sc, K)
    ggrad = np.zeros((P, 8), np.float32)
    dcol = np.zeros((P, K), np.float32)
    final_T = np.ascontiguousarray(fw.final_T.astype(np.float32))
    n_contrib = np.ascontiguousarray(fw.n_contrib.astype(np.uint32))
    if kind == "tcgen05":
        if K != 32 or depth:
            pytest.skip("the tcgen05 backward handles C = 32 precomputed colours")
        rc = emu.emu_backward_tc(W, H, _p(ranges), _p(pl), _p(bg), _p(geo), _p(feats), _p(final_T), _p(n_contrib), _p(dpix), _p(ggrad), _p(dcol))
    elif kind == "warp":
        rc = emu.emu_backward_warp(int(depth), W, H, K, _p(ranges), _p(pl), _p(bg), _p(geo), _p(feats), _p(final_T), _p(n_contrib),
                                   _p(dpix), _p(dmask), _p(ggrad), _p(dcol))
    else:
        rc = emu.emu_backward_tile(1 if kind == "simt_tile" else 2, int(depth), W, H, K, _p(ranges), _p(pl), _p(bg), _p(geo), _p(feats),
                                   _p(final_T), _p(n_contrib), _p(dpix), _p(dmask), _p(ggrad), _p(dcol))
    assert rc == 0

    def close(got, want, what):
        r, d, s = common.float_err(got, want)
        assert r <= 1.0, f"{what}: max|d|={d:.3e} max|ref|={s:.3e} tol-ratio={r:.2f}"
    close(dcol, bw.colors, "dL_dcolors")
    close(ggrad[:, 0:2], bw.means2D[:, 0:2], "dL_dmean2D")
    close(ggrad[:, 2:5], bw.conic[:, [0, 1, 3]], "dL_dconic")
    close(ggrad[:, 5], bw.opacity.reshape(-1), "dL_dopacity")
    if depth:
        close(ggrad[:, 6], bw.mask.reshape(-1), "dL_dmask")
    assert np.abs(bw.colors).max() > 0 and np.abs(bw.conic).max() > 0
