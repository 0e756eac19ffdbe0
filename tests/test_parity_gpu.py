"""GPU parity tests (run with `-m gpu` on a B200): the CUDA path, driven through the reference-shaped operator
API (which calls the C ABI), against (1) the CPU oracle on seeded inputs, (2) golden vectors of the unmodified
reference, (3) sampled golden vectors of the unmodified reference extension up to BASELINE.json's full sizes
(tests/golden/reference, tests/golden/make_golden_sampled.py), and (4) size-independent properties at BASELINE.json's
full size.  Integer state is compared exactly; fp32 within RTOL=1e-4 (tests/common.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from tests import common
from seganygaussians_b200 import synthetic

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference")


@pytest.fixture(scope="module", autouse=True)
def _native_library_loaded():
    from seganygaussians_b200 import _lib
    _lib.load()           # fails loudly when libsagars.so is missing: no fallback
    assert torch.cuda.is_available()


SMALL = [
    # name, P, H, W, K, depth, use_sh, deg, M
    ("cf_small", 3000, 72, 104, 32, False, False, 0, 0),
    ("base_small", 3000, 72, 104, 3, False, False, 0, 0),
    ("depth_small", 3000, 72, 104, 3, True, False, 0, 0),
    ("base_sh3", 2000, 64, 80, 3, False, True, 3, 16),
    ("base_sh1", 1000, 48, 64, 3, False, True, 1, 16),
    ("depth_sh3", 2000, 64, 80, 3, True, True, 3, 16),
    ("cf_ragged", 2500, 75, 101, 32, False, False, 0, 0),     # image not a multiple of the 16x16 tile
    ("k16", 1500, 64, 64, 16, False, False, 0, 0),
    ("k64", 1200, 48, 80, 64, False, False, 0, 0),
    ("k5", 1200, 48, 80, 5, False, False, 0, 0),              # channel count that is not a multiple of 4
    ("one_tile", 300, 16, 16, 32, False, False, 0, 0),
]


@pytest.mark.parametrize("cfg", SMALL, ids=[c[0] for c in SMALL])
def test_cuda_matches_oracle(cfg):
    _, P, H, W, K, depth, use_sh, deg, M = cfg
    sc = synthetic.scene(P, H, W, K, sh_coeffs=M)
    ours = common.run_torch_impl("ours", sc, K, depth=depth, use_sh=use_sh, sh_degree=deg)
    orc = common.run_oracle(sc, K, depth=depth, use_sh=use_sh, sh_degree=deg)
    ok, lines = common.compare(ours, orc, floats=common.FLOAT_FWD + common.GRADS + ("means2D", "conic_opacity", "depths", "cov3D"),
                               verbose=False)
    assert ok, "\n".join(lines)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_cuda_matches_reference_golden(path):
    z = np.load(path)
    P, H, W, K, depth, use_sh, deg, M = [int(v) for v in z["config"]]
    sc = synthetic.scene(P, H, W, K, sh_coeffs=M)
    ours = common.run_torch_impl("ours", sc, K, depth=bool(depth), use_sh=bool(use_sh), sh_degree=deg)
    ref = common.SimpleNamespace(kind="golden(reference)", variant=ours.variant)
    for f in z.files:
        if f != "config":
            setattr(ref, f, z[f])
    ref.num_rendered = int(z["num_rendered"])
    ok, lines = common.compare(ours, ref, floats=common.FLOAT_FWD + common.GRADS + ("means2D", "conic_opacity", "depths", "cov3D"),
                               verbose=False)
    assert ok, "\n".join(lines)


LIVE_REF = [("cf_medium", 200000, 540, 960, 32, False), ("base_medium", 100000, 400, 640, 3, False),
            ("depth_medium", 100000, 400, 640, 3, True), ("cf_full_c2", 1000000, 1080, 1920, 32, False)]


@pytest.mark.parametrize("cfg", LIVE_REF, ids=[c[0] for c in LIVE_REF])
def test_cuda_matches_live_reference(cfg):
    """Against the outputs of the unmodified reference extension on a B200, up to BASELINE.json's full size (c2): integer state
    and final_T to the bit, images, gradients and per-Gaussian state within the parity tolerance (sampled golden vectors)."""
    name, P, H, W, K, depth = cfg
    z = np.load(os.path.join(REF_GOLDEN, name + ".npz"))
    sc = synthetic.scene(P, H, W, K)
    for tensor_cores in (True, False):
        ours = common.run_torch_impl("ours", sc, K, depth=depth, tensor_cores=tensor_cores)
        arrays = common.summary_arrays(ours)
        if not tensor_cores:
            # fp32 SIMT path: images are not merely close, the per-pixel arithmetic is kept operation for operation
            arrays["color_bits"] = ours.color
        ok, lines = common.compare_summaries(z, arrays, skip=("color_bits",) if tensor_cores else ())
        assert ok, f"tensor_cores={tensor_cores}\n" + "\n".join(lines)


# BASELINE.json configs[2] / [3] / [4] at their full sizes, default kernels only (the small LIVE_REF cases above also run the fp32 SIMT
# path): c3-like = SYN(5M, 1036x1600, K=32) -- the garden run's size; c4 = SYN(3M, 1080x1920, K=32) (one of its 8 cameras);
# c5-like = the depth rasterizer on SYN(2M, 1600x1600) with SH degree 3 and a per-Gaussian mask (get_scale.py's workload).
LIVE_REF_LARGE = [("c3_like_5M", 5_000_000, 1036, 1600, 32, False, False), ("c4_3M", 3_000_000, 1080, 1920, 32, False, False),
                  ("c5_like_depth_sh3", 2_000_000, 1600, 1600, 3, True, True)]


@pytest.mark.parametrize("cfg", LIVE_REF_LARGE, ids=[c[0] for c in LIVE_REF_LARGE])
def test_cuda_matches_live_reference_at_baseline_sizes(cfg):
    """Integer state exact, final_T bit-equal, images and all gradients within 1e-4 of the unmodified reference extension
    (sampled golden vectors of its outputs on a B200)."""
    name, P, H, W, K, depth, use_sh = cfg
    z = np.load(os.path.join(REF_GOLDEN, name + ".npz"))
    sc = synthetic.scene(P, H, W, K, sh_coeffs=16 if use_sh else 0)
    ours = common.run_torch_impl("ours", sc, K, depth=depth, use_sh=use_sh, sh_degree=3 if use_sh else 0)
    ok, lines = common.compare_summaries(z, common.summary_arrays(ours))
    assert ok, "\n".join(lines)
    assert ours.num_rendered > 2 * P // 3


def _render(sc, K, colors=None, bg=None, opac=None, cov_precomp=None, use_cub=False, debug=False, backward=False, dL=None,
            tensor_cores=True):
    from seganygaussians_b200 import rasterizer as R
    dev = torch.device("cuda", 0)
    g, c = sc.gauss, sc.cam
    R.set_cub_sort(use_cub)
    R.set_tensor_cores(tensor_cores)
    try:
        Rast = R.GaussianRasterizer if K == 3 else R.GaussianRasterizerContrastiveF
        bg_t = torch.zeros(max(K, 3)) if bg is None else bg
        rs = R.GaussianRasterizationSettings(sc.H, sc.W, c.tanfovx, c.tanfovy, bg_t.to(dev), 1.0, c.world_view_transform.to(dev),
                                             c.full_proj_transform.to(dev), 0, c.camera_center.to(dev), False, debug)
        col = (g.colors if colors is None else colors).to(dev).requires_grad_(True)   # keeps a grad_fn (scratch access)
        kw = dict(scales=g.scales.to(dev), rotations=g.rotations.to(dev)) if cov_precomp is None else dict(cov3D_precomp=cov_precomp.to(dev))
        color, radii = Rast(rs)(means3D=g.means3D.to(dev), means2D=torch.zeros(sc.P, 3, device=dev),
                                opacities=(g.opacities if opac is None else opac).to(dev), colors_precomp=col, **kw)
        if backward:
            color.backward(dL.to(dev))
            torch.cuda.synchronize()
            return color.detach().cpu(), radii.cpu(), col.grad.cpu()
        torch.cuda.synchronize()
        fn = color.grad_fn   # read the scratch while the outputs are alive (saved outputs are weak references)
        scratch = (int(fn.num_rendered),) + tuple(fn.saved_tensors[-3:])
        return color.detach().cpu(), radii.cpu(), scratch
    finally:
        R.set_cub_sort(False)
        R.set_tensor_cores(True)


def test_full_size_properties():
    """Size-independent properties at BASELINE.json's headline size (1M Gaussians, 1080x1920, K=32)."""
    P, H, W, K = 1_000_000, 1080, 1920, 32
    sc = synthetic.scene(P, H, W, K)
    ones = torch.ones(P, K)
    col, radii, (R_, geom, binning, img) = _render(sc, K, colors=ones)
    from seganygaussians_b200 import _lib, rasterizer as R
    # the binning arrays are laid out for the capacity the forward asked for (>= R_ with speculative binning)
    il, bl, gl = _lib.image_layout(W, H), _lib.binning_layout(R.last_binning_capacity), _lib.geom_layout(P)
    final_T = img[il.final_T: il.final_T + 4 * H * W].view(torch.float32).view(H, W).cpu()
    # X5 partition of unity: features == 1, bg == 0  ->  out == 1 - final_T on every channel
    assert torch.allclose(col[0], 1.0 - final_T, rtol=0, atol=3e-6) and torch.equal(col[0], col[K - 1])
    # sortedness + stability of the binning, and ranges partition the list
    keys = binning[bl.point_list_keys: bl.point_list_keys + 8 * R_].view(torch.int64)
    vals = binning[bl.point_list: bl.point_list + 4 * R_].view(torch.int32)
    assert bool((keys[1:] >= keys[:-1]).all())
    same = keys[1:] == keys[:-1]
    assert bool((vals[1:][same] > vals[:-1][same]).all())
    tiles_touched = geom[gl.tiles_touched: gl.tiles_touched + 4 * P].view(torch.int32)
    assert int(tiles_touched.sum()) == R_
    T = ((W + 15) // 16) * ((H + 15) // 16)
    ranges = img[il.ranges: il.ranges + 8 * T].view(torch.int32).view(T, 2).long()
    assert int((ranges[:, 1] - ranges[:, 0]).sum()) == R_
    # idempotence: the forward is deterministic to the bit
    col2, _, _ = _render(sc, K, colors=ones)
    assert torch.equal(col, col2)
    # the library's sort and cub::DeviceRadixSort give the same image bits
    col3, _, _ = _render(sc, K, colors=ones, use_cub=True)
    assert torch.equal(col, col3)


def test_channel_independence_k32_vs_k3():
    """X1: the first three channels of a K=32 render equal the K=3 render of those channels, bit for bit."""
    sc = synthetic.scene(50000, 270, 480, 32)
    c32, r32, _ = _render(sc, 32, tensor_cores=False)
    c3, r3, _ = _render(sc, 3, colors=sc.gauss.colors[:, :3].contiguous(), tensor_cores=False)
    assert torch.equal(c32[:3], c3) and torch.equal(r32, r3)
    # and the tensor-core paths agree with it to fp32 rounding (3xTF32), at both channel counts
    c32_tc, _, _ = _render(sc, 32, tensor_cores=True)
    assert float((c32_tc - c32).abs().max()) <= 1e-5 * float(c32.abs().max())
    c3_tc, _, _ = _render(sc, 3, colors=sc.gauss.colors[:, :3].contiguous(), tensor_cores=True)
    assert float((c3_tc - c3).abs().max()) <= 1e-5 * float(c3.abs().max())


def test_backward_linearity_full_gradient():
    sc = synthetic.scene(30000, 200, 320, 32)
    g1 = torch.randn(32, 200, 320, generator=torch.Generator().manual_seed(3)) / 64000
    g2 = torch.randn(32, 200, 320, generator=torch.Generator().manual_seed(4)) / 64000
    _, _, a = _render(sc, 32, backward=True, dL=g1)
    _, _, b = _render(sc, 32, backward=True, dL=g2)
    _, _, ab = _render(sc, 32, backward=True, dL=2.0 * g1 - 0.5 * g2)
    assert float((2.0 * a - 0.5 * b - ab).abs().max()) <= 1e-4 * float(ab.abs().max())


def test_cov3d_precomp_path_matches_scale_rotation_path():
    """X3: the reference's own Python covariance (build_covariance_from_scaling_rotation) as cov3D_precomp."""
    sc = synthetic.scene(20000, 160, 240, 3)
    g = sc.gauss
    q = g.rotations
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    Rm = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                      2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                      2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], dim=1).view(-1, 3, 3)
    L = Rm * g.scales[:, None, :]
    S = L @ L.transpose(1, 2)
    cov = torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], dim=1).contiguous()
    a, ra, _ = _render(sc, 3, colors=g.colors[:, :3].contiguous())
    b, rb, _ = _render(sc, 3, colors=g.colors[:, :3].contiguous(), cov_precomp=cov)
    assert float((ra != rb).float().mean()) < 1e-3          # radii may flip on fp32 rounding of the covariance
    assert float((a - b).abs().max()) < 5e-3 and float((a - b).abs().mean()) < 1e-5


def mark_visible_cloud():
    """(points, camera): a cloud that straddles the camera's near plane (view z > 0.2)."""
    sc = synthetic.scene(64, 40, 56, 32)
    c = sc.cam
    g = torch.Generator().manual_seed(11)
    pts = c.camera_center[None] + (torch.rand(20000, 3, generator=g) - 0.5) * 8.0          # all around the camera
    return torch.cat([pts, sc.gauss.means3D, (c.camera_center[None] * 3.0).repeat(7, 1)]).contiguous(), c


def test_mark_visible_matches_the_oracle_and_the_reference():
    """a2 / a18: `markVisible` point by point on a cloud that straddles the camera's near plane, against the CPU oracle
    (oracle/sagars_oracle.c, `in_frustum`) and against the unmodified reference's own `GaussianRasterizer.markVisible`
    (its result on a B200, stored as a digest)."""
    from seganygaussians_b200 import rasterizer as R
    from oracle import oracle as orc
    dev = torch.device("cuda", 0)
    pts, c = mark_visible_cloud()
    rs = R.GaussianRasterizationSettings(40, 56, c.tanfovx, c.tanfovy, torch.zeros(32, device=dev), 1.0, c.world_view_transform.to(dev),
                                         c.full_proj_transform.to(dev), 0, c.camera_center.to(dev), False, False)
    ours = R.GaussianRasterizerContrastiveF(rs).markVisible(pts.to(dev))
    assert ours.dtype == torch.bool and ours.shape == (pts.shape[0],)
    want = orc.mark_visible(pts.numpy(), c.world_view_transform.numpy())
    assert 0.2 < want.mean() < 0.8                                                           # the cloud really straddles the plane
    assert np.array_equal(ours.cpu().numpy(), want)
    ok, line = common.check_summary(np.load(os.path.join(REF_GOLDEN, "mark_visible.npz")), "visible", ours.cpu().numpy())
    assert ok, line


def test_edge_cases():
    from seganygaussians_b200 import rasterizer as R
    dev = torch.device("cuda", 0)
    sc = synthetic.scene(64, 40, 56, 32)
    c = sc.cam
    bg = torch.linspace(0.1, 1.0, 32)
    rs = R.GaussianRasterizationSettings(40, 56, c.tanfovx, c.tanfovy, bg.to(dev), 1.0, c.world_view_transform.to(dev),
                                         c.full_proj_transform.to(dev), 0, c.camera_center.to(dev), False, True)  # debug=True
    rast = R.GaussianRasterizerContrastiveF(rs)
    # P == 0: zero-filled outputs, nothing launched (reference rasterize_points.cu:81)
    e = lambda *s: torch.zeros(*s, device=dev)
    color, radii = rast(means3D=e(0, 3), means2D=e(0, 3), opacities=e(0, 1), colors_precomp=e(0, 32), scales=e(0, 3), rotations=e(0, 4))
    assert color.shape == (32, 40, 56) and not color.any() and radii.numel() == 0
    # everything behind the camera: image == background, radii == 0, gradients == 0
    behind = (c.camera_center[None] * 3.0).repeat(64, 1).to(dev).requires_grad_(True)
    cols = sc.gauss.colors.to(dev).requires_grad_(True)
    color, radii = rast(means3D=behind, means2D=e(64, 3), opacities=sc.gauss.opacities.to(dev), colors_precomp=cols,
                        scales=sc.gauss.scales.to(dev), rotations=sc.gauss.rotations.to(dev))
    assert not radii.any() and torch.allclose(color.cpu(), bg[:, None, None].expand(32, 40, 56))
    color.sum().backward()
    assert not cols.grad.any() and not behind.grad.any()
    assert not rast.markVisible(behind.detach()).any() and rast.markVisible(sc.gauss.means3D.to(dev)).any()
    # K != 3 without precomputed colours: the reference's error text
    rs3 = rs._replace(debug=False)
    with pytest.raises(RuntimeError, match="For non-RGB, provide precomputed Gaussian colors"):
        R.GaussianRasterizerContrastiveF(rs3)(means3D=sc.gauss.means3D.to(dev), means2D=e(64, 3), opacities=sc.gauss.opacities.to(dev),
                                              shs=torch.zeros(64, 16, 3, device=dev), scales=sc.gauss.scales.to(dev),
                                              rotations=sc.gauss.rotations.to(dev))


def test_mask_only_path_matches_depth_variant_mask():
    from seganygaussians_b200 import rasterizer as R
    dev = torch.device("cuda", 0)
    sc = synthetic.scene(3000, 72, 104, 3)
    g, c = sc.gauss, sc.cam
    rs = R.GaussianRasterizationSettings(72, 104, c.tanfovx, c.tanfovy, torch.zeros(3, device=dev), 1.0, c.world_view_transform.to(dev),
                                         c.full_proj_transform.to(dev), 0, c.camera_center.to(dev), False, False)
    rast = R.GaussianRasterizerDepth(rs)
    mk = lambda: (torch.rand(3000, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).to(dev).requires_grad_(True)
    m1, m2 = mk(), mk()
    common_kw = dict(means3D=g.means3D.to(dev), means2D=torch.zeros(3000, 3, device=dev), opacities=g.opacities.to(dev),
                     scales=g.scales.to(dev), rotations=g.rotations.to(dev))
    _, out_mask, _, radii = rast(mask=m1, colors_precomp=g.colors.to(dev), **common_kw)
    mask_only, radii2 = rast.forward_mask(mask=m2, **common_kw)
    assert torch.equal(out_mask, mask_only) and torch.equal(radii, radii2)
    gm = sc.dL_dmask.to(dev)
    (out_mask * gm).sum().backward()
    (mask_only * gm).sum().backward()
    assert torch.allclose(m1.grad, m2.grad, rtol=1e-4, atol=1e-9)


def test_speculative_binning_matches_exact_layout():
    """The capacity-hint path (include/sagars.h `binning_capacity_hint`): exact layout, a generous hint and a hint that
    is too small (stages skipped on the device, then re-issued) must all give identical integer state and images."""
    from seganygaussians_b200 import rasterizer as R
    sc = synthetic.scene(4000, 88, 120, 32)
    key = (0, sc.P, sc.W, sc.H)
    try:
        R.set_speculative_binning(False)
        exact = common.run_torch_impl("ours", sc, 32)
        assert exact.binning_capacity == exact.num_rendered
        R.set_speculative_binning(True)
        first = common.run_torch_impl("ours", sc, 32)             # nothing seen yet for this shape: exact layout
        assert first.binning_capacity == first.num_rendered
        roomy = common.run_torch_impl("ours", sc, 32)             # hint = 1.25 x seen
        assert roomy.binning_capacity > roomy.num_rendered
        R._CAPACITY_SEEN[key] = max(1, exact.num_rendered // 3)   # force an overflow
        small = common.run_torch_impl("ours", sc, 32)
        assert small.binning_capacity == small.num_rendered       # re-issued with the exact size
        R._CAPACITY_SEEN[key] = 10 * exact.num_rendered           # far too large is fine as well
        huge = common.run_torch_impl("ours", sc, 32)
    finally:
        R.set_speculative_binning(True)
    for other in (first, roomy, small, huge):
        ok, report = common.compare(other, exact, ints=common.INT_FWD + ("keys",), floats=common.FLOAT_FWD + common.GRADS)
        assert ok, report
        assert np.array_equal(other.color, exact.color)


@pytest.mark.parametrize("cfg", [("cf", 6000, 120, 168, 32, False), ("base", 4000, 90, 130, 3, False),
                                 ("k16", 2500, 80, 96, 16, False), ("k64", 1500, 64, 80, 64, False), ("k5", 1500, 64, 80, 5, False),
                                 ("depth", 4000, 90, 130, 3, True)],
                         ids=lambda c: c[0])
def test_blend_kernel_variants_agree(cfg):
    """Every shipped blend-kernel variant (forward: mma.sync warp / tcgen05 tile / fp32 SIMT; backward: warp-per-block /
    CTA-per-tile / tcgen05 pixel-group / fp32 SIMT) gives the same integer state and the same fp32 results within the parity tolerance."""
    from seganygaussians_b200 import rasterizer as R
    name, P, H, W, K, depth = cfg
    sc = synthetic.scene(P, H, W, K)
    try:
        base = common.run_torch_impl("ours", sc, K, depth=depth, tensor_cores=False)       # fp32 SIMT forward + backward
        runs = {}
        for fwd in ("default", "tile", "warp_any"):
            for bwd in ("default", "tile", "tc"):            # "tc" falls back to the default kernel unless C = 32 precomputed colours
                R.set_blend_kernels(forward=fwd, backward=bwd)
                runs[(fwd, bwd)] = common.run_torch_impl("ours", sc, K, depth=depth, tensor_cores=True)
    finally:
        R.set_blend_kernels()
    for key, other in runs.items():
        ok, report = common.compare(other, base, ints=common.INT_FWD, floats=common.FLOAT_FWD + common.GRADS)
        assert ok, (key, report)


@pytest.mark.parametrize("mod", [0.6, 1.7])
def test_scale_modifier_matches_oracle(mod):
    """scale_modifier != 1 (the viewer's scaling slider): forward state and every gradient against the CPU oracle, including the
    reference's dL_dscales convention (gradient w.r.t. scale_modifier * scale without the factor, CF backward.cu:297-325)."""
    from oracle import oracle
    from seganygaussians_b200 import rasterizer as R
    P, H, W, K = 3000, 72, 104, 3
    sc = synthetic.scene(P, H, W, K)
    g, c = sc.gauss, sc.cam
    dev = torch.device("cuda", 0)
    leaf = lambda t: t.clone().to(dev).requires_grad_(True)
    means3D, opac, scales, rots, colors = leaf(g.means3D), leaf(g.opacities), leaf(g.scales), leaf(g.rotations), leaf(g.colors)
    means2D = torch.zeros(P, 3, device=dev, requires_grad=True)
    rs = R.GaussianRasterizationSettings(image_height=H, image_width=W, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=torch.zeros(3, device=dev),
                                         scale_modifier=mod, viewmatrix=c.world_view_transform.to(dev), projmatrix=c.full_proj_transform.to(dev),
                                         sh_degree=0, campos=c.camera_center.to(dev), prefiltered=False, debug=False)
    color, radii = R.GaussianRasterizer(raster_settings=rs)(means3D=means3D, means2D=means2D, opacities=opac, shs=None, colors_precomp=colors,
                                                            scales=scales, rotations=rots, cov3D_precomp=None)
    (color * sc.dL_dout[:K].to(dev)).sum().backward()
    ofw = oracle.forward(means3D=g.means3D.numpy(), opacities=g.opacities.numpy(), bg=np.zeros(3, np.float32),
                         viewmatrix=c.world_view_transform.numpy(), projmatrix=c.full_proj_transform.numpy(), campos=c.camera_center.numpy(),
                         image_height=H, image_width=W, tanfovx=c.tanfovx, tanfovy=c.tanfovy, scale_modifier=mod,
                         colors_precomp=g.colors.numpy(), scales=g.scales.numpy(), rotations=g.rotations.numpy(), num_channels=K)
    obw = oracle.backward(ofw, sc.dL_dout[:K].numpy())
    assert np.array_equal(radii.cpu().numpy(), ofw.radii) and int(color.grad_fn.num_rendered) == ofw.num_rendered
    for name, got, want in (("color", color, ofw.color), ("dL_dscales", scales.grad, obw.scales), ("dL_drotations", rots.grad, obw.rotations),
                            ("dL_dmeans3D", means3D.grad, obw.means3D), ("dL_dopacity", opac.grad, obw.opacity),
                            ("dL_dcolors", colors.grad, obw.colors), ("dL_dmeans2D", means2D.grad, obw.means2D)):
        r, d, s_ = common.float_err(got.detach().cpu().numpy(), want)
        assert r <= 1.0, f"{name}: max|d|={d:.3e} max|ref|={s_:.3e}"


@pytest.mark.parametrize("cfg", [("cf", 6000, 120, 168, 32, 2.0), ("base_ragged", 4000, 75, 101, 3, 2.0), ("one_tile", 300, 16, 16, 32, 2.0),
                                 ("mid_segments", 12000, 64, 64, 3, 14.0),      # tiles with 1024 < n <= 8192 instances
                                 ("huge_segments", 20000, 32, 48, 3, 60.0),     # tiles with more than 8192 instances
                                 ("sparse", 200, 256, 256, 3, 1.0)],            # mostly empty tiles
                         ids=lambda c: c[0])
def test_tile_sort_binning_is_bit_identical(cfg):
    """SAGARS_FLAG_TILE_SORT (count -> scan -> scatter -> one CTA per tile sorts its segment) must leave exactly the binning
    state of the global radix sort -- point_list, sorted keys, ranges, point_offsets -- and therefore identical images."""
    from seganygaussians_b200 import rasterizer as R
    name, P, H, W, K, sigma = cfg
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    try:
        R.set_binning("radix")
        a = common.run_torch_impl("ours", sc, K, backward=True)
        R.set_binning("tile_sort")
        b = common.run_torch_impl("ours", sc, K, backward=True)
        b2 = common.run_torch_impl("ours", sc, K, backward=False)     # second call: the speculative-capacity path
    finally:
        R.set_binning()
    if name == "mid_segments":
        n = a.ranges[:, 1].astype(np.int64) - a.ranges[:, 0]
        assert n.max() > 1024
    if name == "huge_segments":
        n = a.ranges[:, 1].astype(np.int64) - a.ranges[:, 0]
        assert n.max() > 8192
    for other in (b, b2):
        for f in ("num_rendered", "point_offsets", "point_list", "keys", "ranges", "n_contrib", "final_T", "color"):
            assert np.array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(other, f))), f
    ok, report = common.compare(b, a, ints=(), floats=common.GRADS, verbose=False)
    assert ok, report


@pytest.mark.parametrize("cfg", [("cf", 6000, 120, 168, 32, 2.0), ("base_ragged", 4000, 75, 101, 3, 2.0), ("one_tile", 300, 16, 16, 32, 2.0),
                                 ("many_tiles", 30000, 540, 960, 3, 2.0),       # 2,040 tiles: two passes on the tile bits
                                 ("long_lists", 20000, 32, 48, 3, 60.0), ("sparse", 200, 256, 256, 3, 1.0)], ids=lambda c: c[0])
def test_depth_first_binning_is_bit_identical(cfg):
    """SAGARS_FLAG_DEPTH_FIRST (Gaussians sorted by depth -> instances emitted in that order -> one stable sort on the tile bits)
    must leave exactly the binning state of the reference-style global sort of (tile | depth) keys -- point_list, rebuilt 64-bit
    keys, ranges, point_offsets -- and therefore identical images; exact depth ties included."""
    from seganygaussians_b200 import rasterizer as R
    name, P, H, W, K, sigma = cfg
    sc = synthetic.scene(P, H, W, K, sigma_px=sigma)
    sc.gauss.means3D[1::5] = sc.gauss.means3D[0::5][: len(sc.gauss.means3D[1::5])]     # equal depths: the order falls back to the index
    try:
        R.set_binning("radix")
        a = common.run_torch_impl("ours", sc, K, backward=True)
        R.set_binning("depth_first")
        b = common.run_torch_impl("ours", sc, K, backward=True)
        b2 = common.run_torch_impl("ours", sc, K, backward=False)     # second call: the speculative-capacity path
    finally:
        R.set_binning()
    for other in (b, b2):
        for f in ("num_rendered", "point_offsets", "point_list", "keys", "ranges", "n_contrib", "final_T", "color"):
            assert np.array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(other, f))), f
    ok, report = common.compare(b, a, ints=(), floats=common.GRADS, verbose=False)
    assert ok, report
