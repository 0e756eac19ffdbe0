"""SURVEY.md section 8 rows a19 / a20: the drop-in ``gaussian_renderer`` against the REFERENCE's own ``gaussian_renderer``.

Both bindings are driven with the same duck-typed camera / model / pipe objects (SURVEY.md Appendix F): the reference's
``render``, ``render_mask``, ``render_with_depth`` and ``render_contrastive_feature``, run on a B200 on top of the reference's
own CUDA extensions, left sampled golden vectors of their result dictionaries and of the gradients that flow back into the
model's leaves (tests/golden/reference, tests/golden/make_golden_sampled.py); ours run on top of libsagars and are compared
with them (integer outputs exact, fp32 within the parity tolerance).  Also the DEPTH variant's mask-only API
(``GaussianRasterizer.forward_mask``) against the reference's own ``forward_mask``."""
import importlib.util
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests import common
from seganygaussians_b200 import synthetic

pytestmark = pytest.mark.gpu
ROOT = common.ROOT
REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference")
EXACT_OUTPUTS = ("out.radii", "out.visibility_filter", "out.viewspace_points")


def _load_ours():
    """Our drop-in ``gaussian_renderer`` (bound to libsagars), under a name of its own."""
    spec = importlib.util.spec_from_file_location("sagars_gaussian_renderer",
                                                  os.path.join(ROOT, "seganygaussians_b200", "dropin", "gaussian_renderer", "__init__.py"))
    ours = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ours)
    return ours


class _Model:
    """What the render bindings read from a Gaussian model (reference scene/gaussian_model.py, gaussian_model_ff.py)."""

    def __init__(self, sc, K, dev, sh_degree=3):
        g = sc.gauss
        leaf = lambda t: t.clone().to(dev).requires_grad_(True)
        self._xyz, self._opacity, self._scaling, self._rotation = leaf(g.means3D), leaf(g.opacities), leaf(g.scales), leaf(g.rotations)
        gen = torch.Generator().manual_seed(5)
        self._sh = leaf(torch.randn(sc.P, (sh_degree + 1) ** 2, 3, generator=gen) * 0.3)
        # [P, 1]: the reference's depth rasterizer returns dL_dmask as [P, 1], which autograd only accepts for a mask of that shape
        self._mask = leaf(torch.rand(sc.P, 1, generator=gen) * 0.5 + 0.5)
        self._point_features = leaf(torch.nn.functional.normalize(torch.randn(sc.P, K, generator=gen), dim=1))
        self.active_sh_degree = self.max_sh_degree = sh_degree

    get_xyz = property(lambda s: s._xyz)
    get_opacity = property(lambda s: s._opacity)
    get_scaling = property(lambda s: s._scaling)
    get_rotation = property(lambda s: s._rotation)
    get_features = property(lambda s: s._sh)
    get_mask = property(lambda s: s._mask)
    get_point_features = property(lambda s: s._point_features)

    def get_covariance(self, scaling_modifier=1):
        # what the reference's build_covariance_from_scaling_rotation computes (scene/gaussian_model.py:33-37): R from the
        # normalised quaternion, L = R S, Sigma = L L^T, the 6 unique entries
        r, x, y, z = torch.nn.functional.normalize(self._rotation, dim=1).unbind(1)
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                         2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                         2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], dim=1).view(-1, 3, 3)
        L = R * (scaling_modifier * self._scaling)[:, None, :]
        S = L @ L.transpose(1, 2)
        return S[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]

    def leaves(self):
        return {"xyz": self._xyz, "opacity": self._opacity, "scaling": self._scaling, "rotation": self._rotation, "sh": self._sh,
                "mask": self._mask, "features": self._point_features}

    def zero_grad(self):
        for t in self.leaves().values():
            t.grad = None


def _camera(sc, dev):
    c = sc.cam
    return SimpleNamespace(FoVx=2 * math.atan(c.tanfovx), FoVy=2 * math.atan(c.tanfovy), image_height=sc.H, image_width=sc.W,
                           feature_height=sc.H, feature_width=sc.W, world_view_transform=c.world_view_transform.to(dev),
                           full_proj_transform=c.full_proj_transform.to(dev), camera_center=c.camera_center.to(dev))


def _run(fn, model, loss_keys, dL, **kw):
    model.zero_grad()
    out = fn(**kw)
    loss = sum((out[k] * dL[k]).sum() for k in loss_keys)
    loss.backward()
    grads = {n: (None if t.grad is None else t.grad.clone()) for n, t in model.leaves().items()}
    grads["viewspace_points"] = out["viewspace_points"].grad.clone()
    return out, grads


CASES = [("render", dict(), ("render",)),
         ("render", dict(pipe_kw=dict(convert_SHs_python=True, compute_cov3D_python=True)), ("render",)),
         ("render", dict(filtered=True, scaling_modifier=0.8), ("render",)),
         ("render_mask", dict(), ("mask",)),
         ("render_with_depth", dict(), ("render", "mask")),
         ("render_with_depth", dict(filtered=True), ("render", "mask")),
         ("render_contrastive_feature", dict(call_kw=dict(norm_point_features=True)), ("render",))]


def golden_name(i, case):
    return f"dropin_{i}_{case[0]}"


def case_inputs(case):
    """(function name, keyword arguments, loss keys, upstream gradients, model) of one case: seeded, so identical every run."""
    name, opt, loss_keys = case
    dev = torch.device("cuda", 0)
    P, H, W, K = 30000, 200, 304, 32
    sc = synthetic.scene(P, H, W, K)
    model, cam = _Model(sc, K, dev), _camera(sc, dev)
    pipe = SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    for k, v in opt.get("pipe_kw", {}).items():
        setattr(pipe, k, v)
    nch = K if name == "render_contrastive_feature" else 3
    bg = torch.linspace(0.1, 0.9, nch, device=dev)
    kw = dict(viewpoint_camera=cam, pc=model, pipe=pipe, bg_color=bg, **opt.get("call_kw", {}))
    if "scaling_modifier" in opt:
        kw["scaling_modifier"] = opt["scaling_modifier"]
    if opt.get("filtered"):
        kw["filtered_mask"] = (torch.arange(P, device=dev) % 7) == 0
    gen = torch.Generator().manual_seed(11)
    dL = {"render": (torch.randn(nch, H, W, generator=gen) / (H * W)).to(dev), "mask": (torch.randn(1 if name == "render_with_depth" else 3, H, W, generator=gen) / (H * W)).to(dev)}
    return name, kw, loss_keys, dL, model


def result_arrays(out, grads):
    """``{name: array}`` of a render call's result dictionary and of the gradients of the model's leaves (None: absent)."""
    arrays = {"out." + k: v.detach().cpu().numpy() for k, v in out.items()}
    arrays.update({"grad." + n: g.cpu().numpy() for n, g in grads.items() if g is not None})
    return arrays


@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(CASES)])
def test_dropin_render_functions_match_the_reference_binding(case):
    ours = _load_ours()
    z = np.load(os.path.join(REF_GOLDEN, golden_name(CASES.index(case), case) + ".npz"))
    name, kw, loss_keys, dL, model = case_inputs(case)
    o_our, g_our = _run(getattr(ours, name), model, loss_keys, dL, **kw)
    ok, lines = common.compare_summaries(z, result_arrays(o_our, g_our))
    assert ok, "\n".join(lines)
    assert g_our["viewspace_points"].abs().max() > 0


def forward_mask_run(Settings, Rast):
    """(image, radii, dL/dmask) of ``forward_mask`` of a DEPTH rasterizer class on a seeded scene."""
    dev = torch.device("cuda", 0)
    P, H, W = 20000, 160, 240
    sc = synthetic.scene(P, H, W, 3)
    g, c = sc.gauss, sc.cam
    gen = torch.Generator().manual_seed(3)
    dL = (torch.randn(1, H, W, generator=gen) / (H * W)).to(dev)
    rs = Settings(image_height=H, image_width=W, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=torch.zeros(3, device=dev), scale_modifier=1.0,
                  viewmatrix=c.world_view_transform.to(dev), projmatrix=c.full_proj_transform.to(dev), sh_degree=0,
                  campos=c.camera_center.to(dev), prefiltered=False, debug=False)
    mask = (torch.rand(P, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).to(dev).requires_grad_(True)
    out = Rast(raster_settings=rs).forward_mask(means3D=g.means3D.to(dev), means2D=torch.zeros(P, 3, device=dev), opacities=g.opacities.to(dev),
                                                mask=mask, scales=g.scales.to(dev), rotations=g.rotations.to(dev), cov3D_precomp=None)
    img, radii = out[0], out[-1]
    (img * dL).sum().backward()
    return img.detach().cpu().numpy(), radii.detach().cpu().numpy(), mask.grad.detach().cpu().numpy()


def test_forward_mask_matches_the_reference_forward_mask():
    """DEPTH ``GaussianRasterizer.forward_mask`` (reference diff_gaussian_rasterization_depth/__init__.py:359-391): image and the
    gradient of the per-Gaussian mask against the reference's own mask-only kernels (sampled golden vectors)."""
    from seganygaussians_b200 import rasterizer as R
    img, radii, dmask = forward_mask_run(R.GaussianRasterizationSettings, R.GaussianRasterizerDepth)
    z = np.load(os.path.join(REF_GOLDEN, "forward_mask.npz"))
    ok, lines = common.compare_summaries(z, {"image": img, "radii": radii, "dL_dmask": dmask})
    assert ok, "\n".join(lines)
    assert np.abs(dmask).max() > 0
