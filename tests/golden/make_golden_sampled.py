#!/usr/bin/env python
"""Generate the sampled golden vectors of tests/golden/reference/ and tests/golden/knn/ from the UNMODIFIED reference.

The GPU tests that compare this library with the reference at sizes whose outputs are too large to store whole read these
files (tests/common.py ``summarize`` / ``compare_summaries``): integer state and bit-exact results as SHA-256 digests, fp32
results as a seeded sample of elements together with max |x| and sum |x| of the whole array.  The inputs are regenerated from
the seeds by the tests' own case lists, which this script imports, so only the reference's outputs are stored.

It needs a GPU and the reference extensions and render binding built into oracle/_ref (oracle/build_ref.py):
    python tests/golden/make_golden_sampled.py --out <dir>      # then copy <dir>/reference and <dir>/knn into tests/golden/
"""
import argparse
import importlib
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import common, knn_cases  # noqa: E402
from tests import test_parity_gpu as parity  # noqa: E402
from tests import test_renderer_dropin_gpu as dropin  # noqa: E402
from seganygaussians_b200 import synthetic  # noqa: E402


def _save(path, d):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, **d)
    print(f"[golden] {path} ({os.path.getsize(path) / 1e3:.1f} kB)", flush=True)


def live_reference(out):
    for name, P, H, W, K, depth in parity.LIVE_REF:
        sc = synthetic.scene(P, H, W, K)
        ref = common.run_torch_impl("ref", sc, K, depth=depth)
        arrays = dict(common.summary_arrays(ref), color_bits=ref.color)
        _save(os.path.join(out, "reference", name + ".npz"),
              common.summarize_all(arrays, exact=common.SUMMARY_EXACT + ("color_bits",)))
    for name, P, H, W, K, depth, use_sh in parity.LIVE_REF_LARGE:
        sc = synthetic.scene(P, H, W, K, sh_coeffs=16 if use_sh else 0)
        ref = common.run_torch_impl("ref", sc, K, depth=depth, use_sh=use_sh, sh_degree=3 if use_sh else 0)
        _save(os.path.join(out, "reference", name + ".npz"),
              common.summarize_all(common.summary_arrays(ref), exact=common.SUMMARY_EXACT))
        del ref, sc
        torch.cuda.empty_cache()


def mark_visible(out):
    dev = torch.device("cuda", 0)
    pts, c = parity.mark_visible_cloud()
    ref = common.ref_module("cf")
    rs = ref.GaussianRasterizationSettings(40, 56, c.tanfovx, c.tanfovy, torch.zeros(32, device=dev), 1.0, c.world_view_transform.to(dev),
                                           c.full_proj_transform.to(dev), 0, c.camera_center.to(dev), False, False)
    visible = ref.GaussianRasterizer(rs).markVisible(pts.to(dev)).to(torch.bool).cpu().numpy()
    _save(os.path.join(out, "reference", "mark_visible.npz"), common.summarize("visible", visible, exact=True))


def _reference_renderer():
    """The reference's own ``gaussian_renderer`` on top of the reference's own extensions (both under oracle/_ref)."""
    import seganygaussians_b200 as S
    renderer_dir = os.path.join(common.REF_DIR, "renderer")
    if not os.path.exists(os.path.join(renderer_dir, "gaussian_renderer", "__init__.py")):
        raise FileNotFoundError("oracle/_ref/renderer: run oracle/build_ref.py first")
    sys.path.append(S.SHIMS_DIR)                      # plyfile / pytorch3d stand-ins for the reference's `scene` package
    for p in (renderer_dir, common.REF_DIR):          # the reference's python packages and its extensions win
        sys.path.insert(0, p)
    ref = importlib.import_module("gaussian_renderer")
    assert os.path.realpath(ref.__file__).startswith(os.path.realpath(renderer_dir)), ref.__file__
    assert os.path.realpath(sys.modules["diff_gaussian_rasterization"].__file__).startswith(os.path.realpath(common.REF_DIR))
    return ref


def renderer(out):
    ref = _reference_renderer()
    for i, case in enumerate(dropin.CASES):
        name, fn_kw, loss_keys, dL, model = dropin.case_inputs(case)
        o, g = dropin._run(getattr(ref, name), model, loss_keys, dL, **fn_kw)
        _save(os.path.join(out, "reference", dropin.golden_name(i, case) + ".npz"),
              common.summarize_all(dropin.result_arrays(o, g), exact=dropin.EXACT_OUTPUTS))
    refmod = common.ref_module("depth")
    img, radii, dmask = dropin.forward_mask_run(refmod.GaussianRasterizationSettings, refmod.GaussianRasterizer)
    _save(os.path.join(out, "reference", "forward_mask.npz"),
          common.summarize_all({"image": img, "radii": radii, "dL_dmask": dmask}, exact=("radii",)))


def simple_knn(out):
    so = os.path.join(common.REF_DIR, "simple_knn", "_C.so")
    spec = importlib.util.spec_from_file_location("_C", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    d = mod.distCUDA2(torch.from_numpy(knn_cases.scene_cloud()).cuda()).float().cpu().numpy()
    _save(os.path.join(out, "knn", "simple_knn_scene_300k.npz"), common.summarize("scene_300k", d, samples=1024))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.dirname(os.path.abspath(__file__)))
    a = ap.parse_args()
    for step in (simple_knn, mark_visible, renderer, live_reference):
        step(a.out)
