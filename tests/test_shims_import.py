"""The stand-ins make the reference's own modules importable (SURVEY.md section 8(f) rank 1): every import statement that the
reference's ``scene`` package, its ``gaussian_renderer`` and its scripts make of the packages this library stands in for
(recorded below) runs in a fresh interpreter after ``activate()`` and resolves inside this package."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the import statements of the reference's scene/gaussian_model.py, scene/gaussian_model_ff.py, scene/dataset_readers.py,
# gaussian_renderer/__init__.py, train_scene.py, train_contrastive_feature.py, render.py and saga_gui.py that name a stood-in package
REFERENCE_IMPORTS = (
    "from plyfile import PlyData, PlyElement",
    "from simple_knn._C import distCUDA2",
    "import pytorch3d.ops",
    "from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer",
    "from diff_gaussian_rasterization_depth import GaussianRasterizationSettings as GaussianRasterizationSettingsDepth, "
    "GaussianRasterizer as GaussianRasterizerDepth",
    "from diff_gaussian_rasterization_contrastive_f import GaussianRasterizationSettings as GaussianRasterizationSettingsContrastiveF",
    "from diff_gaussian_rasterization_contrastive_f import GaussianRasterizer as GaussianRasterizerContrastiveF",
    "from gaussian_renderer import render, network_gui",
    "from gaussian_renderer import render, render_contrastive_feature, render_mask",
)


def test_reference_scene_modules_import_with_the_stand_ins():
    code = "\n".join(
        ["import sys; sys.path.insert(0, %r)" % ROOT, "import seganygaussians_b200 as S; S.activate()"] + list(REFERENCE_IMPORTS) + [
            "import plyfile, simple_knn._C, diff_gaussian_rasterization, diff_gaussian_rasterization_depth",
            "import diff_gaussian_rasterization_contrastive_f as cf, gaussian_renderer",
            "callable(pytorch3d.ops.knn_points) or sys.exit('pytorch3d.ops.knn_points')",
            "for m in (plyfile, simple_knn._C, pytorch3d.ops, diff_gaussian_rasterization, diff_gaussian_rasterization_depth, cf, gaussian_renderer):",
            "    assert 'seganygaussians_b200' in m.__file__, m.__file__",
            "print('ok')"])
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]
