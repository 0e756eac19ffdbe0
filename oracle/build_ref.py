#!/usr/bin/env python
"""Build recipe for ``oracle/_ref`` -- the UNMODIFIED reference rasterizer, rebuilt for sm_100a.

TEST INFRASTRUCTURE ONLY.  Nothing in the product path (``seganygaussians_b200``) may
import anything from ``oracle/``.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py`` (``--impl reference`` / ``cpu_baseline``) use it, as the checker / the baseline.

What it does
------------
The reference (``<root>/submodules/diff-gaussian-rasterization{,_contrastive_f,-depth}``, where ``<root>`` is
``$SAGA_REFERENCE_ROOT``, by default ``/root/reference``)
has no CPU implementation: its only implementation of the hot path is the CUDA extension
(``cuda_rasterizer/{rasterizer_impl,forward,backward}.cu`` + ``rasterize_points.cu`` + ``ext.cpp``).
Those five source files compile directly with nvcc 12.9 + the torch 2.11 headers once
``-include cstdint`` is added (``cuda_rasterizer/rasterizer_impl.h:58-61`` uses ``uint32_t``
without ``<cstdint>``).  We do NOT run the reference's own ``setup.py`` / CMake; this script
invokes the compiler on the sources *where they lie* under ``<root>`` (read-only) and
writes every output into ``oracle/_ref/<package>/`` (git-ignored).  No reference source is copied
into the repository history; the package's ``__init__.py`` (the reference's public Python API,
needed to drive it "through its own public API" in ``bench.py --impl reference``) is *installed*
next to the built ``_C`` module inside the git-ignored output directory, exactly like
``pip install --target`` would do.

Usage:  [SAGA_REFERENCE_ROOT=<reference checkout>] python oracle/build_ref.py [--variants cf base depth] [--force]
"""
import argparse
import os
import shutil
import sys

# the reference checkout: SAGA_REFERENCE_ROOT, by default /root/reference (where the project's build recipe expects it)
REF_ROOT = os.environ.get("SAGA_REFERENCE_ROOT") or "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
OUT_ROOT = os.path.join(HERE, "_ref")

VARIANTS = {
    # tag: (submodule dir, python package name)
    "cf": ("diff-gaussian-rasterization_contrastive_f", "diff_gaussian_rasterization_contrastive_f"),
    "base": ("diff-gaussian-rasterization", "diff_gaussian_rasterization"),
    "depth": ("diff-gaussian-rasterization-depth", "diff_gaussian_rasterization_depth"),
}
SOURCES = [
    "cuda_rasterizer/rasterizer_impl.cu",
    "cuda_rasterizer/forward.cu",
    "cuda_rasterizer/backward.cu",
    "rasterize_points.cu",
    "ext.cpp",
]
# the reference's 3-nearest-neighbour extension (oracle for the sagars_knn shim, SURVEY.md section 8(f) rank 1)
VARIANTS["simple_knn"] = ("simple-knn", "simple_knn")
SIMPLE_KNN_SOURCES = ["spatial.cu", "simple_knn.cu", "ext.cpp"]


def build_variant(tag: str, verbose: bool = False) -> str:
    sub, pkg = VARIANTS[tag]
    src_dir = os.path.join(REF_ROOT, "submodules", sub)
    if not os.path.isdir(src_dir):
        raise FileNotFoundError(f"reference sources not found: {src_dir}")
    out_dir = os.path.join(OUT_ROOT, pkg)
    build_dir = os.path.join(OUT_ROOT, "_build", pkg)
    os.makedirs(out_dir, exist_ok=True)
    os.makedirs(build_dir, exist_ok=True)

    from torch.utils import cpp_extension

    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    is_knn = tag == "simple_knn"
    cpp_extension.load(
        name="_C",
        sources=[os.path.join(src_dir, s) for s in (SIMPLE_KNN_SOURCES if is_knn else SOURCES)],
        extra_include_paths=[src_dir] if is_knn else [os.path.join(src_dir, "third_party", "glm"), src_dir],
        extra_cflags=["-O3", "-include", "cstdint"],
        extra_cuda_cflags=[
            "-O3",
            "-gencode", "arch=compute_100a,code=sm_100a",
            "-include", "cstdint",
            "-include", "cfloat",      # simple_knn.cu uses FLT_MAX without <cfloat>
            "-lineinfo",
        ],
        build_directory=build_dir,
        is_python_module=False,
        verbose=verbose,
    )
    so = os.path.join(build_dir, "_C.so")
    if not os.path.exists(so):
        raise RuntimeError(f"build produced no {so}")
    shutil.copy2(so, os.path.join(out_dir, "_C.so"))
    # install the reference's public python API next to the built module (git-ignored output)
    init_src = os.path.join(src_dir, pkg, "__init__.py")
    if os.path.exists(init_src):
        shutil.copy2(init_src, os.path.join(out_dir, "__init__.py"))
    else:   # simple_knn ships an empty package directory; the module is imported as simple_knn._C
        open(os.path.join(out_dir, "__init__.py"), "w").close()
    return out_dir


# The reference's render binding (``gaussian_renderer/__init__.py``) and the pure-Python packages its import chain
# executes (``scene``, ``utils``, ``arguments``): installed, like the rasterizers' ``__init__.py`` above, into the
# git-ignored output directory so that the GPU tests can drive the reference's OWN ``render*`` functions on top of the
# reference's OWN extensions (tests/test_renderer_dropin_gpu.py).  Nothing here enters the repository history.
RENDERER_PACKAGES = ("gaussian_renderer", "scene", "utils", "arguments")


def install_renderer() -> str:
    out = os.path.join(OUT_ROOT, "renderer")
    for pkg in RENDERER_PACKAGES:
        src = os.path.join(REF_ROOT, pkg)
        if not os.path.isdir(src):
            raise FileNotFoundError(src)
        dst = os.path.join(out, pkg)
        os.makedirs(dst, exist_ok=True)
        for f in os.listdir(src):
            if f.endswith(".py"):
                shutil.copy2(os.path.join(src, f), os.path.join(dst, f))
    return out


def have_renderer() -> bool:
    return os.path.exists(os.path.join(OUT_ROOT, "renderer", "gaussian_renderer", "__init__.py"))


def have_variant(tag: str) -> bool:
    _, pkg = VARIANTS[tag]
    d = os.path.join(OUT_ROOT, pkg)
    return os.path.exists(os.path.join(d, "_C.so")) and os.path.exists(os.path.join(d, "__init__.py"))


def have_sources() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "submodules"))


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", nargs="*", default=list(VARIANTS))
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--one", default=None, help="(internal) build exactly this variant in-process")
    a = ap.parse_args()
    if a.one is not None:
        d = build_variant(a.one, a.verbose)
        print(f"[build_ref] {a.one}: -> {d}")
        return 0
    if not have_sources():
        print(f"[build_ref] no reference checkout at {REF_ROOT} (set SAGA_REFERENCE_ROOT)", file=sys.stderr)
        return 1
    import subprocess
    for tag in a.variants:
        if have_variant(tag) and not a.force:
            print(f"[build_ref] {tag}: already built")
            continue
        print(f"[build_ref] building {tag} from {REF_ROOT} ...", flush=True)
        # one process per variant: torch's JIT loader version-bumps a module name (``_C`` ->
        # ``_C_v1``) when the same name is built twice with different sources in one process.
        cmd = [sys.executable, os.path.abspath(__file__), "--one", tag] + (["--verbose"] if a.verbose else [])
        subprocess.check_call(cmd)
    if os.path.isdir(os.path.join(REF_ROOT, "gaussian_renderer")):
        print(f"[build_ref] renderer binding installed -> {install_renderer()}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
