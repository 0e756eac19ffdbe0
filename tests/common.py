"""Shared helpers of the parity tests: run a synthetic scene through (a) this library's CUDA path via the
reference-shaped operator API, (b) the CPU oracle, (c) the unmodified reference CUDA extension
(``oracle/_ref``, GPU box only), and compare.

Tolerances (stated once, used everywhere):
  * integer / index state (radii, tiles_touched, point_offsets, num_rendered, point_list, ranges,
    n_contrib): EXACT;
  * fp32 images, final_T and all gradient tensors: |a-b| <= RTOL*max(|a|,|b|) + ATOL_SCALE*max|ref|, with
    RTOL = 1e-4 (the north-star tolerance) and a small absolute floor because the reference's own
    gradients are sums of float atomics in random order (not reproducible to the last bits run to run).
"""
from __future__ import annotations

import ctypes
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from seganygaussians_b200 import synthetic  # noqa: E402

RTOL = 1e-4
ATOL_SCALE = 2e-5

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_PKG = {"base": "diff_gaussian_rasterization", "cf": "diff_gaussian_rasterization_contrastive_f",
           "depth": "diff_gaussian_rasterization_depth"}


def have_gpu() -> bool:
    return torch.cuda.is_available()


def have_ref(variant: str) -> bool:
    d = os.path.join(REF_DIR, REF_PKG[variant])
    return os.path.exists(os.path.join(d, "_C.so")) and os.path.exists(os.path.join(d, "__init__.py"))


def ref_module(variant: str):
    """Import the UNMODIFIED reference package (built by oracle/build_ref.py) under its own name."""
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import importlib
    mod = importlib.import_module(REF_PKG[variant])
    assert os.path.realpath(mod.__file__).startswith(os.path.realpath(REF_DIR)), mod.__file__
    return mod


def variant_of(K: int, depth: bool) -> str:
    return "depth" if depth else ("base" if K == 3 else "cf")


# ----------------------------------------------------------------------------------------------
# runners: all return a namespace with identical field names
# ----------------------------------------------------------------------------------------------
FLOAT_FWD = ("color", "final_T", "out_mask", "out_depth")
INT_FWD = ("radii", "tiles_touched", "point_offsets", "num_rendered", "point_list", "ranges", "n_contrib")
GRADS = ("g_means3D", "g_means2D", "g_colors", "g_opacity", "g_scales", "g_rotations", "g_cov3D", "g_sh", "g_mask")


def _settings(mod_settings, sc, dev, K, sh_degree, debug=False, bg=None):
    c = sc.cam
    bg_t = (torch.zeros(max(K, 3)) if bg is None else bg).to(dev)
    return mod_settings(image_height=sc.H, image_width=sc.W, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=bg_t,
                        scale_modifier=1.0, viewmatrix=c.world_view_transform.to(dev),
                        projmatrix=c.full_proj_transform.to(dev), sh_degree=sh_degree,
                        campos=c.camera_center.to(dev), prefiltered=False, debug=debug)


def _leafs(sc, dev, use_sh, use_cov_precomp=False):
    g = sc.gauss
    L = SimpleNamespace()
    mk = lambda t: t.clone().to(dev).requires_grad_(True)
    L.means3D = mk(g.means3D)
    L.means2D = torch.zeros_like(g.means3D).to(dev).requires_grad_(True)
    L.opacities = mk(g.opacities)
    L.scales = mk(g.scales)
    L.rotations = mk(g.rotations)
    L.colors = None if use_sh else mk(g.colors)
    L.shs = mk(g.shs) if use_sh else None
    # [P,1]: the reference returns dL_dmask as [P,1], so a [P] mask cannot be back-propagated through it
    L.mask = (torch.rand(sc.P, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).to(dev).requires_grad_(True)
    return L


def run_torch_impl(kind: str, sc, K: int, depth: bool = False, use_sh: bool = False, sh_degree: int = 0,
                   backward: bool = True, bg=None, debug=False, tensor_cores: bool = True):
    """kind = 'ours' (libsagars through seganygaussians_b200.rasterizer) or 'ref' (oracle/_ref).
    tensor_cores=False routes the K=32 blend through the fp32 SIMT kernels (bit-exact colours)."""
    dev = torch.device("cuda", 0)
    variant = variant_of(K, depth)
    if kind == "ours":
        from seganygaussians_b200 import rasterizer as R
        R.set_tensor_cores(tensor_cores)
        Settings = R.GaussianRasterizationSettings
        Rast = {"base": R.GaussianRasterizer, "cf": R.GaussianRasterizerContrastiveF, "depth": R.GaussianRasterizerDepth}[variant]
    else:
        mod = ref_module(variant)
        Settings, Rast = mod.GaussianRasterizationSettings, mod.GaussianRasterizer
    L = _leafs(sc, dev, use_sh)
    rs = _settings(Settings, sc, dev, K, sh_degree, debug=debug, bg=bg)
    rast = Rast(raster_settings=rs)
    kw = dict(means3D=L.means3D, means2D=L.means2D, opacities=L.opacities, shs=L.shs, colors_precomp=L.colors,
              scales=L.scales, rotations=L.rotations, cov3D_precomp=None)
    if depth:
        color, out_mask, out_depth, radii = rast(mask=L.mask, **kw)
    else:
        color, radii = rast(**kw)
        out_mask = out_depth = None
    o = SimpleNamespace(kind=kind, variant=variant)
    o.color = color.detach().cpu().numpy()
    o.radii = radii.detach().cpu().numpy().astype(np.int32)
    o.out_mask = None if out_mask is None else out_mask.detach().cpu().numpy()
    o.out_depth = None if out_depth is None else out_depth.detach().cpu().numpy()
    # scratch decode (integer state)
    ctx = color.grad_fn
    saved = ctx.saved_tensors
    geom, binning, img = saved[-3], saved[-2], saved[-1]
    o.num_rendered = int(ctx.num_rendered)
    if kind == "ours":
        from seganygaussians_b200 import rasterizer as _R
        o.binning_capacity = int(_R.last_binning_capacity)
    _decode(o, kind, sc, geom, binning, img)
    if backward:
        loss = (color * sc.dL_dout[:K].to(dev)).sum()
        if depth:
            loss = loss + (out_mask * sc.dL_dmask.to(dev)).sum()
        loss.backward()
        torch.cuda.synchronize()
        gr = lambda t: None if (t is None or t.grad is None) else t.grad.detach().cpu().numpy()
        o.g_means3D, o.g_means2D, o.g_opacity = gr(L.means3D), gr(L.means2D), gr(L.opacities)
        o.g_scales, o.g_rotations = gr(L.scales), gr(L.rotations)
        o.g_colors, o.g_sh = gr(L.colors), gr(L.shs)
        o.g_mask = gr(L.mask).reshape(-1) if depth else None
        o.g_cov3D = None
    return o


def _bytes_view(t: torch.Tensor, offset: int, dtype, count: int):
    nbytes = count * np.dtype(dtype).itemsize
    raw = t[offset:offset + nbytes].cpu().numpy()
    return raw.view(dtype).copy()


def _al(x, a=128):
    return (x + a - 1) // a * a


def _decode(o, kind, sc, geom, binning, img):
    P, H, W, R = sc.P, sc.H, sc.W, o.num_rendered
    T = ((W + 15) // 16) * ((H + 15) // 16)
    N = H * W
    if kind == "ours":
        from seganygaussians_b200 import _lib
        # the binning arrays are laid out for the capacity the forward asked for (>= R with speculative binning)
        gl, il, bl = _lib.geom_layout(P), _lib.image_layout(W, H), _lib.binning_layout(getattr(o, "binning_capacity", R))
        o.tiles_touched = _bytes_view(geom, gl.tiles_touched, np.uint32, P)
        o.point_offsets = _bytes_view(geom, gl.point_offsets, np.uint32, P)
        geo = _bytes_view(geom, gl.geo, np.float32, P * 8).reshape(P, 8)
        o.means2D, o.conic_opacity = geo[:, 0:2].copy(), geo[:, 2:6].copy()
        o.depths = _bytes_view(geom, gl.depths, np.float32, P)
        o.cov3D = _bytes_view(geom, gl.cov3D, np.float32, P * 6).reshape(P, 6)
        o.final_T = _bytes_view(img, il.final_T, np.float32, N).reshape(H, W)
        o.n_contrib = _bytes_view(img, il.n_contrib, np.uint32, N).reshape(H, W)
        o.ranges = _bytes_view(img, il.ranges, np.uint32, T * 2).reshape(T, 2)
        o.point_list = _bytes_view(binning, bl.point_list, np.uint32, R) if R > 0 else np.zeros(0, np.uint32)
        o.keys = _bytes_view(binning, bl.point_list_keys, np.uint64, R) if R > 0 else np.zeros(0, np.uint64)
    else:
        # reference layouts: SURVEY.md Appendix B (each field at the next 128-byte boundary)
        off = 0
        depths_o = off; off = _al(off + 4 * P)
        clamped_o = off; off = _al(off + 3 * P)
        radii_o = off; off = _al(off + 4 * P)
        means2D_o = off; off = _al(off + 8 * P)
        cov3D_o = off; off = _al(off + 24 * P)
        conic_o = off; off = _al(off + 16 * P)
        rgb_o = off; off = _al(off + 12 * P)
        tiles_o = off
        o.tiles_touched = _bytes_view(geom, tiles_o, np.uint32, P)
        o.point_offsets = np.cumsum(o.tiles_touched.astype(np.uint64)).astype(np.uint32)
        o.means2D = _bytes_view(geom, means2D_o, np.float32, 2 * P).reshape(P, 2)
        o.conic_opacity = _bytes_view(geom, conic_o, np.float32, 4 * P).reshape(P, 4)
        o.depths = _bytes_view(geom, depths_o, np.float32, P)
        o.cov3D = _bytes_view(geom, cov3D_o, np.float32, 6 * P).reshape(P, 6)
        off = 0
        o.final_T = _bytes_view(img, off, np.float32, N).reshape(H, W); off = _al(off + 4 * N)
        o.n_contrib = _bytes_view(img, off, np.uint32, N).reshape(H, W); off = _al(off + 4 * N)
        o.ranges = _bytes_view(img, off, np.uint32, 2 * T).reshape(T, 2)
        off = 0
        o.point_list = _bytes_view(binning, off, np.uint32, R) if R > 0 else np.zeros(0, np.uint32)
        off = _al(off + 4 * R); off = _al(off + 4 * R)
        o.keys = _bytes_view(binning, off, np.uint64, R) if R > 0 else np.zeros(0, np.uint64)
    # entries of culled Gaussians are never written by either implementation: mask them out
    vis = o.radii > 0
    for name in ("means2D", "conic_opacity", "depths"):
        a = getattr(o, name)
        a[~vis] = 0
    if not np.all(vis):
        o.cov3D = o.cov3D.copy()
        o.cov3D[~vis] = 0


def run_oracle(sc, K: int, depth: bool = False, use_sh: bool = False, sh_degree: int = 0, backward: bool = True,
               bg=None, nthreads: int = 1):
    from oracle import oracle
    g, c = sc.gauss, sc.cam
    bg_np = (np.zeros(max(K, 3), np.float32) if bg is None else bg.numpy())
    mask = None
    if depth:
        mask = (torch.rand(sc.P, 1, generator=torch.Generator().manual_seed(7)) * 0.5 + 0.5).numpy().reshape(-1)
    fw = oracle.forward(means3D=g.means3D.numpy(), opacities=g.opacities.numpy(), bg=bg_np,
                        viewmatrix=c.world_view_transform.numpy(), projmatrix=c.full_proj_transform.numpy(),
                        campos=c.camera_center.numpy(), image_height=sc.H, image_width=sc.W, tanfovx=c.tanfovx,
                        tanfovy=c.tanfovy, sh_degree=sh_degree, shs=g.shs.numpy() if use_sh else None,
                        colors_precomp=None if use_sh else g.colors.numpy(), scales=g.scales.numpy(),
                        rotations=g.rotations.numpy(), mask=mask, num_channels=K, nthreads=nthreads)
    o = SimpleNamespace(kind="oracle", variant=variant_of(K, depth))
    o.color, o.radii, o.final_T, o.n_contrib = fw.color, fw.radii, fw.final_T, fw.n_contrib
    o.out_mask = fw.out_mask if depth else None
    o.out_depth = fw.out_depth if depth else None
    o.tiles_touched, o.point_offsets, o.num_rendered = fw.tiles_touched, fw.point_offsets, fw.num_rendered
    o.point_list, o.keys, o.ranges = fw.point_list, fw.keys, fw.ranges
    vis = fw.radii > 0   # per-Gaussian scratch of culled Gaussians is unspecified in every implementation
    o.means2D, o.conic_opacity, o.depths, o.cov3D = (np.where(vis[:, None], fw.means2D, 0), np.where(vis[:, None], fw.conic_opacity, 0),
                                                      np.where(vis, fw.depths, 0), np.where(vis[:, None], fw.cov3D, 0))
    if backward:
        bw = oracle.backward(fw, sc.dL_dout[:K].numpy(), sc.dL_dmask.numpy() if depth else None, nthreads=nthreads)
        o.g_means3D, o.g_means2D, o.g_opacity = bw.means3D, bw.means2D, bw.opacity
        o.g_scales, o.g_rotations, o.g_cov3D = bw.scales, bw.rotations, bw.cov3D
        o.g_colors = None if use_sh else bw.colors
        o.g_sh = bw.sh if use_sh else None
        o.g_mask = bw.mask.reshape(-1) if depth else None
    return o


# ----------------------------------------------------------------------------------------------
# comparison
# ----------------------------------------------------------------------------------------------
def float_err(a, b):
    """(max elementwise violation ratio w.r.t. the tolerance, max abs diff, max |ref|)."""
    a = np.asarray(a, np.float64).reshape(-1)
    b = np.asarray(b, np.float64).reshape(-1)
    if a.size == 0:
        return 0.0, 0.0, 0.0
    scale = float(np.max(np.abs(b)))
    tol = RTOL * np.maximum(np.abs(a), np.abs(b)) + ATOL_SCALE * scale + 1e-30
    d = np.abs(a - b)
    return float(np.max(d / tol)), float(np.max(d)), scale


# ----------------------------------------------------------------------------------------------
# sampled golden vectors: outputs of the unmodified reference too large to store whole
# ----------------------------------------------------------------------------------------------
GOLDEN_SAMPLES = 128
GOLDEN_BLOCKS = 32


def _block_sums(flat: np.ndarray, nblocks: int) -> np.ndarray:
    """(sum a, sum |a|) over each of ``nblocks`` contiguous, near-equal blocks of a flat array, in float64: shape (2, nblocks)."""
    f = np.asarray(flat, np.float64)
    edges = (np.arange(nblocks, dtype=np.int64) * f.size) // nblocks
    return np.stack([np.add.reduceat(f, edges), np.add.reduceat(np.abs(f), edges)])


def digest(a) -> np.ndarray:
    """SHA-256 of an array's shape, dtype and bytes, as 32 uint8: stands in for the array where equality must be exact."""
    import hashlib
    a = np.ascontiguousarray(np.asarray(a))
    h = hashlib.sha256(repr((a.shape, a.dtype.str)).encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def summarize(name: str, a, exact: bool = False, samples: int = GOLDEN_SAMPLES, seed: int = 0) -> dict:
    """The entries a sampled golden file keeps of one array: its digest when it must match exactly; otherwise a seeded
    sample of elements (most of them where the array is non-zero), ``meta`` = (max |a|, sum |a|, *shape) and ``blocks`` =
    sum a and sum |a| over GOLDEN_BLOCKS contiguous blocks of the flat array (for a per-Gaussian array: ranges of Gaussians;
    for an image: bands of rows).  max |a| is the tolerance's absolute scale (float_err), so a sampled comparison applies the
    same bound as one over the whole array."""
    a = np.asarray(a)
    if exact:
        return {name + ".digest": digest(a)}
    flat = a.reshape(-1).astype(np.float32)
    rng = np.random.default_rng(seed)
    nz = np.flatnonzero(flat)
    parts = [rng.choice(flat.size, min(samples // 4, flat.size), replace=False)]
    if nz.size:
        parts.append(rng.choice(nz, min(samples - parts[0].size, nz.size), replace=False))
    idx = np.unique(np.concatenate(parts)).astype(np.int32)
    meta = [np.abs(flat).max() if flat.size else 0.0, np.abs(flat.astype(np.float64)).sum()] + list(a.shape)
    return {name + ".idx": idx, name + ".val": flat[idx], name + ".meta": np.array(meta, np.float64),
            name + ".blocks": _block_sums(flat, min(GOLDEN_BLOCKS, flat.size)).astype(np.float32)}


def check_summary(z, name: str, a, rtol: float = RTOL, atol_scale: float = ATOL_SCALE):
    """Compare an array with its entries in a sampled golden file ``z``.  Returns (ok, report line).

    Sampled elements must meet the elementwise bound of float_err (scale = max |ref| of the whole array).  max |a|, sum |a|
    and, per block, sum a and sum |a| are checked against the bounds that the elementwise one implies for them
    (|sum a - sum b| <= sum |a - b| <= rtol * (sum |a| + sum |b|) + atol_scale * scale * n), so an error confined to a part of
    the array (a range of Gaussians, a band of rows) that is large enough to move its block's sums is caught even where no
    sample lies.  The block sums are stored in float32: their rounding (1e-6 of the block's sum |ref|) is allowed for."""
    if name + ".digest" in z:
        ok = np.array_equal(digest(a), z[name + ".digest"])
        return ok, f"  EXACT {name:22s} " + ("equal" if ok else "DIFFERS")
    a = np.asarray(a)
    meta = z[name + ".meta"]
    scale, ref_sum, shape = float(meta[0]), float(meta[1]), tuple(int(s) for s in meta[2:])
    if a.shape != shape:
        return False, f"  FLOAT {name:22s} shape {a.shape} vs {shape}  MISMATCH"
    flat = np.asarray(a, np.float64).reshape(-1)
    x, v = flat[z[name + ".idx"]], np.asarray(z[name + ".val"], np.float64)
    r = d = 0.0
    if x.size:
        diff = np.abs(x - v)
        r = float(np.max(diff / (rtol * np.maximum(np.abs(x), np.abs(v)) + atol_scale * scale + 1e-30)))
        d = float(diff.max())
    amax, asum = float(np.abs(flat).max()) if flat.size else 0.0, float(np.abs(flat).sum())
    max_ok = abs(amax - scale) <= rtol * max(amax, scale) + atol_scale * scale + 1e-30
    sum_ok = abs(asum - ref_sum) <= rtol * (asum + ref_sum) + atol_scale * scale * flat.size + 1e-30
    ref_blocks = np.asarray(z[name + ".blocks"], np.float64)
    nb = ref_blocks.shape[1]
    blocks = _block_sums(flat, nb)
    n_b = np.diff(np.append((np.arange(nb, dtype=np.int64) * flat.size) // nb, flat.size))
    block_tol = rtol * (blocks[1] + ref_blocks[1]) + atol_scale * scale * n_b + 1e-6 * ref_blocks[1] + 1e-30
    block_r = float(np.max(np.abs(blocks - ref_blocks) / block_tol)) if nb else 0.0
    ok = r <= 1.0 and max_ok and sum_ok and block_r <= 1.0 and not bool(np.isnan(flat).any())
    return ok, (f"  FLOAT {name:22s} samples={z[name + '.idx'].size} max|d|={d:.3e} tol-ratio={r:.3f} max|a|={amax:.6e}/{scale:.6e} "
                f"sum|a|={asum:.6e}/{ref_sum:.6e} block-tol-ratio={block_r:.3f}" + ("" if ok else "  MISMATCH"))


# what a sampled golden file keeps of a runner output (run_torch_impl): integer state and final_T exactly, the rest sampled
SUMMARY_EXACT = INT_FWD + ("final_T",)
SUMMARY_FLOAT = ("color", "out_mask", "out_depth") + GRADS + ("means2D", "conic_opacity", "depths", "cov3D")


def summary_arrays(o) -> dict:
    """``{name: array}`` of a runner output for compare_summaries (fields the runner left as None are absent)."""
    return {f: getattr(o, f) for f in SUMMARY_EXACT + SUMMARY_FLOAT if getattr(o, f, None) is not None}


def summarize_all(arrays: dict, exact=()) -> dict:
    out = {}
    for name, a in arrays.items():
        out.update(summarize(name, a, exact=name in exact))
    return out


def compare_summaries(z, arrays: dict, skip=()):
    """check_summary over ``{name: array}``; every name in the file but those in ``skip`` must be given.
    Returns (ok, report lines)."""
    stored = {f.rsplit(".", 1)[0] for f in z.files if f != "config"} - set(skip)
    lines = [f"  names: stored {sorted(stored)} given {sorted(arrays)}"] if stored != set(arrays) else []
    ok = not lines
    for name in sorted(set(arrays) & stored):
        o, line = check_summary(z, name, arrays[name])
        ok &= o
        lines.append(line)
    return ok, lines


def compare(a, b, ints=INT_FWD, floats=FLOAT_FWD + GRADS, verbose=True):
    """Compare two runner outputs. Returns (ok, report lines)."""
    ok = True
    lines = []
    for name in ints:
        x, y = getattr(a, name, None), getattr(b, name, None)
        if x is None or y is None:
            continue
        x, y = np.asarray(x), np.asarray(y)
        if x.shape != y.shape:
            ok = False
            lines.append(f"  INT   {name:14s} shape {x.shape} vs {y.shape}  MISMATCH")
            continue
        nbad = int(np.count_nonzero(x != y))
        if nbad:
            ok = False
        lines.append(f"  INT   {name:14s} n={x.size:9d} mismatches={nbad}" + ("  MISMATCH" if nbad else ""))
    for name in floats:
        x, y = getattr(a, name, None), getattr(b, name, None)
        if x is None or y is None:
            continue
        x, y = np.asarray(x), np.asarray(y)
        if x.size != y.size:
            ok = False
            lines.append(f"  FLOAT {name:14s} shape {x.shape} vs {y.shape}  MISMATCH")
            continue
        r, d, s = float_err(x, y)
        bad = not (r <= 1.0) or bool(np.isnan(x).any())
        if bad:
            ok = False
        lines.append(f"  FLOAT {name:14s} max|d|={d:.3e} max|ref|={s:.3e} rel={d / (s + 1e-30):.2e} tol-ratio={r:.3f}" +
                     ("  MISMATCH" if bad else ""))
    if verbose:
        print(f"compare {a.kind} vs {b.kind} [{a.variant}]: {'OK' if ok else 'FAIL'}")
        print("\n".join(lines))
    return ok, lines
