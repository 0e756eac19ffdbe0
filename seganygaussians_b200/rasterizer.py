"""Host-side mirror of the reference's operator API for the rasterizer hot path.

Same names, argument meaning, return tuples and error behaviour as the reference's three packages

* ``diff_gaussian_rasterization``                (BASE, 3 channels)   -- ``.../diff_gaussian_rasterization/__init__.py``
* ``diff_gaussian_rasterization_contrastive_f``  (CF, 32 channels)    -- ``.../diff_gaussian_rasterization_contrastive_f/__init__.py:21-219``
* ``diff_gaussian_rasterization_depth``          (DEPTH, 3 + mask + depth) -- ``.../diff_gaussian_rasterization_depth/__init__.py:21-391``

but backed by ``libsagars.so`` (hand-written sm_100a kernels behind the C ABI of ``include/sagars.h``)
instead of the pybind ``_C`` module.  PyTorch is only plumbing here: it owns device memory (outputs
and the three scratch buffers handed to the library through allocator callbacks), the stream, and
autograd.  There is no CPU or eager fallback: a missing library raises.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

from . import _lib


class GaussianRasterizationSettings(NamedTuple):
    """Field-for-field the reference's settings tuple (CF ``__init__.py:156-168``)."""
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


def cpu_deep_copy_tuple(input_tuple):
    copied = [item.cpu().clone() if isinstance(item, torch.Tensor) else item for item in input_tuple]
    return tuple(copied)


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
def _f32(t: Optional[torch.Tensor], device) -> Optional[torch.Tensor]:
    """contiguous fp32 on `device`, or None for an absent (None / 0-element) optional input.

    The reference maps 0-element CPU tensors to nullptr (CF ``__init__.py:196-206``)."""
    if t is None or t.numel() == 0:
        return None
    if t.device != device or t.dtype != torch.float32:
        t = t.to(device=device, dtype=torch.float32)
    t = t.contiguous()
    if t.data_ptr() % 16:       # the kernels read rows as float4 / 16-byte async copies: a contiguous VIEW at an odd storage offset
        t = t.clone()           # (e.g. a slice of a flat parameter buffer) gets its own 256-byte-aligned allocation
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class _Scratch:
    """Allocator callbacks: torch owns the three scratch buffers, like the reference's resize lambdas
    (CF ``rasterize_points.cu:27-33``).

    One instance per thread, reused by every forward call: the three ctypes callback objects are created once, and no
    reference cycle (callback -> closure -> instance -> callback) is left behind per call.  A per-call instance with such
    a cycle kept the previous calls' scratch buffers alive until the cyclic garbage collector ran, which turned the next
    ``torch.empty`` into a ``cudaMalloc`` (measured: 1-2 ms inside the geometry-buffer callback every few calls)."""

    def __init__(self):
        self.device = None
        self.buffers = [None, None, None]
        self.error = None
        self._cbs = [_lib.ALLOC_FN(self._make(i)) for i in range(3)]

    def _make(self, i):
        def alloc(_user, nbytes):
            try:
                buf = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
                self.buffers[i] = buf
                return buf.data_ptr()
            except BaseException as e:  # pragma: no cover - reported through EALLOC
                self.error = e
                return None
        return alloc

    def begin(self, device):
        self.device = device
        self.buffers = [None, None, None]
        self.error = None

    def take(self):
        """Hand the buffers to the caller and drop every reference held here."""
        bufs, err = self.buffers, self.error
        self.buffers = [None, None, None]
        self.error = None
        return bufs, err

    def cb(self, i):
        return self._cbs[i]


_TLS = threading.local()


def _scratch_for_thread() -> "_Scratch":
    s = getattr(_TLS, "scratch", None)
    if s is None:
        s = _TLS.scratch = _Scratch()
    return s


def _stream_ptr(device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def _flags(settings: GaussianRasterizationSettings, extra: int = 0) -> int:
    f = extra
    if settings.prefiltered:
        f |= _lib.FLAG_PREFILTERED
    if settings.debug:
        f |= _lib.FLAG_DEBUG
    if _USE_CUB_SORT:
        f |= _lib.FLAG_CUB_SORT
    if not _USE_TENSOR_CORES:
        f |= _lib.FLAG_NO_TENSOR_CORES
    if _FORWARD_KERNEL == "tile":
        f |= _lib.FLAG_FWD_TILE
    elif _FORWARD_KERNEL == "warp_any":
        f |= _lib.FLAG_FWD_WARP_ANY
    if _BACKWARD_KERNEL == "tile":
        f |= _lib.FLAG_BWD_TILE
    elif _BACKWARD_KERNEL == "tc":
        f |= _lib.FLAG_BWD_TC
    if _BINNING == "tile_sort":
        f |= _lib.FLAG_TILE_SORT
    elif _BINNING == "depth_first":
        f |= _lib.FLAG_DEPTH_FIRST
    return f


_USE_CUB_SORT = False
_USE_TENSOR_CORES = True
_FORWARD_KERNEL = "default"    # "default": mma.sync warp kernel at K = 32, fp32 SIMT otherwise; "tile": tcgen05 tile kernel at
                               # K = 32; "warp_any": the warp kernel for every colour-only channel count
_BACKWARD_KERNEL = "default"   # "default": one warp per 8x4 pixel block (mma.sync); "tile": one CTA per 16x16 tile (mma.sync);
                               # "tc": tcgen05 / TMEM kernel, one CTA per 16x8 pixel group (C = 32 precomputed colours)
_BINNING = "depth_first"       # "depth_first" (default): Gaussians sorted by depth, instances emitted in that order, one stable sort on
                               # the tile bits; "radix": the reference's scheme -- global LSD radix sort of the duplicated tile|depth
                               # keys; "tile_sort": per-tile counts -> scan -> scatter -> one CTA per tile sorts its segment
                               # (measured slower, round 2).  All three leave bit-identical binning state.
_SPECULATIVE_BINNING = True
# (device index, P, W, H) -> largest instance count seen so far: the next forward of that shape asks for a binning
# buffer 25 % larger than this BEFORE the count is known (include/sagars.h, `binning_capacity_hint`)
_CAPACITY_SEEN: dict = {}
# capacity the binning buffer of the most recent forward was laid out for (tests decode the scratch with it)
last_binning_capacity = 0


def set_speculative_binning(enabled: bool) -> None:
    """Queue sort / ranges / blend behind a capacity guess instead of waiting for the instance count (default on).
    Off: the reference's order -- read the count back, then size the binning buffer exactly."""
    global _SPECULATIVE_BINNING
    _SPECULATIVE_BINNING = bool(enabled)
    _CAPACITY_SEEN.clear()


def set_tensor_cores(enabled: bool) -> None:
    """Route the K=32 blend through the tensor cores (default) or through the fp32 SIMT kernels (bit-exact colours)."""
    global _USE_TENSOR_CORES
    _USE_TENSOR_CORES = bool(enabled)


def set_blend_kernels(forward: str = "default", backward: str = "default") -> None:
    """Select between the tensor-core blend kernel variants (all give the same results to fp32 rounding)."""
    global _FORWARD_KERNEL, _BACKWARD_KERNEL
    if forward not in ("default", "tile", "warp_any") or backward not in ("default", "tile", "tc"):
        raise ValueError("forward in {'default', 'tile', 'warp_any'}, backward in {'default', 'tile', 'tc'}")
    _FORWARD_KERNEL, _BACKWARD_KERNEL = forward, backward


_BLEND_WAIT_EVENT = None       # torch.cuda.Event the NEXT forward's blend stage waits for (set_blend_wait_event)


def set_blend_wait_event(event) -> None:
    """Gate the blend stage of the NEXT forward on a recorded ``torch.cuda.Event`` (``blend_wait_event`` of include/sagars.h).
    The geometry stages (preprocess, binning) of that forward run ahead of the event; only the stage that reads the features
    waits.  A data-parallel trainer records the event on the stream that all-reduces the feature gradient and applies the
    optimiser step (``data_parallel.FeatureGradReducer.ready_event``): the exchange then overlaps the next forward's geometry
    stages.  One-shot; ``None`` clears it."""
    global _BLEND_WAIT_EVENT
    _BLEND_WAIT_EVENT = event


def set_binning(method: str = "depth_first") -> None:
    """How the (Gaussian, tile) instances are ordered: "radix" (the library's global radix sort of the R duplicated tile|depth
    keys, as the reference does with CUB), "depth_first" (``SAGARS_FLAG_DEPTH_FIRST``: sort the P Gaussians by depth, emit their
    instances in that order, one stable sort on the tile bits) or "tile_sort" (``SAGARS_FLAG_TILE_SORT``: no global sort, every
    tile's segment is sorted by its own CTA).  Bit-identical results."""
    global _BINNING
    if method not in ("radix", "tile_sort", "depth_first"):
        raise ValueError("method in {'radix', 'depth_first', 'tile_sort'}")
    _BINNING = method


def set_cub_sort(enabled: bool) -> None:
    """Test hook: route the binning sort through cub::DeviceRadixSort (cross-check of the library's own sort)."""
    global _USE_CUB_SORT
    _USE_CUB_SORT = bool(enabled)


def _check_means(means3D: torch.Tensor):
    if means3D.dim() != 2 or means3D.shape[1] != 3:
        # same message as CF rasterize_points.cu:57-59
        raise RuntimeError("means3D must have dimensions (num_points, 3)")
    if not means3D.is_cuda:
        raise RuntimeError("means3D must be a CUDA tensor (libsagars has no CPU path)")


def _forward_impl(settings, variant_flags, default_channels, means3D, sh, colors_precomp, opacities, mask,
                  scales, rotations, cov3Ds_precomp):
    """Shared forward: returns (num_rendered, color, out_mask, out_depth, radii, geom, binning, img, C)."""
    lib = _lib.load()
    _check_means(means3D)
    device = means3D.device
    P = int(means3D.shape[0])
    H, W = int(settings.image_height), int(settings.image_width)
    mask_only = bool(variant_flags & _lib.FLAG_MASK_ONLY)
    has_md = bool(variant_flags & (_lib.FLAG_MASK_DEPTH | _lib.FLAG_MASK_ONLY))

    means3D_c = _f32(means3D, device)
    sh_c = _f32(sh, device)
    colors_c = _f32(colors_precomp, device)
    opac_c = _f32(opacities, device)
    mask_c = _f32(mask, device) if has_md else None
    scales_c = _f32(scales, device)
    rots_c = _f32(rotations, device)
    cov_c = _f32(cov3Ds_precomp, device)
    bg_c = _f32(settings.bg, device)
    view_c = _f32(settings.viewmatrix, device)
    proj_c = _f32(settings.projmatrix, device)
    campos_c = _f32(settings.campos, device)

    if colors_c is not None:
        if colors_c.dim() != 2 or colors_c.shape[0] != P:
            raise RuntimeError("colors_precomp must have dimensions (num_points, num_channels)")
        num_ch = int(colors_c.shape[1])
    else:
        num_ch = default_channels
    M = 0
    if sh_c is not None:
        M = int(sh_c.shape[1])
    # cheap shape checks: a short tensor must become an error here, not an out-of-bounds read on the device
    for name, t, n in (("opacities", opac_c, P), ("mask", mask_c, P), ("scales", scales_c, 3 * P), ("rotations", rots_c, 4 * P),
                       ("cov3D_precomp", cov_c, 6 * P), ("shs", sh_c, 3 * M * P)):
        if t is not None and t.numel() != n:
            raise RuntimeError(f"{name} has {t.numel()} elements, expected {n} for {P} points")
    if P > 0 and opac_c is None:
        raise RuntimeError("opacities must have dimensions (num_points, 1)")
    if P > 0 and has_md and mask_c is None:
        raise RuntimeError("mask must have dimensions (num_points,)")
    if sh_c is not None and (int(settings.sh_degree) + 1) ** 2 > M:
        raise RuntimeError(f"sh_degree {int(settings.sh_degree)} needs {(int(settings.sh_degree) + 1) ** 2} coefficients, shs has {M}")
    if bg_c is None or bg_c.numel() < (1 if mask_only else num_ch):
        raise RuntimeError(f"bg must hold at least {num_ch} floats")

    with torch.cuda.device(device):
        opts = dict(dtype=torch.float32, device=device)
        if P == 0:
            # nothing is launched; zero-filled outputs like CF rasterize_points.cu:68-81
            color = torch.zeros((num_ch, H, W), **opts)
            radii = torch.zeros((0,), dtype=torch.int32, device=device)
            om = torch.zeros((1, H, W), **opts) if has_md else None
            od = torch.zeros((1, H, W), **opts) if (has_md and not mask_only) else None
            empty = torch.empty(0, dtype=torch.uint8, device=device)
            return 0, color, om, od, radii, empty, empty, empty, num_ch

        color = None if mask_only else torch.empty((num_ch, H, W), **opts)
        out_mask = torch.empty((1, H, W), **opts) if has_md else None
        out_depth = torch.empty((1, H, W), **opts) if (has_md and not mask_only) else None
        radii = torch.empty((P,), dtype=torch.int32, device=device)

        a = _lib.ForwardArgs()
        a.device = device.index if device.index is not None else torch.cuda.current_device()
        a.flags = _flags(settings, variant_flags)
        _TLS.last_flags = int(a.flags)       # the matching backward reuses exactly these (set_* calls in between must not split a pair)
        a.P, a.D, a.M, a.num_channels = P, int(settings.sh_degree), M, num_ch
        a.width, a.height = W, H
        a.tan_fovx, a.tan_fovy = float(settings.tanfovx), float(settings.tanfovy)
        a.scale_modifier = float(settings.scale_modifier)
        a.background = _ptr(bg_c)
        a.means3D = _ptr(means3D_c)
        a.shs = _ptr(sh_c)
        a.colors_precomp = _ptr(colors_c)
        a.opacities = _ptr(opac_c)
        a.mask = _ptr(mask_c)
        a.scales = _ptr(scales_c)
        a.rotations = _ptr(rots_c)
        a.cov3D_precomp = _ptr(cov_c)
        a.viewmatrix = _ptr(view_c)
        a.projmatrix = _ptr(proj_c)
        a.cam_pos = _ptr(campos_c)
        a.out_color = _ptr(color)
        a.out_mask = _ptr(out_mask)
        a.out_depth = _ptr(out_depth)
        a.radii = _ptr(radii)
        cap_key = (a.device, P, W, H)
        seen = _CAPACITY_SEEN.get(cap_key, 0) if _SPECULATIVE_BINNING else 0
        a.binning_capacity_hint = min(seen + seen // 4 + 4096, 2**31 - 1) if seen > 0 else 0
        cap_out = C.c_int32(0)
        a.binning_capacity_out = C.pointer(cap_out)
        global _BLEND_WAIT_EVENT
        gate = _BLEND_WAIT_EVENT
        _BLEND_WAIT_EVENT = None                      # one-shot: it gates exactly the next forward
        if gate is not None:
            handle = gate.cuda_event                  # cudaEvent_t of a RECORDED torch.cuda.Event (int; c_void_p in old versions)
            a.blend_wait_event = int(getattr(handle, "value", handle))
        else:
            a.blend_wait_event = None

        scratch = _scratch_for_thread()
        scratch.begin(device)
        num_rendered = C.c_int32(0)
        rc = lib.sagars_forward(C.byref(a), scratch.cb(0), None, scratch.cb(1), None, scratch.cb(2), None,
                                C.byref(num_rendered), _stream_ptr(device))
        (geom, binning, img), alloc_error = scratch.take()
        if alloc_error is not None:
            raise alloc_error
        _lib.check(rc)
        global last_binning_capacity
        last_binning_capacity = int(cap_out.value)
        if _SPECULATIVE_BINNING and num_rendered.value > seen:
            _CAPACITY_SEEN[cap_key] = int(num_rendered.value)
        if binning is None:
            binning = torch.empty(0, dtype=torch.uint8, device=device)
    return int(num_rendered.value), color, out_mask, out_depth, radii, geom, binning, img, num_ch


def _backward_impl(settings, variant_flags, num_ch, num_rendered, means3D, radii, colors_precomp, mask, scales,
                   rotations, cov3Ds_precomp, sh, geom, binning, img, grad_out_color, grad_out_mask, flags=None):
    """Shared backward: returns dict of gradient tensors (reference shapes, CF rasterize_points.cu:151-159).
    `flags`: the flags the matching forward ran with (None: current module settings)."""
    lib = _lib.load()
    device = means3D.device
    P = int(means3D.shape[0])
    mask_only = bool(variant_flags & _lib.FLAG_MASK_ONLY)
    has_md = bool(variant_flags & (_lib.FLAG_MASK_DEPTH | _lib.FLAG_MASK_ONLY))
    if mask_only:
        H, W = int(grad_out_mask.shape[1]), int(grad_out_mask.shape[2])
    else:
        H, W = int(grad_out_color.shape[1]), int(grad_out_color.shape[2])

    means3D_c = _f32(means3D, device)
    sh_c = _f32(sh, device)
    colors_c = _f32(colors_precomp, device)
    scales_c = _f32(scales, device)
    rots_c = _f32(rotations, device)
    cov_c = _f32(cov3Ds_precomp, device)
    bg_c = _f32(settings.bg, device)
    view_c = _f32(settings.viewmatrix, device)
    proj_c = _f32(settings.projmatrix, device)
    campos_c = _f32(settings.campos, device)
    gcol_c = _f32(grad_out_color, device) if not mask_only else None
    gmask_c = _f32(grad_out_mask, device) if has_md else None
    M = int(sh_c.shape[1]) if sh_c is not None else 0

    with torch.cuda.device(device):
        opts = dict(dtype=torch.float32, device=device)
        if P == 0:
            z = lambda *s: torch.zeros(s, **opts)
            return dict(means2D=z(0, 3), colors=z(0, num_ch), opacity=z(0, 1), mask=z(0, 1), means3D=z(0, 3),
                        cov3D=z(0, 6), sh=z(0, M, 3), scales=z(0, 3), rotations=z(0, 4))
        e = lambda *s: torch.empty(s, **opts)
        if mask_only:   # the only gradient of the mask-only path is dL_dmask (DEPTH __init__.py:280-289): nothing else is allocated
            g = dict(means2D=None, colors=None, opacity=None, means3D=None, cov3D=None, sh=None, scales=None, rotations=None)
        else:
            g = dict(means2D=e(P, 3), colors=e(P, num_ch), opacity=e(P, 1), means3D=e(P, 3), cov3D=e(P, 6),
                     sh=e(P, M, 3), scales=e(P, 3), rotations=e(P, 4))
        g["mask"] = e(P, 1) if has_md else None
        scratch = torch.empty(int(lib.sagars_grad_scratch_bytes(P)), dtype=torch.uint8, device=device)

        a = _lib.BackwardArgs()
        a.device = device.index if device.index is not None else torch.cuda.current_device()
        a.flags = int(flags) if flags is not None else _flags(settings, variant_flags)
        a.P, a.D, a.M, a.R = P, int(settings.sh_degree), M, int(num_rendered)
        a.num_channels = num_ch
        a.width, a.height = W, H
        a.tan_fovx, a.tan_fovy = float(settings.tanfovx), float(settings.tanfovy)
        a.scale_modifier = float(settings.scale_modifier)
        a.background = _ptr(bg_c)
        a.means3D = _ptr(means3D_c)
        a.shs = _ptr(sh_c)
        a.colors_precomp = _ptr(colors_c)
        a.mask = _ptr(_f32(mask, device)) if has_md else None
        a.scales = _ptr(scales_c)
        a.rotations = _ptr(rots_c)
        a.cov3D_precomp = _ptr(cov_c)
        a.viewmatrix = _ptr(view_c)
        a.projmatrix = _ptr(proj_c)
        a.cam_pos = _ptr(campos_c)
        a.radii = _ptr(radii)
        a.geom_buffer = _ptr(geom)
        a.binning_buffer = _ptr(binning) if binning.numel() > 0 else None
        a.image_buffer = _ptr(img)
        a.dL_dout_color = _ptr(gcol_c)
        a.dL_dout_mask = _ptr(gmask_c)
        a.grad_scratch = _ptr(scratch)
        a.dL_dmeans2D = _ptr(g["means2D"])
        a.dL_dopacity = _ptr(g["opacity"])
        a.dL_dcolors = _ptr(g["colors"])
        a.dL_dmask = _ptr(g["mask"])
        a.dL_dmeans3D = _ptr(g["means3D"])
        a.dL_dcov3D = _ptr(g["cov3D"])
        a.dL_dsh = _ptr(g["sh"]) if (M > 0 and not mask_only) else None
        a.dL_dscales = _ptr(g["scales"])
        a.dL_drotations = _ptr(g["rotations"])
        _lib.check(lib.sagars_backward(C.byref(a), _stream_ptr(device)))
    return g


# ----------------------------------------------------------------------------------------------
# autograd functions (one per reference variant; argument order = the reference's)
# ----------------------------------------------------------------------------------------------
def _make_rasterize_function(default_channels: int):
    class _RasterizeGaussians(torch.autograd.Function):
        """CF ``__init__.py:44-154``: forward returns (color[C,H,W], radii[P]); backward returns the nine
        input gradients in input order."""

        @staticmethod
        def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                    raster_settings):
            args = (means3D, sh, colors_precomp, opacities, None, scales, rotations, cov3Ds_precomp)
            if raster_settings.debug:
                cpu_args = cpu_deep_copy_tuple((raster_settings.bg,) + args)
                try:
                    out = _forward_impl(raster_settings, 0, default_channels, *args)
                except Exception as ex:
                    torch.save(cpu_args, "snapshot_fw.dump")
                    print("\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
                    raise ex
            else:
                out = _forward_impl(raster_settings, 0, default_channels, *args)
            num_rendered, color, _, _, radii, geom, binning, img, num_ch = out
            ctx.raster_settings = raster_settings
            ctx.sagars_flags = getattr(_TLS, "last_flags", None)
            ctx.num_rendered = num_rendered
            ctx.num_ch = num_ch
            ctx.save_for_backward(colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, img)
            ctx.mark_non_differentiable(radii)
            return color, radii

        @staticmethod
        def backward(ctx, grad_out_color, _):
            rs = ctx.raster_settings
            colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, img = ctx.saved_tensors
            call = lambda: _backward_impl(rs, 0, ctx.num_ch, ctx.num_rendered, means3D, radii, colors_precomp, None,
                                          scales, rotations, cov3Ds_precomp, sh, geom, binning, img, grad_out_color, None,
                                          flags=ctx.sagars_flags)
            if rs.debug:
                cpu_args = cpu_deep_copy_tuple((rs.bg, means3D, radii, colors_precomp, scales, rotations, cov3Ds_precomp,
                                                grad_out_color, sh, geom, binning, img))
                try:
                    g = call()
                except Exception as ex:
                    torch.save(cpu_args, "snapshot_bw.dump")
                    print("\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
                    raise ex
            else:
                g = call()
            return (g["means3D"], g["means2D"], g["sh"], g["colors"], g["opacity"], g["scales"], g["rotations"],
                    g["cov3D"], None)

    return _RasterizeGaussians


class _RasterizeGaussiansDepth(torch.autograd.Function):
    """DEPTH ``__init__.py:67-182``: forward returns (color, mask[1,H,W], depth[1,H,W], radii); the depth
    output is not differentiable (its upstream gradient is ignored, like the reference)."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, mask, scales, rotations, cov3Ds_precomp,
                raster_settings):
        args = (means3D, sh, colors_precomp, opacities, mask, scales, rotations, cov3Ds_precomp)
        if raster_settings.debug:
            cpu_args = cpu_deep_copy_tuple((raster_settings.bg,) + args)
            try:
                out = _forward_impl(raster_settings, _lib.FLAG_MASK_DEPTH, 3, *args)
            except Exception as ex:
                torch.save(cpu_args, "snapshot_fw.dump")
                print("\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
                raise ex
        else:
            out = _forward_impl(raster_settings, _lib.FLAG_MASK_DEPTH, 3, *args)
        num_rendered, color, out_mask, out_depth, radii, geom, binning, img, num_ch = out
        ctx.raster_settings = raster_settings
        ctx.sagars_flags = getattr(_TLS, "last_flags", None)
        ctx.num_rendered = num_rendered
        ctx.num_ch = num_ch
        ctx.mask_shape = tuple(mask.shape)
        ctx.save_for_backward(colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, img)
        ctx.mark_non_differentiable(radii)
        return color, out_mask, out_depth, radii

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_mask, grad_out_depth, _):
        rs = ctx.raster_settings
        colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, img = ctx.saved_tensors
        call = lambda: _backward_impl(rs, _lib.FLAG_MASK_DEPTH, ctx.num_ch, ctx.num_rendered, means3D, radii,
                                      colors_precomp, None, scales, rotations, cov3Ds_precomp, sh, geom, binning, img,
                                      grad_out_color, grad_out_mask, flags=ctx.sagars_flags)
        if rs.debug:
            cpu_args = cpu_deep_copy_tuple((rs.bg, means3D, radii, colors_precomp, scales, rotations, cov3Ds_precomp,
                                            grad_out_color, grad_out_mask, sh, geom, binning, img))
            try:
                g = call()
            except Exception as ex:
                torch.save(cpu_args, "snapshot_bw.dump")
                print("\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
                raise ex
        else:
            g = call()
        # the reference returns dL_dmask as [P,1] (DEPTH rasterize_points.cu:167); autograd needs the input's shape
        grad_mask = g["mask"].reshape(ctx.mask_shape) if g["mask"] is not None else None
        return (g["means3D"], g["means2D"], g["sh"], g["colors"], g["opacity"], grad_mask, g["scales"],
                g["rotations"], g["cov3D"], None)


class _RasterizeMaskGaussians(torch.autograd.Function):
    """DEPTH ``__init__.py:185-291`` (mask-only composite; only the mask receives a gradient)."""

    @staticmethod
    def forward(ctx, means3D, means2D, opacities, mask, scales, rotations, cov3Ds_precomp, raster_settings):
        out = _forward_impl(raster_settings, _lib.FLAG_MASK_ONLY, 3, means3D, None, None, opacities, mask, scales,
                            rotations, cov3Ds_precomp)
        num_rendered, _, out_mask, _, radii, geom, binning, img, num_ch = out
        ctx.raster_settings = raster_settings
        ctx.sagars_flags = getattr(_TLS, "last_flags", None)
        ctx.num_rendered = num_rendered
        ctx.num_ch = num_ch
        ctx.mask_shape = tuple(mask.shape)
        ctx.save_for_backward(means3D, means2D, scales, rotations, cov3Ds_precomp, radii, geom, binning, img)
        ctx.mark_non_differentiable(radii)
        return out_mask, radii

    @staticmethod
    def backward(ctx, grad_out_mask, _):
        rs = ctx.raster_settings
        means3D, means2D, scales, rotations, cov3Ds_precomp, radii, geom, binning, img = ctx.saved_tensors
        g = _backward_impl(rs, _lib.FLAG_MASK_ONLY, ctx.num_ch, ctx.num_rendered, means3D, radii, None, None, scales,
                           rotations, cov3Ds_precomp, None, geom, binning, img, None, grad_out_mask, flags=ctx.sagars_flags)
        grad_mask = g["mask"].reshape(ctx.mask_shape)
        z = lambda t: torch.zeros_like(t, dtype=torch.float32, device=grad_mask.device)
        return (z(means3D), z(means2D), z(grad_mask), grad_mask, z(scales), z(rotations), z(cov3Ds_precomp), None)


_RasterizeBase = _make_rasterize_function(3)
_RasterizeContrastiveF = _make_rasterize_function(32)


# ----------------------------------------------------------------------------------------------
# nn.Module front ends
# ----------------------------------------------------------------------------------------------
def _validate(shs, colors_precomp, scales, rotations, cov3D_precomp, need_color=True):
    # the reference raises a plain Exception with these texts (CF __init__.py:190-194)
    if need_color and ((shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None)):
        raise Exception('Please provide excatly one of either SHs or precomputed colors!')
    if ((scales is None or rotations is None) and cov3D_precomp is None) or \
            ((scales is not None or rotations is not None) and cov3D_precomp is not None):
        raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')


def _empty_if_none(t):
    return torch.Tensor([]) if t is None else t


class _RasterizerBase(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        """Boolean mask of points in front of the near plane (CF ``__init__.py:175-184``)."""
        with torch.no_grad():
            rs = self.raster_settings
            _check_means(positions)
            device = positions.device
            P = int(positions.shape[0])
            present = torch.zeros((P,), dtype=torch.bool, device=device)
            if P > 0:
                pos = _f32(positions, device)
                view = _f32(rs.viewmatrix, device)
                proj = _f32(rs.projmatrix, device)
                with torch.cuda.device(device):
                    dev = device.index if device.index is not None else torch.cuda.current_device()
                    _lib.check(_lib.load().sagars_mark_visible(dev, P, pos.data_ptr(), view.data_ptr(), proj.data_ptr(),
                                                               present.data_ptr(), _stream_ptr(device)))
        return present


def _make_rasterizer(fn):
    class GaussianRasterizer(_RasterizerBase):
        """CF ``__init__.py:170-219``."""

        def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                    cov3D_precomp=None):
            _validate(shs, colors_precomp, scales, rotations, cov3D_precomp)
            return fn.apply(means3D, means2D, _empty_if_none(shs), _empty_if_none(colors_precomp), opacities,
                            _empty_if_none(scales), _empty_if_none(rotations), _empty_if_none(cov3D_precomp),
                            self.raster_settings)

    return GaussianRasterizer


GaussianRasterizer = _make_rasterizer(_RasterizeBase)
GaussianRasterizerContrastiveF = _make_rasterizer(_RasterizeContrastiveF)


class GaussianRasterizerDepth(_RasterizerBase):
    """DEPTH ``__init__.py:306-391``."""

    def forward(self, means3D, means2D, opacities, mask, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        _validate(shs, colors_precomp, scales, rotations, cov3D_precomp)
        return _RasterizeGaussiansDepth.apply(means3D, means2D, _empty_if_none(shs), _empty_if_none(colors_precomp),
                                              opacities, mask, _empty_if_none(scales), _empty_if_none(rotations),
                                              _empty_if_none(cov3D_precomp), self.raster_settings)

    def forward_mask(self, means3D, means2D, opacities, mask, scales=None, rotations=None, cov3D_precomp=None):
        _validate(None, None, scales, rotations, cov3D_precomp, need_color=False)
        return _RasterizeMaskGaussians.apply(means3D, means2D, opacities, mask, _empty_if_none(scales),
                                             _empty_if_none(rotations), _empty_if_none(cov3D_precomp),
                                             self.raster_settings)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings, variant: str = "base"):
    fn = {"base": _RasterizeBase, "cf": _RasterizeContrastiveF}[variant]
    return fn.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings)
