"""ctypes binding of ``libsagars.so`` (the C ABI declared in ``include/sagars.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C seganygaussians_b200/csrc``
into ``seganygaussians_b200/lib/libsagars.so``.  There is NO fallback: if the shared library is
missing or does not export the ABI this module raises, and so does every operator built on it.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_DEFAULT_LIB_PATH = os.path.join(_HERE, "lib", "libsagars.so")
# SAGARS_LIBRARY: developer switch to load a differently built libsagars.so (a build variant under lib/variants/); never a fallback
LIB_PATH = os.environ.get("SAGARS_LIBRARY") or _DEFAULT_LIB_PATH

ABI_VERSION = 4

# flags (include/sagars.h)
FLAG_PREFILTERED = 1
FLAG_DEBUG = 2
FLAG_MASK_DEPTH = 4
FLAG_MASK_ONLY = 8
FLAG_CUB_SORT = 16
FLAG_NO_TENSOR_CORES = 32
FLAG_FWD_TILE = 64
FLAG_BWD_TILE = 128
FLAG_BWD_TC = 2048
FLAG_DEPTH_FIRST = 4096
FLAG_FWD_WARP_ANY = 256
FLAG_TILE_SORT = 1024

ERROR_NAMES = {0: "OK", 1: "EINVAL", 2: "ECUDA", 3: "ENOCOLOR", 4: "EALLOC", 5: "EPREFILTER"}

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)

_fp = C.c_void_p  # device pointers travel as plain integers


class ForwardArgs(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("flags", C.c_uint32),
        ("P", C.c_int32), ("D", C.c_int32), ("M", C.c_int32), ("num_channels", C.c_int32),
        ("width", C.c_int32), ("height", C.c_int32),
        ("tan_fovx", C.c_float), ("tan_fovy", C.c_float), ("scale_modifier", C.c_float),
        ("background", _fp), ("means3D", _fp), ("shs", _fp), ("colors_precomp", _fp), ("opacities", _fp),
        ("mask", _fp), ("scales", _fp), ("rotations", _fp), ("cov3D_precomp", _fp),
        ("viewmatrix", _fp), ("projmatrix", _fp), ("cam_pos", _fp),
        ("out_color", _fp), ("out_mask", _fp), ("out_depth", _fp), ("radii", _fp),
        ("binning_capacity_hint", C.c_int32), ("binning_capacity_out", C.POINTER(C.c_int32)),
        ("blend_wait_event", C.c_void_p),
    ]


class BackwardArgs(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("flags", C.c_uint32),
        ("P", C.c_int32), ("D", C.c_int32), ("M", C.c_int32), ("R", C.c_int32),
        ("num_channels", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
        ("tan_fovx", C.c_float), ("tan_fovy", C.c_float), ("scale_modifier", C.c_float),
        ("background", _fp), ("means3D", _fp), ("shs", _fp), ("colors_precomp", _fp), ("mask", _fp),
        ("scales", _fp), ("rotations", _fp), ("cov3D_precomp", _fp),
        ("viewmatrix", _fp), ("projmatrix", _fp), ("cam_pos", _fp),
        ("radii", _fp), ("geom_buffer", _fp), ("binning_buffer", _fp), ("image_buffer", _fp),
        ("dL_dout_color", _fp), ("dL_dout_mask", _fp), ("grad_scratch", _fp),
        ("dL_dmeans2D", _fp), ("dL_dopacity", _fp), ("dL_dcolors", _fp), ("dL_dmask", _fp),
        ("dL_dmeans3D", _fp), ("dL_dcov3D", _fp), ("dL_dsh", _fp), ("dL_dscales", _fp), ("dL_drotations", _fp),
    ]


class GeomLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in
                ("depths", "geo", "cov3D", "rgb", "clamped", "tiles_touched", "point_offsets", "status", "total")]


class ImageLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("final_T", "n_contrib", "ranges", "total")]


class BinningLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("point_list", "point_list_keys", "total")]


# every symbol include/sagars.h declares (tests check the .so exports exactly these)
ABI_SYMBOLS = (
    "sagars_forward", "sagars_backward", "sagars_mark_visible",
    "sagars_geom_bytes", "sagars_image_bytes", "sagars_binning_bytes", "sagars_grad_scratch_bytes",
    "sagars_get_geom_layout", "sagars_get_image_layout", "sagars_get_binning_layout",
    "sagars_sort_temp_bytes", "sagars_sort_pairs", "sagars_knn_temp_bytes", "sagars_knn", "sagars_smooth_forward", "sagars_smooth_backward", "sagars_sample_rays_forward", "sagars_sample_rays_backward",
    "sagars_launch_count", "sagars_reset_launch_count",
    "sagars_profile_enable", "sagars_profile_num_stages", "sagars_profile_stage_name", "sagars_profile_read",
    "sagars_sizeof_forward_args", "sagars_sizeof_backward_args", "sagars_multimem_allreduce_f32",
    "sagars_last_error", "sagars_abi_version", "sagars_arch",
)

_lib = None
_lock = threading.Lock()


class SagarsLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libsagars.so once; raise loudly when it is absent or stale."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SagarsLibraryError(
                f"{LIB_PATH} not found: the sm_100a CUDA library has not been built. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` (or `make -C seganygaussians_b200/csrc`). "
                "There is no CPU / PyTorch fallback for the rasterizer.")
        lib = C.CDLL(LIB_PATH)
        missing = [s for s in ABI_SYMBOLS if not hasattr(lib, s)]
        if missing:
            raise SagarsLibraryError(f"{LIB_PATH} does not export {missing}")
        lib.sagars_abi_version.restype = C.c_int
        if lib.sagars_abi_version() != ABI_VERSION:
            raise SagarsLibraryError(f"ABI version mismatch: library {lib.sagars_abi_version()}, binding {ABI_VERSION}")
        lib.sagars_arch.restype = C.c_char_p
        for fn, st in (("sagars_sizeof_forward_args", ForwardArgs), ("sagars_sizeof_backward_args", BackwardArgs)):
            getattr(lib, fn).restype = C.c_size_t
            if getattr(lib, fn)() != C.sizeof(st):
                raise SagarsLibraryError(f"{fn}() = {getattr(lib, fn)()} but the binding's struct has {C.sizeof(st)} bytes")
        lib.sagars_last_error.restype = C.c_char_p
        lib.sagars_launch_count.restype = C.c_int64
        lib.sagars_reset_launch_count.restype = None
        lib.sagars_profile_enable.restype = None
        lib.sagars_profile_enable.argtypes = [C.c_int]
        lib.sagars_profile_stage_name.restype = C.c_char_p
        lib.sagars_profile_stage_name.argtypes = [C.c_int]
        lib.sagars_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int]
        for fn in ("sagars_geom_bytes", "sagars_binning_bytes", "sagars_grad_scratch_bytes", "sagars_sort_temp_bytes"):
            getattr(lib, fn).restype = C.c_size_t
            getattr(lib, fn).argtypes = [C.c_int32]
        lib.sagars_knn_temp_bytes.restype = C.c_size_t
        lib.sagars_knn_temp_bytes.argtypes = [C.c_int32]
        lib.sagars_knn.restype = C.c_int
        lib.sagars_knn.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.sagars_smooth_forward.restype = C.c_int
        lib.sagars_smooth_forward.argtypes = [C.c_int32] * 4 + [C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 3
        lib.sagars_sample_rays_forward.restype = C.c_int
        lib.sagars_sample_rays_forward.argtypes = [C.c_int32] * 6 + [C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 3
        lib.sagars_sample_rays_backward.restype = C.c_int
        lib.sagars_sample_rays_backward.argtypes = [C.c_int32] * 6 + [C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 4
        lib.sagars_smooth_backward.restype = C.c_int
        lib.sagars_smooth_backward.argtypes = [C.c_int32] * 4 + [C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 6
        lib.sagars_image_bytes.restype = C.c_size_t
        lib.sagars_image_bytes.argtypes = [C.c_int32, C.c_int32]
        lib.sagars_get_geom_layout.argtypes = [C.c_int32, C.POINTER(GeomLayout)]
        lib.sagars_get_image_layout.argtypes = [C.c_int32, C.c_int32, C.POINTER(ImageLayout)]
        lib.sagars_get_binning_layout.argtypes = [C.c_int32, C.POINTER(BinningLayout)]
        lib.sagars_multimem_allreduce_f32.restype = C.c_int
        lib.sagars_multimem_allreduce_f32.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
        lib.sagars_forward.restype = C.c_int
        lib.sagars_forward.argtypes = [C.POINTER(ForwardArgs), ALLOC_FN, C.c_void_p, ALLOC_FN, C.c_void_p,
                                       ALLOC_FN, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]
        lib.sagars_backward.restype = C.c_int
        lib.sagars_backward.argtypes = [C.POINTER(BackwardArgs), C.c_void_p]
        lib.sagars_mark_visible.restype = C.c_int
        lib.sagars_mark_visible.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.sagars_sort_pairs.restype = C.c_int
        lib.sagars_sort_pairs.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        _lib = lib
    return _lib


def last_error() -> str:
    return load().sagars_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Turn a status code into the exception the reference would have thrown (RuntimeError)."""
    if rc != 0:
        raise RuntimeError(last_error() or f"libsagars error {ERROR_NAMES.get(rc, rc)}")


def geom_layout(P: int) -> GeomLayout:
    out = GeomLayout()
    check(load().sagars_get_geom_layout(P, C.byref(out)))
    return out


def image_layout(W: int, H: int) -> ImageLayout:
    out = ImageLayout()
    check(load().sagars_get_image_layout(W, H, C.byref(out)))
    return out


def binning_layout(R: int) -> BinningLayout:
    out = BinningLayout()
    check(load().sagars_get_binning_layout(R, C.byref(out)))
    return out


def profile_enable(on: bool) -> None:
    load().sagars_profile_enable(1 if on else 0)


def profile_read(reset: bool = True) -> dict:
    """{stage name: (milliseconds, launches)} accumulated since the last reset."""
    lib = load()
    n = lib.sagars_profile_num_stages()
    ms = (C.c_double * n)()
    cnt = (C.c_int64 * n)()
    check(lib.sagars_profile_read(ms, cnt, 1 if reset else 0))
    return {lib.sagars_profile_stage_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n)}


def launch_count() -> int:
    return int(load().sagars_launch_count())


def reset_launch_count() -> None:
    load().sagars_reset_launch_count()
