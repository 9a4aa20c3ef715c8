"""ctypes binding of libunetdc_b200.so -- one-to-one with include/unetdc_b200.h.

There is no fallback: if the shared library is missing (and cannot be built) or the device is not
an sm_100 GPU, every call raises.
"""
from __future__ import annotations

import ctypes as C
from ctypes import POINTER, Structure, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_void_p

from . import build as _build

DC_OK = 0
DC_EINVAL, DC_ECUDA, DC_EDEVICE, DC_ECAPACITY, DC_EWORKSPACE = -1, -2, -3, -4, -5
DC_KIND_CONV3X3, DC_KIND_UPCONV2 = 0, 1
DC_EPI_STORE, DC_EPI_STORE_POOL, DC_EPI_HEAD, DC_EPI_UPSCATTER = 0, 1, 2, 3
DC_NUM_LAYERS = 23
DC_CONV_FAMILY_AUTO, DC_CONV_FAMILY_GENERIC = 0, 2
DC_PRECISION_BF16, DC_PRECISION_FP32 = 0, 1
ABI_VERSION = 211          # DC_ABI_VERSION of include/unetdc_b200.h these ctypes structures mirror

EXPORTS = [
    "dc_last_error", "dc_version", "dc_device_check", "dc_conv_tc", "dc_conv_upfused", "dc_debug_upfuse_schedule", "dc_debug_set_conv_family", "dc_stem", "dc_model_create",
    "dc_model_destroy", "dc_forward_workspace_bytes", "dc_forward", "dc_forward_num_launches", "dc_forward_profile",
    "dc_rolling_ball_workspace_bytes", "dc_rolling_ball", "dc_rolling_ball_tiled", "dc_rolling_ball_banded", "dc_rolling_ball_max_radius",
    "dc_rolling_ball_tiled_max_radius", "dc_debug_rolling_ball_plan", "dc_debug_rolling_ball_bands", "dc_label_workspace_bytes", "dc_label_stats",
    "dc_resize_linear_u8", "dc_overlay_workspace_bytes", "dc_overlay_stencil",
    "dc_roi_workspace_bytes", "dc_roi_mask", "dc_radial_workspace_bytes", "dc_radial_density",
    "dc_spatial_workspace_bytes", "dc_spatial_density",
    "dc_table_csv_bounds", "dc_table_csv", "dc_debug_format_values", "dc_debug_table_csv_host",
    "dc_png_bounds", "dc_png_encode", "dc_debug_png_host",
]


class DcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libunetdc_b200: {msg} (code {code})")
        self.code = code


class ConvArgs(Structure):
    _fields_ = [
        ("kind", c_int), ("epilogue", c_int), ("relu", c_int),
        ("B", c_int), ("H", c_int), ("W", c_int),
        ("Cin", c_int), ("Cout", c_int), ("dilation", c_int),
        ("in_", c_void_p), ("in_stride", c_int),
        ("weight", c_void_p), ("bias", c_void_p),
        ("out", c_void_p), ("out_stride", c_int), ("out_offset", c_int),
        ("pool_out", c_void_p), ("pool_stride", c_int),
        ("head_w", c_void_p), ("head_b", c_float), ("thresh", c_float),
        ("prob_out", c_void_p), ("mask_out", c_void_p),
        ("weight_par", c_void_p),
        ("planes", c_int), ("in_plane_stride", c_int), ("out_plane_stride", c_int), ("pool_plane_stride", c_int),
    ]


class StemArgs(Structure):
    _fields_ = [
        ("in_kind", c_int), ("B", c_int), ("H", c_int), ("W", c_int), ("Cout", c_int), ("dilation", c_int),
        ("in_", c_void_p), ("weight", c_void_p), ("bias", c_void_p), ("out", c_void_p),
        ("out_stride", c_int), ("out_offset", c_int),
    ]


class ModelDesc(Structure):
    _fields_ = [
        ("weight", c_void_p * DC_NUM_LAYERS), ("bias", c_void_p * DC_NUM_LAYERS),
        ("dilations", c_int * 5), ("base_channels", c_int), ("in_channels", c_int), ("out_channels", c_int),
        ("fused_weight1", c_void_p), ("fused_bias1", c_void_p),
        ("fused_wide_x", c_void_p * 3), ("fused_wide_s", c_void_p * 3), ("fused_wide_b", c_void_p * 3),
        ("par_weight", c_void_p * 2),
        ("precision", c_int),
    ]


class UpfuseArgs(Structure):
    _fields_ = [
        ("B", c_int), ("H", c_int), ("W", c_int),
        ("x", c_void_p), ("x_stride", c_int),
        ("skip", c_void_p), ("skip_stride", c_int),
        ("weight", c_void_p), ("bias9", c_void_p), ("relu", c_int),
        ("out", c_void_p), ("out_stride", c_int), ("out_offset", c_int),
        ("channels", c_int), ("weight_skip", c_void_p),
    ]


class RollingBallArgs(Structure):
    _fields_ = [
        ("in_", c_void_p), ("out", c_void_p),
        ("B", c_int), ("H", c_int), ("W", c_int), ("C", c_int), ("radius", c_int),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class ResizeArgs(Structure):
    _fields_ = [
        ("in_", c_void_p), ("out", c_void_p), ("B", c_int), ("C", c_int),
        ("src_h", c_int), ("src_w", c_int), ("dst_h", c_int), ("dst_w", c_int),
    ]


class LabelArgs(Structure):
    _fields_ = [
        ("mask", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int),
        ("min_area", c_int64), ("px_per_um", c_double),
        ("labels_out", c_void_p), ("capacity", c_int), ("counts", c_void_p),
        ("area", c_void_p), ("centroid0", c_void_p), ("centroid1", c_void_p), ("eq_diam", c_void_p),
        ("area_um2", c_void_p), ("diam_um", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class TableCsvArgs(Structure):
    _fields_ = [
        ("B", c_int), ("capacity", c_int), ("counts", c_void_p), ("area", c_void_p),
        ("eq_diam", c_void_p), ("centroid0", c_void_p), ("centroid1", c_void_p),
        ("area_um2", c_void_p), ("diam_um", c_void_p),
        ("names", c_void_p), ("name_offsets", c_void_p), ("names_bytes", c_int64),
        ("out", c_void_p), ("out_bytes", c_int64), ("frame_offsets", c_void_p), ("area_sum", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class PngArgs(Structure):
    _fields_ = [
        ("images", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int), ("C", c_int),
        ("out", c_void_p), ("out_bytes", c_int64), ("offsets", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class OverlayArgs(Structure):
    _fields_ = [
        ("mask", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int), ("stencil", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class RoiArgs(Structure):
    _fields_ = [
        ("rgb", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int), ("roi", c_void_p), ("centroid", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class RadialArgs(Structure):
    _fields_ = [
        ("roi", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int), ("centroid", c_void_p), ("counts", c_void_p),
        ("centroid0", c_void_p), ("centroid1", c_void_p), ("capacity", c_int), ("nb_layers", c_int), ("out", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class SpatialArgs(Structure):
    _fields_ = [
        ("mask", c_void_p), ("roi", c_void_p), ("B", c_int), ("H", c_int), ("W", c_int), ("radius", c_int),
        ("weights", c_void_p), ("out", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


_LIB = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen the CUDA library (building it first when the in-tree copy is missing or stale)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB_PATH
    if build_if_missing and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:
            # a stale library may have been built against other struct layouts: loading it would corrupt memory
            what = "is out of date with its sources" if path.exists() else "is missing"
            raise RuntimeError(
                f"{path} {what} and could not be rebuilt ({exc}); unet_dc_segmentation_b200 has "
                "no CPU or PyTorch fallback") from exc
    if not path.exists():
        raise RuntimeError(f"{path} is missing; run `python -m unet_dc_segmentation_b200.build`")
    lib = C.CDLL(str(path))
    lib.dc_last_error.restype = C.c_char_p
    lib.dc_last_error.argtypes = []
    lib.dc_version.restype = c_int
    lib.dc_version.argtypes = []
    if lib.dc_version() != ABI_VERSION:
        raise RuntimeError(f"{path} reports ABI version {lib.dc_version()}, this binding is for {ABI_VERSION}: "
                           "rebuild with `python -m unet_dc_segmentation_b200.build --force`")
    lib.dc_device_check.argtypes = [c_int, POINTER(c_int)]
    lib.dc_conv_tc.argtypes = [POINTER(ConvArgs), c_void_p]
    lib.dc_conv_upfused.argtypes = [POINTER(UpfuseArgs), c_void_p]
    lib.dc_debug_upfuse_schedule.argtypes = [POINTER(c_int), c_int]
    lib.dc_debug_set_conv_family.argtypes = [c_int]
    lib.dc_stem.argtypes = [POINTER(StemArgs), c_void_p]
    lib.dc_model_create.argtypes = [POINTER(c_void_p), c_int, POINTER(ModelDesc)]
    lib.dc_model_destroy.argtypes = [c_void_p]
    lib.dc_forward_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_forward.argtypes = [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                               c_void_p, c_size_t, c_void_p]
    lib.dc_forward_num_launches.argtypes = [c_void_p]
    lib.dc_forward_profile.argtypes = [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_void_p, POINTER(c_float)]
    lib.dc_rolling_ball_workspace_bytes.argtypes = [c_int, c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_rolling_ball.argtypes = [POINTER(RollingBallArgs), c_void_p]
    lib.dc_rolling_ball_tiled.argtypes = [POINTER(RollingBallArgs), c_void_p]
    lib.dc_rolling_ball_banded.argtypes = [POINTER(RollingBallArgs), c_void_p]
    lib.dc_rolling_ball_max_radius.argtypes = []
    lib.dc_rolling_ball_tiled_max_radius.argtypes = []
    lib.dc_debug_rolling_ball_plan.argtypes = [c_int, c_int, POINTER(c_int), c_int]
    lib.dc_debug_rolling_ball_bands.argtypes = [c_int, POINTER(c_int), c_int]
    lib.dc_label_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_label_stats.argtypes = [POINTER(LabelArgs), c_void_p]
    lib.dc_table_csv_bounds.argtypes = [c_int, c_int, c_int, c_int64, POINTER(c_int64), POINTER(c_size_t)]
    lib.dc_table_csv.argtypes = [POINTER(TableCsvArgs), c_void_p]
    lib.dc_debug_format_values.argtypes = [c_void_p, c_int, c_int64, c_void_p, c_int64, c_void_p]
    lib.dc_debug_table_csv_host.argtypes = [POINTER(TableCsvArgs)]
    lib.dc_png_bounds.argtypes = [c_int, c_int, c_int, c_int, POINTER(c_int64), POINTER(c_size_t)]
    lib.dc_png_encode.argtypes = [POINTER(PngArgs), c_void_p]
    lib.dc_debug_png_host.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_int64, POINTER(c_int64), c_void_p,
                                      c_int64, POINTER(c_int64)]
    lib.dc_resize_linear_u8.argtypes = [POINTER(ResizeArgs), c_void_p]
    lib.dc_overlay_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_overlay_stencil.argtypes = [POINTER(OverlayArgs), c_void_p]
    lib.dc_roi_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_roi_mask.argtypes = [POINTER(RoiArgs), c_void_p]
    lib.dc_radial_workspace_bytes.argtypes = [c_int, POINTER(c_size_t)]
    lib.dc_radial_density.argtypes = [POINTER(RadialArgs), c_void_p]
    lib.dc_spatial_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    lib.dc_spatial_density.argtypes = [POINTER(SpatialArgs), c_void_p]
    for name in EXPORTS:
        if name not in ("dc_last_error",):
            getattr(lib, name).restype = c_int
    lib.dc_last_error.restype = C.c_char_p
    _LIB = lib
    return lib


def check(rc: int) -> None:
    if rc != DC_OK:
        msg = load().dc_last_error()
        raise DcError(rc, msg.decode("utf-8", "replace") if msg else "unknown error")


def stream_ptr(device=None) -> c_void_p:
    """torch's current CUDA stream as the `void* stream` the C ABI takes."""
    import torch
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name: str):
    """The product path is device-only: a CPU tensor is an error, never a fallback."""
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: unet_dc_segmentation_b200 computes on sm_100a GPUs "
                           "only and has no CPU path")
    return t
