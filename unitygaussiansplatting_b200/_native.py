"""ctypes bindings of the two product libraries.

libgsplat_b200.so (include/gsplat_b200.h) is the CUDA hot path.  There is no fallback:
if the extension is missing or no CUDA device is present, loading / gs_create raise.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
NATIVE_LIB = PKG / "libgsplat_b200.so"
ASSET_LIB = PKG / "libgsplat_asset.so"

GS_OK = 0
GS_ERR_NO_DEVICE = -6
GS_PIX_RGBA16F, GS_PIX_RGBA32F = 0, 1
GS_MEM_HOST, GS_MEM_DEVICE = 0, 1
GS_BLEND_FP16_ROP, GS_BLEND_FP32 = 0, 1


class GsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("gsplat_b200 error %d: %s" % (code, msg))
        self.code = code


class GsAssetDesc(C.Structure):
    _fields_ = [
        ("splat_count", C.c_uint32),
        ("pos_format", C.c_uint32), ("scale_format", C.c_uint32), ("sh_format", C.c_uint32), ("color_format", C.c_uint32),
        ("pos", C.c_void_p), ("other", C.c_void_p), ("sh", C.c_void_p), ("color", C.c_void_p), ("chunks", C.c_void_p),
        ("pos_bytes", C.c_uint64), ("other_bytes", C.c_uint64), ("sh_bytes", C.c_uint64), ("color_bytes", C.c_uint64),
        ("chunk_bytes", C.c_uint64),
    ]


class GsCutout(C.Structure):
    _fields_ = [("mat", C.c_float * 16), ("type_and_flags", C.c_uint32)]


class GsFrameParams(C.Structure):
    _fields_ = [
        ("mat_object_to_world", C.c_float * 16), ("mat_world_to_object", C.c_float * 16),
        ("mat_view", C.c_float * 16), ("mat_proj_gpu", C.c_float * 16),
        ("screen_w", C.c_float), ("screen_h", C.c_float),
        ("cam_pos_world", C.c_float * 3),
        ("splat_scale", C.c_float), ("opacity_scale", C.c_float),
        ("sh_order", C.c_uint32), ("sh_only", C.c_uint32),
        ("cutout_count", C.c_uint32), ("reserved0", C.c_uint32),
        ("cutouts", C.c_void_p), ("deleted_bits", C.c_void_p), ("selected_bits", C.c_void_p),
        ("scene_depth", C.c_void_p), ("scene_depth_on_device", C.c_uint32), ("reserved1", C.c_uint32),
    ]


class GsImage(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("row_pitch_bytes", C.c_uint32),
                ("format", C.c_uint32), ("memory", C.c_uint32)]


class GsRenderOptions(C.Structure):
    _fields_ = [("blend_mode", C.c_uint32), ("band_packed", C.c_uint32), ("partition_index", C.c_uint32),
                ("partition_count", C.c_uint32), ("band_rows", C.c_uint32), ("flags", C.c_uint32),
                ("row_begin", C.c_uint32), ("row_end", C.c_uint32)]


GS_FLAG_ASYNC_READBACK = 1
GS_FLAG_LOAD_RT = 2
GS_GROUP_EMULATE = 1
GS_GROUP_ID_BYTES = 128
GS_GROUP_MAX_GPUS = 16
GS_TILE_PIXELS = 16


class GsGroupStats(C.Structure):
    _fields_ = [("distances_ms", C.c_float), ("slab_sort_ms", C.c_float), ("order_exchange_ms", C.c_float), ("view_ms", C.c_float),
                ("bin_ms", C.c_float), ("raster_ms", C.c_float), ("image_exchange_ms", C.c_float), ("total_ms", C.c_float),
                ("group_size", C.c_uint32), ("rank", C.c_uint32), ("row_bounds", C.c_uint32 * (GS_GROUP_MAX_GPUS + 1)),
                ("slab_counts", C.c_uint32 * GS_GROUP_MAX_GPUS)]


class GsUnityFrameEvent(C.Structure):   # include/gsplat_b200.h: the payload of CommandBuffer.IssuePluginEventAndData
    _fields_ = [("ctx", C.c_void_p), ("asset", C.c_void_p), ("params", GsFrameParams), ("options", GsRenderOptions),
                ("do_sort", C.c_int32), ("status", C.c_int32), ("has_rt", C.c_uint32), ("has_camera_target", C.c_uint32),
                ("rt", GsImage), ("camera_target", GsImage)]


GS_UNITY_EVENT_FRAME, GS_UNITY_EVENT_SYNC = 1, 2
GsUnityRenderEventAndDataFunc = C.CFUNCTYPE(None, C.c_int, C.c_void_p)


class GsStageTimes(C.Structure):
    _fields_ = [("distances_ms", C.c_float), ("sort_ms", C.c_float), ("view_ms", C.c_float), ("bin_ms", C.c_float),
                ("raster_ms", C.c_float), ("composite_ms", C.c_float), ("total_ms", C.c_float),
                ("sort_pass_ms", C.c_float * 4), ("tile_entries", C.c_uint64), ("kernel_launches", C.c_uint32),
                ("reserved", C.c_uint32)]


class GsaSizes(C.Structure):
    _fields_ = [("pos_bytes", C.c_uint64), ("other_bytes", C.c_uint64), ("color_bytes", C.c_uint64), ("sh_bytes", C.c_uint64),
                ("chunk_bytes", C.c_uint64), ("tex_width", C.c_uint32), ("tex_height", C.c_uint32)]


# every symbol include/gsplat_b200.h declares: name -> (restype, argtypes)
NATIVE_SYMBOLS = {
    "gs_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "gs_destroy": (None, [C.c_void_p]),
    "gs_last_error": (C.c_char_p, [C.c_void_p]),
    "gs_sync": (C.c_int, [C.c_void_p]),
    "gs_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "gs_get_stage_times": (C.c_int, [C.c_void_p, C.POINTER(GsStageTimes)]),
    "gs_version": (C.c_char_p, []),
    "gs_asset_upload": (C.c_int, [C.c_void_p, C.POINTER(GsAssetDesc), C.POINTER(C.c_void_p)]),
    "gs_asset_destroy": (None, [C.c_void_p]),
    "gs_asset_reset_order": (C.c_int, [C.c_void_p]),
    "gs_asset_splat_count": (C.c_uint32, [C.c_void_p]),
    "gs_sort": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GsFrameParams)]),
    "gs_calc_view": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GsFrameParams)]),
    "gs_render": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GsFrameParams), C.POINTER(GsRenderOptions), C.POINTER(GsImage)]),
    "gs_composite": (C.c_int, [C.c_void_p, C.POINTER(GsImage), C.POINTER(GsImage)]),
    "gs_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GsFrameParams), C.POINTER(GsRenderOptions), C.c_int,
                           C.POINTER(GsImage), C.POINTER(GsImage)]),
    "gs_unshuffle_bands": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(GsImage)]),
    "gs_group_unique_id": (C.c_int, [C.c_void_p]),
    "gs_group_join": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "gs_group_create": (C.c_int, [C.POINTER(C.c_int), C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "gs_group_destroy": (None, [C.c_void_p]),
    "gs_group_size": (C.c_uint32, [C.c_void_p]),
    "gs_group_local_count": (C.c_uint32, [C.c_void_p]),
    "gs_group_context": (C.c_void_p, [C.c_void_p, C.c_uint32]),
    "gs_group_asset_upload": (C.c_int, [C.c_void_p, C.POINTER(GsAssetDesc), C.POINTER(C.c_void_p)]),
    "gs_group_frame": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(GsFrameParams), C.POINTER(GsRenderOptions), C.c_int,
                                 C.POINTER(C.POINTER(GsImage))]),
    "gs_group_sync": (C.c_int, [C.c_void_p]),
    "gs_group_get_stats": (C.c_int, [C.c_void_p, C.POINTER(GsGroupStats)]),
    "gs_group_balance_rows": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "gs_sort_pairs_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "gs_sort_pairs_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "gs_readback_order": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gs_readback_keys": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gs_readback_view": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gs_upload_order": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gs_unity_get_render_event_func": (GsUnityRenderEventAndDataFunc, []),
    "gs_unity_frame_event_size": (C.c_uint32, []),
    "gs_export_splats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "gs_context_stream": (C.c_void_p, [C.c_void_p]),
    "gs_asset_device_ptr": (C.c_void_p, [C.c_void_p, C.c_int]),
}

ASSET_SYMBOLS = {
    "gsa_generate": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "gsa_calc_sizes": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(GsaSizes)]),
    "gsa_create_asset": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsa_ply_vertex_count": (C.c_int64, [C.c_char_p]),
    "gsa_ply_read": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint32]),
    "gsa_spz_vertex_count": (C.c_int64, [C.c_char_p]),
    "gsa_spz_read": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint32]),
    "gsa_morton_encode3": (C.c_uint64, [C.c_uint32, C.c_uint32, C.c_uint32]),
    "gsa_splat_index_to_texture_index": (C.c_uint32, [C.c_uint32]),
    "gsa_pack_smallest3": (None, [C.c_void_p, C.c_void_p]),
    "gsa_f32tof16": (C.c_uint32, [C.c_float]),
    "gsa_kmeans": (C.c_int, [C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_void_p, C.c_uint32, C.c_void_p]),
    "gsa_bc7_encode_block": (None, [C.c_void_p, C.c_void_p]),
    "gsa_bake_transform": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsa_ply_write": (C.c_int64, [C.c_char_p, C.c_void_p, C.c_uint32, C.c_void_p]),
}


def _bind(lib, table):
    for name, (res, args) in table.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    return lib


_native = None
_asset = None


def native():
    """The CUDA library.  Raises if it has not been built: the product has no CPU path."""
    global _native
    if _native is None:
        if not NATIVE_LIB.exists():
            raise GsError(-100, "CUDA extension %s is missing; run `python -c 'import __graft_entry__ as g; g.build()'`" % NATIVE_LIB)
        _native = _bind(C.CDLL(str(NATIVE_LIB)), NATIVE_SYMBOLS)
    return _native


def asset_lib():
    global _asset
    if _asset is None:
        if not ASSET_LIB.exists():
            raise GsError(-100, "asset packer %s is missing; run the build first" % ASSET_LIB)
        _asset = _bind(C.CDLL(str(ASSET_LIB)), ASSET_SYMBOLS)
    return _asset


def check(ctx, rc: int):
    if rc != GS_OK:
        msg = native().gs_last_error(ctx)
        raise GsError(rc, msg.decode("utf-8", "replace") if msg else "")
