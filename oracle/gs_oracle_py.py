"""ctypes binding of the CPU oracle (oracle/libgs_oracle.so).  TEST INFRASTRUCTURE ONLY.

May be imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs.  Never by the product package.  Pinning: see gs_oracle.h (the reference's own shader source compiled for the CPU, oracle/refhlsl/).
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "libgs_oracle.so"


class GsoAsset(C.Structure):
    _fields_ = [("splat_count", C.c_uint32), ("pos_format", C.c_uint32), ("scale_format", C.c_uint32), ("sh_format", C.c_uint32),
                ("color_format", C.c_uint32), ("pos", C.c_void_p), ("other", C.c_void_p), ("sh", C.c_void_p), ("color", C.c_void_p),
                ("chunks", C.c_void_p), ("pos_bytes", C.c_uint64), ("other_bytes", C.c_uint64), ("sh_bytes", C.c_uint64),
                ("color_bytes", C.c_uint64), ("chunk_bytes", C.c_uint64)]


class GsoCutout(C.Structure):
    _fields_ = [("mat", C.c_float * 16), ("type_and_flags", C.c_uint32)]


class GsoFrame(C.Structure):
    _fields_ = [("mat_object_to_world", C.c_float * 16), ("mat_world_to_object", C.c_float * 16), ("mat_view", C.c_float * 16),
                ("mat_proj_gpu", C.c_float * 16), ("screen_w", C.c_float), ("screen_h", C.c_float), ("cam_pos_world", C.c_float * 3),
                ("splat_scale", C.c_float), ("opacity_scale", C.c_float), ("sh_order", C.c_uint32), ("sh_only", C.c_uint32),
                ("cutout_count", C.c_uint32), ("reserved0", C.c_uint32), ("cutouts", C.c_void_p), ("deleted_bits", C.c_void_p),
                ("selected_bits", C.c_void_p), ("scene_depth", C.c_void_p), ("scene_depth_on_device", C.c_uint32), ("reserved1", C.c_uint32)]


class GsoSplat(C.Structure):
    _fields_ = [("pos", C.c_float * 3), ("rot", C.c_float * 4), ("scale", C.c_float * 3), ("opacity", C.c_float),
                ("col", C.c_float * 3), ("sh", C.c_float * 45)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not LIB.exists():
            subprocess.run(["make", "-C", str(HERE)], check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
        L = C.CDLL(str(LIB))
        L.gso_f32tof16.restype, L.gso_f32tof16.argtypes = C.c_uint32, [C.c_float]
        L.gso_f16tof32.restype, L.gso_f16tof32.argtypes = C.c_float, [C.c_uint32]
        L.gso_exp_neg.restype, L.gso_exp_neg.argtypes = C.c_float, [C.c_float]
        L.gso_float_to_sortable_uint.restype, L.gso_float_to_sortable_uint.argtypes = C.c_uint32, [C.c_float]
        L.gso_inv_square_centered01.restype, L.gso_inv_square_centered01.argtypes = C.c_float, [C.c_float]
        L.gso_splat_index_to_pixel_index.restype = C.c_uint32
        L.gso_splat_index_to_pixel_index.argtypes = [C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.gso_load_splat_pos.restype, L.gso_load_splat_pos.argtypes = None, [C.POINTER(GsoAsset), C.c_uint32, C.c_void_p]
        L.gso_load_splat_data.restype, L.gso_load_splat_data.argtypes = None, [C.POINTER(GsoAsset), C.c_uint32, C.POINTER(GsoSplat)]
        L.gso_set_indices.restype, L.gso_set_indices.argtypes = None, [C.c_void_p, C.c_uint32]
        L.gso_calc_distances.restype = None
        L.gso_calc_distances.argtypes = [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_void_p, C.c_void_p, C.c_int]
        L.gso_sort_pairs.restype, L.gso_sort_pairs.argtypes = None, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int]
        L.gso_calc_view.restype, L.gso_calc_view.argtypes = None, [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_void_p, C.c_int]
        L.gso_render.restype = None
        L.gso_render.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]
        L.gso_render_sel.restype = None
        L.gso_render_sel.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p]
        L.gso_render_ex.restype = None
        L.gso_render_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.gso_composite.restype, L.gso_composite.argtypes = None, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.gso_max_threads.restype, L.gso_max_threads.argtypes = C.c_int, []
        L.gso_export_data.restype, L.gso_export_data.argtypes = None, [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_void_p, C.c_int]
        L.gso_bc7_decode_block.restype, L.gso_bc7_decode_block.argtypes = None, [C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def max_threads() -> int:
    return int(lib().gso_max_threads())


def bc7_decode_blocks(blocks: np.ndarray) -> np.ndarray:
    """(n,16) uint8 BC7 blocks -> (n,16,4) uint8 RGBA pixels, raster order inside each block."""
    blocks = np.ascontiguousarray(blocks, np.uint8).reshape(-1, 16)
    out = np.zeros((blocks.shape[0], 16, 4), np.uint8)
    L = lib()
    for i in range(blocks.shape[0]):
        L.gso_bc7_decode_block(blocks[i].ctypes.data, out[i].ctypes.data)
    return out


def asset_struct(asset) -> GsoAsset:
    """asset: unitygaussiansplatting_b200.asset.GaussianSplatAsset (numpy blobs, borrowed)."""
    a = GsoAsset()
    a.splat_count = asset.splatCount
    a.pos_format, a.scale_format = int(asset.posFormat), int(asset.scaleFormat)
    a.sh_format, a.color_format = int(asset.shFormat), int(asset.colorFormat)
    a.pos, a.pos_bytes = asset.posData.ctypes.data, asset.posData.nbytes
    a.other, a.other_bytes = asset.otherData.ctypes.data, asset.otherData.nbytes
    a.sh, a.sh_bytes = asset.shData.ctypes.data, asset.shData.nbytes
    a.color, a.color_bytes = asset.colorData.ctypes.data, asset.colorData.nbytes
    if asset.chunkData is not None and asset.chunkData.nbytes:
        a.chunks, a.chunk_bytes = asset.chunkData.ctypes.data, asset.chunkData.nbytes
    else:
        a.chunks, a.chunk_bytes = None, 0
    return a


def frame_struct(fp) -> GsoFrame:
    """fp: the product's GsFrameParams (same field layout); copied byte for byte."""
    f = GsoFrame()
    assert C.sizeof(f) == C.sizeof(fp)
    C.memmove(C.byref(f), C.byref(fp), C.sizeof(f))
    return f


def load_splat(asset, idx: int) -> dict:
    a, s = asset_struct(asset), GsoSplat()
    lib().gso_load_splat_data(C.byref(a), idx, C.byref(s))
    return {"pos": np.array(s.pos[:], np.float32), "rot": np.array(s.rot[:], np.float32), "scale": np.array(s.scale[:], np.float32),
            "opacity": np.float32(s.opacity), "col": np.array(s.col[:], np.float32), "sh": np.array(s.sh[:], np.float32).reshape(15, 3)}


def calc_distances(asset, fp, order: np.ndarray, threads: int = 1) -> np.ndarray:
    a, f = asset_struct(asset), frame_struct(fp)
    order = np.ascontiguousarray(order, np.uint32)
    keys = np.empty(asset.splatCount, np.uint32)
    lib().gso_calc_distances(C.byref(a), C.byref(f), order.ctypes.data, keys.ctypes.data, threads)
    return keys


def sort_pairs(keys: np.ndarray, payload: np.ndarray, threads: int = 1):
    assert keys.dtype == np.uint32 and payload.dtype == np.uint32 and keys.flags.c_contiguous and payload.flags.c_contiguous
    lib().gso_sort_pairs(keys.ctypes.data, payload.ctypes.data, keys.size, threads)


def calc_view(asset, fp, threads: int = 1) -> np.ndarray:
    a, f = asset_struct(asset), frame_struct(fp)
    view = np.zeros((asset.splatCount, 10), np.uint32)
    lib().gso_calc_view(C.byref(a), C.byref(f), view.ctypes.data, threads)
    return view


def export_data(asset, fp=None, threads: int = 1) -> np.ndarray:
    """CSExportData: (n, 62) float32 raw .ply attribute records; `fp` only supplies the cutouts."""
    a = asset_struct(asset)
    out = np.zeros((asset.splatCount, 62), np.float32)
    f = frame_struct(fp) if fp is not None else None
    lib().gso_export_data(C.byref(a), C.byref(f) if f is not None else None, out.ctypes.data, threads)
    return out


def render(view: np.ndarray, order: np.ndarray, width: int, height: int, blend_mode: int = 0, threads: int = 1,
           selected_bits=None, scene_depth=None) -> np.ndarray:
    view = np.ascontiguousarray(view, np.uint32)
    order = np.ascontiguousarray(order, np.uint32)
    rt = np.zeros((height, width, 4), np.float32)
    if scene_depth is not None:
        depth = np.ascontiguousarray(scene_depth, np.float32)
        assert depth.shape == (height, width)
        bits = None if selected_bits is None else np.ascontiguousarray(selected_bits, np.uint32)
        lib().gso_render_ex(view.ctypes.data, order.ctypes.data, order.size, width, height, blend_mode, rt.ctypes.data, threads,
                            bits.ctypes.data if bits is not None else None, depth.ctypes.data)
    elif selected_bits is None:
        lib().gso_render(view.ctypes.data, order.ctypes.data, order.size, width, height, blend_mode, rt.ctypes.data, threads)
    else:
        bits = np.ascontiguousarray(selected_bits, np.uint32)
        assert bits.size >= (view.shape[0] + 31) // 32
        lib().gso_render_sel(view.ctypes.data, order.ctypes.data, order.size, width, height, blend_mode, rt.ctypes.data, threads, bits.ctypes.data)
    return rt


def composite(rt: np.ndarray, target: np.ndarray, target_fp16: bool = False) -> np.ndarray:
    rt = np.ascontiguousarray(rt, np.float32)
    out = np.ascontiguousarray(target, np.float32).copy()
    lib().gso_composite(rt.ctypes.data, out.ctypes.data, rt.shape[1], rt.shape[0], 1 if target_fp16 else 0)
    return out


def frame(asset, fp, prev_order=None, width=None, height=None, blend_mode: int = 0, threads: int = 1):
    """Whole path: distances -> stable sort -> view -> draw.  Returns dict of every intermediate."""
    n = asset.splatCount
    order = np.arange(n, dtype=np.uint32) if prev_order is None else np.ascontiguousarray(prev_order, np.uint32).copy()
    keys = calc_distances(asset, fp, order, threads)
    sort_pairs(keys, order, threads)
    view = calc_view(asset, fp, threads)
    W, H = int(width or fp.screen_w), int(height or fp.screen_h)
    sel = C.cast(fp.selected_bits, C.POINTER(C.c_uint32)) if getattr(fp, "selected_bits", None) else None
    bits = np.ctypeslib.as_array(sel, shape=((n + 31) // 32,)) if sel else None
    depth = None
    if getattr(fp, "scene_depth", None):
        assert not fp.scene_depth_on_device, "the oracle reads host memory"
        depth = np.ctypeslib.as_array(C.cast(fp.scene_depth, C.POINTER(C.c_float)), shape=(H, W))
    rt = render(view, order, W, H, blend_mode, threads, bits, depth)
    return {"keys": keys, "order": order, "view": view, "rt": rt}


# ---- oracle/_ref/libref_hlsl.so: the reference's OWN shader source compiled for the CPU (oracle/refhlsl/) ----------------
REF_HLSL_LIB = HERE / "_ref" / "libref_hlsl.so"
_ref_hlsl = None


def ref_hlsl():
    """Loads the compiled-reference library, built by oracle/refhlsl/build_ref_hlsl.py from a checkout of the reference.
    Only tests/golden/make_ref_hlsl_golden.py needs it; the tests read what it computed from tests/golden/ref_hlsl.npz."""
    global _ref_hlsl
    if _ref_hlsl is None:
        if not REF_HLSL_LIB.exists():
            raise FileNotFoundError("%s is missing: run oracle/refhlsl/build_ref_hlsl.py <reference checkout>" % REF_HLSL_LIB)
        L = C.CDLL(str(REF_HLSL_LIB))
        L.refhlsl_calc_distances.restype, L.refhlsl_calc_distances.argtypes = C.c_int, [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_void_p, C.c_void_p]
        L.refhlsl_calc_view.restype, L.refhlsl_calc_view.argtypes = C.c_int, [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_void_p]
        L.refhlsl_export.restype = C.c_int
        L.refhlsl_export.argtypes = [C.POINTER(GsoAsset), C.POINTER(GsoFrame), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.refhlsl_vert.restype, L.refhlsl_vert.argtypes = None, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
        L.refhlsl_frag.restype, L.refhlsl_frag.argtypes = C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.refhlsl_vert_sel.restype, L.refhlsl_vert_sel.argtypes = None, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        L.refhlsl_pack_rotation.restype, L.refhlsl_pack_rotation.argtypes = C.c_uint32, [C.c_void_p, C.c_void_p]
        L.refhlsl_decode_rotation.restype, L.refhlsl_decode_rotation.argtypes = None, [C.c_uint32, C.c_void_p]
        _ref_hlsl = L
    return _ref_hlsl


def ref_calc_distances(asset, fp, order: np.ndarray) -> np.ndarray:
    a, f = asset_struct(asset), frame_struct(fp)
    order = np.ascontiguousarray(order, np.uint32)
    keys = np.zeros(asset.splatCount, np.uint32)
    if ref_hlsl().refhlsl_calc_distances(C.byref(a), C.byref(f), order.ctypes.data, keys.ctypes.data) != 0:
        raise ValueError("compiled reference: unsupported asset format")
    return keys


def ref_calc_view(asset, fp) -> np.ndarray:
    a, f = asset_struct(asset), frame_struct(fp)
    view = np.zeros((asset.splatCount, 10), np.uint32)
    if ref_hlsl().refhlsl_calc_view(C.byref(a), C.byref(f), view.ctypes.data) != 0:
        raise ValueError("compiled reference: unsupported asset format")
    return view


def ref_export(asset, fp, bake=False, rotation=None, scale=None) -> np.ndarray:
    a, f = asset_struct(asset), frame_struct(fp)
    out = np.zeros((asset.splatCount, 62), np.float32)
    q = np.ascontiguousarray(rotation if rotation is not None else [0, 0, 0, 1], np.float32)
    s = np.ascontiguousarray(scale if scale is not None else [1, 1, 1], np.float32)
    if ref_hlsl().refhlsl_export(C.byref(a), C.byref(f), 1 if bake else 0, q.ctypes.data, s.ctypes.data, out.ctypes.data) != 0:
        raise ValueError("compiled reference: unsupported asset format")
    return out


def ref_vert(view: np.ndarray, order: np.ndarray, inst: int, width: float, height: float):
    """RenderGaussianSplats.shader vert for the four quad corners of draw instance `inst`: (clip[4,4], quadpos[4,2], colour[4])."""
    view = np.ascontiguousarray(view, np.uint32)
    order = np.ascontiguousarray(order, np.uint32)
    clip, pos, col = np.zeros((4, 4), np.float32), np.zeros((4, 2), np.float32), np.zeros(4, np.float32)
    ref_hlsl().refhlsl_vert(view.ctypes.data, order.ctypes.data, inst, width, height, clip.ctypes.data, pos.ctypes.data, col.ctypes.data)
    return clip, pos, col


def ref_vert_selected(view: np.ndarray, order: np.ndarray, inst: int, width: float, height: float, selected_bits: np.ndarray):
    """vert with _SplatSelectedBits bound: the colour (rgba) draw instance `inst` leaves the vertex shader with."""
    view = np.ascontiguousarray(view, np.uint32)
    order = np.ascontiguousarray(order, np.uint32)
    bits = np.ascontiguousarray(selected_bits, np.uint32)
    col = np.zeros(4, np.float32)
    ref_hlsl().refhlsl_vert_sel(view.ctypes.data, order.ctypes.data, inst, width, height, bits.ctypes.data, col.ctypes.data)
    return col


def ref_frag(col, pos_x: float, pos_y: float):
    """RenderGaussianSplats.shader frag on given interpolants: (rgba, discarded)."""
    col = np.ascontiguousarray(col, np.float32)
    out = np.zeros(4, np.float32)
    d = ref_hlsl().refhlsl_frag(col.ctypes.data, pos_x, pos_y, out.ctypes.data)
    return out, bool(d)
