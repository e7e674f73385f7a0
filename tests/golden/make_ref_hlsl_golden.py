#!/usr/bin/env python
"""Regenerates tests/golden/ref_hlsl.npz: what the reference's own shader code computes on the inputs of
tests/test_reference_hlsl.py and tests/test_zz_reference_hlsl_gpu.py.

The shader code runs on the CPU as oracle/_ref/libref_hlsl.so, which oracle/refhlsl/build_ref_hlsl.py builds from a
checkout of the reference.  The tests compare the oracle and the CUDA path with the stored arrays, so they need neither
that checkout nor the library.  Per-splat results are stored for a fixed, seeded sample of the splats (all of them would
be megabytes); which splats the reference culls is stored for every splat.  The inputs are built by the functions below,
which the tests call too.
Run from the repo root:  python tests/golden/make_ref_hlsl_golden.py <checkout of aras-p/UnityGaussianSplatting>
"""
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

OUT = Path(__file__).with_name("ref_hlsl.npz")
VIEW_QUALITIES = ["Medium", "VeryHigh", "High", "Low", "custom-f16sh", "custom-norm6pos"]
KEY_QUALITIES = ["Medium", "VeryHigh"]
GPU_QUALITIES = ["Medium", "VeryHigh"]
VIEW_SAMPLE, KEY_SAMPLE, EXPORT_SAMPLE = 256, 1024, 128
DRAW_W, DRAW_H = 200, 150


def sample(n, k, salt):
    """The stored rows of an n-splat result: k distinct indices, ascending, the same on every run."""
    return np.sort(np.random.default_rng(0x5EED0094 + salt).choice(n, k, replace=False)).astype(np.int64)


def packbits(mask):
    return np.packbits(np.asarray(mask, bool))


def unpackbits(bits, n):
    return np.unpackbits(bits)[:n].astype(bool)


def view_case(g, quality):
    """test_view_data_matches_the_reference_shader_code: (asset, frame params, keep-alive)."""
    from util import camera
    n = 20000
    if quality.startswith("custom"):     # format combinations no preset uses: Float16 SH, Norm6 positions, Norm16 scale
        fmts = {"custom-f16sh": (g.VectorFormat.Norm16, g.VectorFormat.Norm6, g.ColorFormat.Float16x4, g.SHFormat.Float16),
                "custom-norm6pos": (g.VectorFormat.Norm6, g.VectorFormat.Norm16, g.ColorFormat.Float32x4, g.SHFormat.Norm11)}[quality]
        asset = g.create_asset(g.generate_input_splats(g.SCENE_CLUSTERED, n, 0x5EED0091), formats=fmts)
    else:
        asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0091, quality)
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = np.array([[0.8, -0.6, 0.0], [0.6, 0.8, 0.0], [0.0, 0.0, 1.0]], np.float32) * 1.1
    T[:3, 3] = (0.3, -0.1, 0.2)
    box = np.diag([1 / 9.0, 1 / 9.0, 1 / 9.0, 1.0]).astype(np.float32)
    deleted = np.zeros((n + 31) // 32, np.uint32)
    deleted[3] = 0xF0F0F0F0
    fp, keep = g.make_frame_params(camera(g, 320, 240), localToWorld=T, splat_scale=0.9, opacity_scale=1.3, sh_order=3,
                                   cutouts=[(box, 1)], deleted_bits=deleted, splat_count=n)
    return asset, fp, (keep, deleted)


def keys_case(g, quality):
    """test_sort_keys_match_the_reference_shader_code: (asset, frame params, keep-alive, order)."""
    from util import camera
    n = 30000
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0092, quality)
    fp, keep = g.make_frame_params(camera(g, 320, 240))
    order = np.random.default_rng(1).permutation(n).astype(np.uint32)
    return asset, fp, keep, order


def export_case(g):
    """test_export_and_baked_transform_match_the_reference_shader_code: asset, plain and transformed frame params, the
    transform and its rotation / scale, keep-alive."""
    from unitygaussiansplatting_b200.renderer import decompose_trs
    from util import camera
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 3000, 0x5EED0093, "VeryHigh")
    fp, keep = g.make_frame_params(camera(g, 64, 64))
    ang = np.radians(50.0)
    Rm = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]]) @ \
        np.array([[1, 0, 0], [0, np.cos(0.4), -np.sin(0.4)], [0, np.sin(0.4), np.cos(0.4)]])
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = (Rm * 1.25).astype(np.float32)
    T[:3, 3] = (0.5, 0.25, -0.75)
    q, s = decompose_trs(T)
    fpT, keepT = g.make_frame_params(camera(g, 64, 64), localToWorld=T)
    return asset, fp, fpT, T, q, s, (keep, keepT)


def draw_case(g, selected):
    """test_draw_stages_* (one opaque-ish splat) and test_selected_splat_* (the same splat at opacity 0.02 among 40
    far-away padding splats): (asset, frame params, keep-alive)."""
    from util import camera, one_splat
    cam = camera(g, DRAW_W, DRAW_H, fov=50.0, pos=(0.1, 0.0, -3.0))
    if selected:
        asset = one_splat(g, pos=(0.2, -0.1, 0.3), scale=(0.25, 0.08, 0.05), quat=(0.3, 0.5, -0.2, 0.78), opacity=0.02, dc0=(0.7, 0.5, 0.9), n_pad=40)
    else:
        asset = one_splat(g, pos=(0.2, -0.1, 0.3), scale=(0.25, 0.08, 0.05), quat=(0.3, 0.5, -0.2, 0.78), opacity=0.65, dc0=(0.7, 0.5, 0.9))
    fp, keep = g.make_frame_params(cam, sh_order=0)
    return asset, fp, keep


def quad_map(clip, qpos, width, height):
    """The rasteriser's linear interpolation of the quad coordinates: A with [x y 1] @ A = quad position at pixel (x, y)."""
    px = np.stack([(clip[:, 0] / clip[:, 3] * 0.5 + 0.5) * width, (0.5 - 0.5 * clip[:, 1] / clip[:, 3]) * height], 1).astype(np.float64)
    return np.linalg.solve(np.column_stack([px[:3], np.ones(3)]), qpos[:3].astype(np.float64)), px


def quad_pixels(A, width, height):
    """(x, y, qx, qy) of every pixel whose quad coordinates are within 2.3 of the centre, raster order."""
    for y in range(height):
        for x in range(width):
            qx, qy = np.array([x + 0.5, y + 0.5, 1.0]) @ A
            if abs(qx) <= 2.3 and abs(qy) <= 2.3:
                yield x, y, qx, qy


def rotation_quats():
    rng = np.random.default_rng(3)
    out = []
    for _ in range(300):
        q = rng.standard_normal(4).astype(np.float32)
        q /= np.linalg.norm(q)
        out.append(q)
    return out


def _frag_image(R, col, A):
    """What the reference's pixel shader gives at each pixel of the quad (0 where it discards or outside the quad)."""
    want = np.zeros((DRAW_H, DRAW_W, 4), np.float32)
    for x, y, qx, qy in quad_pixels(A, DRAW_W, DRAW_H):
        out, discarded = R.ref_frag(col, float(qx), float(qy))
        if not discarded and abs(qx) <= 2 and abs(qy) <= 2:
            want[y, x] = out
    return want


def build(R):
    import unitygaussiansplatting_b200 as g
    from unitygaussiansplatting_b200 import _native as N
    from util import camera
    d = {}
    for i, quality in enumerate(VIEW_QUALITIES):
        asset, fp, _keep = view_case(g, quality)
        v = R.ref_calc_view(asset, fp)
        w = v[:, 3].view(np.float32)
        idx = sample(asset.splatCount, VIEW_SAMPLE, i)
        d["view_%s_idx" % quality], d["view_%s_rows" % quality] = idx.astype(np.uint32), v[idx]
        d["view_%s_w_le0" % quality], d["view_%s_w_eq0" % quality] = packbits(w <= 0), packbits(w == 0)
    for i, quality in enumerate(KEY_QUALITIES):
        asset, fp, _keep, order = keys_case(g, quality)
        k = R.ref_calc_distances(asset, fp, order)
        idx = sample(asset.splatCount, KEY_SAMPLE, 10 + i)
        first = np.argsort(k, kind="stable")[:100]
        d["keys_%s_idx" % quality], d["keys_%s_keys" % quality] = idx.astype(np.uint32), k[idx]
        d["keys_%s_first100" % quality] = first.astype(np.uint32)
    asset, fp, fpT, T, q, s, _keep = export_case(g)
    idx = sample(asset.splatCount, EXPORT_SAMPLE, 20)
    d["export_idx"] = idx.astype(np.uint32)
    d["export_plain"] = R.ref_export(asset, fp)[idx]
    d["export_baked"] = R.ref_export(asset, fpT, bake=True, rotation=q, scale=s)[idx]
    for selected, name in ((False, "draw"), (True, "selected")):
        asset, fp, _keep = draw_case(g, selected)
        view = R.calc_view(asset, fp)       # the oracle's view data is what the reference's vertex shader is handed
        order = np.arange(asset.splatCount, dtype=np.uint32)
        clip, qpos, col = R.ref_vert(view, order, 0, DRAW_W, DRAW_H)
        d[name + "_view_in"], d[name + "_clip"], d[name + "_qpos"], d[name + "_col"] = view[:2], clip, qpos, col
        if selected:
            bits = np.zeros(2, np.uint32)
            bits[0] = 1
            col = R.ref_vert_selected(view, order, 0, DRAW_W, DRAW_H, bits)
            d["selected_col_sel"] = col
            d["selected_col_sel_1"] = R.ref_vert_selected(view, order, 1, DRAW_W, DRAW_H, bits)
        A, _px = quad_map(clip, qpos, DRAW_W, DRAW_H)
        d[name + "_frag"] = _frag_image(R, col, A)
    L = R.ref_hlsl()
    enc, packed, back = [], [], []
    for q in rotation_quats():
        ref = np.zeros(4, np.float32)
        enc.append(L.refhlsl_pack_rotation(q.ctypes.data, ref.ctypes.data))
        b = np.zeros(4, np.float32)
        L.refhlsl_decode_rotation(enc[-1], b.ctypes.data)
        packed.append(ref)
        back.append(b)
    d["rot_enc"], d["rot_packed"], d["rot_decoded"] = np.array(enc, np.uint32), np.array(packed), np.array(back)
    for i, quality in enumerate(GPU_QUALITIES):
        asset = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0091, quality)
        fp, _keep = g.make_frame_params(camera(g, 320, 240))
        v = R.ref_calc_view(asset, fp)
        k = R.ref_calc_distances(asset, fp, np.arange(asset.splatCount, dtype=np.uint32))    # key of each splat, by index
        idx = sample(asset.splatCount, VIEW_SAMPLE, 30 + i)
        kidx = sample(asset.splatCount, KEY_SAMPLE, 40 + i)
        d["gpu_%s_idx" % quality], d["gpu_%s_rows" % quality] = idx.astype(np.uint32), v[idx]
        d["gpu_%s_w_le0" % quality] = packbits(v[:, 3].view(np.float32) <= 0)
        d["gpu_%s_key_idx" % quality], d["gpu_%s_keys" % quality] = kidx.astype(np.uint32), k[kidx]
    return d


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    subprocess.run([sys.executable, str(ROOT / "oracle" / "refhlsl" / "build_ref_hlsl.py"), sys.argv[1]], check=True)
    from oracle import gs_oracle_py as O
    data = build(O)
    np.savez_compressed(OUT, **data)
    print(OUT, OUT.stat().st_size, "bytes")
