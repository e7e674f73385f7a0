"""The oracle against THE REFERENCE'S OWN SHADER CODE.

The reference is package/Shaders/{GaussianSplatting.hlsl, SplatUtilities.compute, SphericalHarmonics.hlsl,
RenderGaussianSplats.shader} themselves, syntactically rewritten to C++ spelling and compiled with g++ against a shim of
HLSL's types and intrinsics (oracle/refhlsl/).  Expressions, constants, operation order and branches are the reference's;
scalar arithmetic is IEEE float32 without contraction.  What that code computed on the inputs below is stored in
tests/golden/ref_hlsl.npz (generator: tests/golden/make_ref_hlsl_golden.py, which builds the inputs these tests build):
per-splat results for a fixed sample of the splats, cull decisions for all of them.  The oracle (and the CUDA path,
bit-identical to it) evaluates the same formulas under its own arithmetic contract (explicit fmaf chains, reciprocal
constants), so the two agree to float rounding, not to the bit: tolerances below are a few ulp, scaled by conditioning
where a formula cancels."""
import sys
from pathlib import Path

import numpy as np
import pytest

from util import view_fields

GOLD = Path(__file__).parent / "golden"
sys.path.insert(0, str(GOLD))
import make_ref_hlsl_golden as RG  # noqa: E402


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD / "ref_hlsl.npz")


def _unsortable(keys):
    k = keys.astype(np.uint32)
    u = np.where(k & 0x80000000, k ^ np.uint32(0x80000000), ~k).astype(np.uint32)
    return u.view(np.float32)


def _cov(v):
    a1, a2 = v["axis1"].astype(np.float64), v["axis2"].astype(np.float64)
    return 0.5 * (a1[:, :, None] * a1[:, None, :] + a2[:, :, None] * a2[:, None, :])


@pytest.mark.parametrize("quality", RG.VIEW_QUALITIES)
def test_view_data_matches_the_reference_shader_code(g, O, gold, quality):
    asset, fp, _keep = RG.view_case(g, quality)
    view = O.calc_view(asset, fp)
    n, idx = asset.splatCount, gold["view_%s_idx" % quality].astype(np.int64)
    w = view[:, 3].view(np.float32)
    # which splats are culled (w = 0: deleted / cut) or behind the camera is decided identically, for every splat
    assert np.array_equal(RG.unpackbits(gold["view_%s_w_le0" % quality], n), w <= 0)
    assert (RG.unpackbits(gold["view_%s_w_eq0" % quality], n) & (w == 0)).sum() > 100
    ref, ora = view_fields(gold["view_%s_rows" % quality]), view_fields(view[idx])
    assert np.array_equal(ref["pos"][:, 3] <= 0, ora["pos"][:, 3] <= 0)
    assert (np.abs(ref["pos"] - ora["pos"]).max(1) <= 2e-6 * (1 + np.abs(ora["pos"]).max(1))).all()
    vis = ora["pos"][:, 3] > 0
    for ch in "rgb":                                         # half-precision results: at most one unit in the last place apart
        d = np.abs(ref[ch][vis] - ora[ch][vis])
        assert (d <= np.maximum(np.abs(ora[ch][vis]), 2.0 ** -14) * 2.0 ** -9).all(), ch     # <= 2 half ulps
        assert (d == 0).mean() > 0.9
    assert np.array_equal(ref["a"][vis], ora["a"][vis])
    # the two screen axes, through the covariance they encode (eigenvectors of near-circular footprints are ill-defined)
    cr, co = _cov(ref)[vis], _cov(ora)[vis]
    rel = np.abs(cr - co).reshape(-1, 4).max(1) / (co[:, 0, 0] + co[:, 1, 1])
    assert np.percentile(rel, 50) < 1e-6 and np.percentile(rel, 99) < 2e-5 and rel.max() < 2e-3


@pytest.mark.parametrize("quality", RG.KEY_QUALITIES)
def test_sort_keys_match_the_reference_shader_code(g, O, gold, quality):
    asset, fp, _keep, order = RG.keys_case(g, quality)
    ko = O.calc_distances(asset, fp, order)
    kr, idx = gold["keys_%s_keys" % quality], gold["keys_%s_idx" % quality].astype(np.int64)
    zr, zo = _unsortable(kr), _unsortable(ko[idx])
    assert np.abs(zr - zo).max() <= 4e-6 and (kr == ko[idx]).mean() > 0.5     # view-space depth of +-36: a couple of ulp
    assert np.array_equal(gold["keys_%s_first100" % quality], np.argsort(ko, kind="stable")[:100]) or (kr == ko[idx]).mean() < 1.0


def test_export_and_baked_transform_match_the_reference_shader_code(g, O, gold):
    """CSExportData incl. the _ExportTransformFlags branch: QuatMul, scale, and RotateSH (the closed form after sh-lib,
    S/SphericalHarmonics.hlsl) against the oracle's export and the product's gsa_bake_transform (least-squares band matrices)."""
    from unitygaussiansplatting_b200.renderer import bake_transform
    asset, fp, _fpT, T, q, s, _keep = RG.export_case(g)
    idx = gold["export_idx"].astype(np.int64)
    plain_ref, plain_ora = gold["export_plain"], O.export_data(asset, fp)[idx]
    assert np.allclose(plain_ref, plain_ora, rtol=2e-6, atol=2e-6)
    baked_ref = gold["export_baked"]
    baked_ours = bake_transform(O.export_data(asset, fp), T, rotation=q, scale=s)[idx]
    assert np.allclose(baked_ref[:, 0:3], baked_ours[:, 0:3], atol=1e-5)                  # positions
    assert np.allclose(baked_ref[:, 55:58], baked_ours[:, 55:58], atol=1e-5)              # log scale
    same = np.abs(baked_ref[:, 58:62] - baked_ours[:, 58:62]).max(1)
    flip = np.abs(baked_ref[:, 58:62] + baked_ours[:, 58:62]).max(1)
    assert np.minimum(same, flip).max() < 1e-5                                            # rotation (q and -q are the same)
    assert np.array_equal(baked_ref[:, 6:9], baked_ours[:, 6:9])                          # band 0
    assert np.abs(baked_ref[:, 9:54] - plain_ref[:, 9:54]).max() > 0.05                   # the rotation does something ...
    assert np.abs(baked_ref[:, 9:54] - baked_ours[:, 9:54]).max() < 2e-5                  # ... and ours is the same rotation


def _stored_vert(gold, name, view):
    """The reference's vertex-shader output for instance 0, computed from the oracle's view data: that view data must
    still be what the stored output was computed from."""
    assert np.array_equal(view[:2], gold[name + "_view_in"]), "the oracle's view data changed: regenerate tests/golden/ref_hlsl.npz"
    return gold[name + "_clip"], gold[name + "_qpos"], gold[name + "_col"]


def test_draw_stages_match_the_reference_shader_code(g, O, gold):
    """vert + frag of RenderGaussianSplats.shader on one rotated, anisotropic splat: the quad the reference emits maps pixel
    centres to quad coordinates (the rasteriser's linear interpolation), frag gives the fragment; the oracle's render of that
    splat (fp32 blend, so the image IS the fragment) must be the same picture."""
    W, H = RG.DRAW_W, RG.DRAW_H
    asset, fp, _keep = RG.draw_case(g, selected=False)
    view = O.calc_view(asset, fp)
    order = np.arange(1, dtype=np.uint32)
    rt = O.render(view, order, W, H, blend_mode=1)
    clip, qpos, col = _stored_vert(gold, "draw", view)
    frag = gold["draw_frag"]
    assert np.array_equal(np.abs(qpos), np.full((4, 2), 2.0, np.float32))                 # quad corners at +-2 (:54-55)
    # pixel position of each corner; interpolation inside a parallelogram is affine: solve quad coords from three corners
    A, px = RG.quad_map(clip, qpos, W, H)
    assert np.allclose(np.array([*px[3], 1.0]) @ A, qpos[3], atol=1e-4)
    quad = np.zeros((H, W), bool)
    checked = drawn = 0
    for x, y, qx, qy in RG.quad_pixels(A, W, H):
        quad[y, x] = True
        edge = min(abs(abs(qx) - 2), abs(abs(qy) - 2)) < 2e-3
        want = frag[y, x]
        if edge or abs(float(np.exp(-(qx * qx + qy * qy))) * col[3] - 1 / 255) < 2e-5:
            continue                                                                       # on the quad edge / discard threshold
        assert np.abs(rt[y, x] - want).max() < 3e-6, (x, y, rt[y, x], want)
        checked += 1
        drawn += int(want[3] > 0)
    assert (rt[~quad, 3] == 0).all()
    assert checked > 700 and drawn > 400


def test_selected_splat_branch_matches_the_reference_shader_code(g, O, gold):
    """With an edit selection bound the reference's vertex shader hands a selected splat to the pixel shader with col.a = -1
    (S/RenderGaussianSplats.shader:63-73) and the pixel shader takes its "selected" branch (:87-101: opacity from the gaussian
    alone, +0.3, a solid magenta ring where exp(power) is in (7/255, 10/255), magenta tint).  The oracle's draw with
    selected_bits must give the picture the compiled reference vert + frag give."""
    W, H = RG.DRAW_W, RG.DRAW_H
    asset, fp, _keep = RG.draw_case(g, selected=True)
    view = O.calc_view(asset, fp)
    order = np.arange(asset.splatCount, dtype=np.uint32)
    bits = np.zeros(2, np.uint32)
    bits[0] = 1                                                                            # splat 0 selected, the padding splats not
    clip, qpos, _col = _stored_vert(gold, "selected", view)
    col = gold["selected_col_sel"]
    assert col[3] == -1.0
    assert gold["selected_col_sel_1"][3] >= 0.0
    plain = O.render(view, order[:1], W, H, blend_mode=1)
    rt = O.render(view, order[:1], W, H, blend_mode=1, selected_bits=bits)
    assert plain[..., 3].max() < 0.03 and rt[..., 3].max() == 1.0                          # opacity 0.02 alone is almost nothing
    frag = gold["selected_frag"]
    A, _px = RG.quad_map(clip, qpos, W, H)
    quad = np.zeros((H, W), bool)
    checked = ring = 0
    for x, y, qx, qy in RG.quad_pixels(A, W, H):
        quad[y, x] = True
        e = float(np.exp(-(qx * qx + qy * qy)))
        if min(abs(abs(qx) - 2), abs(abs(qy) - 2)) < 2e-3 or min(abs(e - 1 / 255), abs(e - 7 / 255), abs(e - 10 / 255)) < 3e-5:
            continue                                                                       # on the quad edge / one of the three thresholds
        want = frag[y, x]
        assert np.abs(rt[y, x] - want).max() < 3e-6, (x, y, rt[y, x], want)
        checked += 1
        ring += int(want[3] == 1.0 and want[0] == 1.0 and want[1] == 0.0)
    assert (rt[~quad, 3] == 0).all()
    assert checked > 700 and ring > 20


def test_rotation_packing_matches_the_reference_shader_code(gold):
    """The importer packs rotations with C# twins of these HLSL functions; the packer (gsa_pack_smallest3 + its 10.10.10.2
    encoder, checked through a one-splat asset) must produce the same code words, and decoding must agree."""
    from unitygaussiansplatting_b200 import _native as N
    lib = N.asset_lib()
    for q, enc_ref, packed_ref, back in zip(RG.rotation_quats(), gold["rot_enc"], gold["rot_packed"], gold["rot_decoded"]):
        ours = np.zeros(4, np.float32)
        lib.gsa_pack_smallest3(q.ctypes.data, ours.ctypes.data)
        assert np.allclose(ours, packed_ref, atol=1e-7)
        enc_ours = (int(ours[0] * 1023.5) | (int(ours[1] * 1023.5) << 10) | (int(ours[2] * 1023.5) << 20) | (int(ours[3] * 3.5) << 30)) & 0xFFFFFFFF
        assert enc_ours == int(enc_ref) or np.abs(ours - packed_ref).max() > 0      # same code word whenever the packed floats are identical
        assert min(np.abs(back - q).max(), np.abs(back + q).max()) < 2.5e-3                # 10-bit components
