"""The CUDA path against the reference's own shader code: what it computed is stored in tests/golden/ref_hlsl.npz (see
tests/test_reference_hlsl.py).  Same comparisons as tests/test_reference_hlsl.py, with the C-ABI library's output in place
of the oracle's.  Named test_zz_* so that it runs after the parity tests proper."""
import numpy as np
import pytest

from test_reference_hlsl import GOLD, RG, _cov, _unsortable
from util import camera, view_fields

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("quality", RG.GPU_QUALITIES)
def test_cuda_view_data_and_keys_match_the_reference_shader_code(g, ctx, quality):
    gold = np.load(GOLD / "ref_hlsl.npz")
    n = 20000
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0091, quality)
    cam = camera(g, 320, 240)
    r = g.GaussianSplatRenderer(asset, ctx)
    r.SortPoints(cam)
    r.CalcViewData(cam)
    view, keys, order = r.readback_view(), r.readback_keys(), r.readback_order()
    fp, _keep = g.make_frame_params(cam, r.localToWorldMatrix, r.m_SplatScale, r.m_OpacityScale, r.m_SHOrder, r.m_SHOnly)
    assert bytes(fp) == bytes(g.make_frame_params(cam)[0]), "the stored reference results were computed with the default uniforms"
    assert np.array_equal(RG.unpackbits(gold["gpu_%s_w_le0" % quality], n), view[:, 3].view(np.float32) <= 0)
    ref, got = view_fields(gold["gpu_%s_rows" % quality]), view_fields(view[gold["gpu_%s_idx" % quality].astype(np.int64)])
    assert np.array_equal(ref["pos"][:, 3] <= 0, got["pos"][:, 3] <= 0)
    assert (np.abs(ref["pos"] - got["pos"]).max(1) <= 2e-6 * (1 + np.abs(got["pos"]).max(1))).all()
    vis = got["pos"][:, 3] > 0
    for ch in "rgb":
        d = np.abs(ref[ch][vis] - got[ch][vis])
        assert (d <= np.maximum(np.abs(got[ch][vis]), 2.0 ** -14) * 2.0 ** -9).all(), ch
    assert np.array_equal(ref["a"][vis], got["a"][vis])
    cr, cg = _cov(ref)[vis], _cov(got)[vis]
    rel = np.abs(cr - cg).reshape(-1, 4).max(1) / (cg[:, 0, 0] + cg[:, 1, 1])
    assert np.percentile(rel, 50) < 1e-6 and np.percentile(rel, 99) < 2e-5 and rel.max() < 2e-3
    # sorted keys: the reference's key of each stored splat, at the position the sort gave it, is the same depth to a
    # couple of ulp, and those keys ascend in draw order
    kidx = gold["gpu_%s_key_idx" % quality].astype(np.int64)
    where = np.argsort(order)[kidx]                      # position of each stored splat in the draw order
    by_pos = np.argsort(where)
    kr, kg = gold["gpu_%s_keys" % quality][by_pos], keys[where[by_pos]]
    assert np.abs(_unsortable(kr) - _unsortable(kg)).max() <= 4e-6
    assert (np.diff(_unsortable(kr).astype(np.float64)) >= -8e-6).all()
    r.Dispose()
