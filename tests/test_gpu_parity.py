"""GPU parity tests proper: the CUDA path through the C ABI vs the CPU oracle on the same seeded inputs.
Bar: bit-exact keys / order / SplatViewData; render target within 1e-3 per channel (it is in fact
bit-exact in GS_BLEND_FP16_ROP mode because both sides share one arithmetic contract)."""
import numpy as np
import pytest

from util import camera, lattice_camera, one_splat

pytestmark = pytest.mark.gpu

RT_TOL = 1e-3  # BASELINE.json north_star: pixels within 1e-3 per channel


def _frame_pair(g, O, ctx, asset, cam, blend=0, prev_order=None, **knobs):
    r = g.GaussianSplatRenderer(asset, ctx)
    for k, v in knobs.items():
        setattr(r, k, v)
    r.blend_mode = blend
    if prev_order is not None:
        r.upload_order(prev_order)
    rt = np.zeros((cam.pixelHeight, cam.pixelWidth, 4), np.float32 if blend == 1 else np.float16)
    r.SortAndRenderSplats(cam, rt=rt)
    fp, _keep = g.make_frame_params(cam, r.localToWorldMatrix, r.m_SplatScale, r.m_OpacityScale, r.m_SHOrder, r.m_SHOnly,
                                    r.m_Cutouts, r.m_DeletedBits, asset.splatCount)
    ref = O.frame(asset, fp, prev_order=prev_order, blend_mode=blend, threads=O.max_threads())
    with pytest.raises(g.GsError) as e:       # the fused frame does not materialise _SplatViewData (dead store) ...
        r.readback_view()
    assert e.value.code == -5
    r.CalcViewData(cam)                        # ... the stand-alone entry point does, in full
    got = {"keys": r.readback_keys(), "order": r.readback_order(), "view": r.readback_view(), "rt": rt.astype(np.float32)}
    # and drawing from the stand-alone view data gives the same pixels as the fused frame
    rt2 = np.zeros_like(rt)
    r.DrawSplats(cam, rt2)
    assert np.array_equal(rt2, rt)
    r.Dispose()
    return got, ref


def _assert_frame(got, ref, exact_rt=True):
    assert np.array_equal(got["keys"], ref["keys"]), "sorted distance keys differ"
    assert np.array_equal(got["order"], ref["order"]), "sorted splat indices differ"
    bad = np.nonzero((got["view"] != ref["view"]).any(axis=1))[0]
    assert bad.size == 0, "SplatViewData differs for %d splats, first %s" % (bad.size, bad[:5])
    err = np.abs(got["rt"] - ref["rt"])
    assert np.nanmax(err) <= RT_TOL, "render target max err %g at %s" % (err.max(), np.unravel_index(err.argmax(), err.shape))
    assert not np.isnan(got["rt"]).any()
    if exact_rt:
        assert np.array_equal(got["rt"], ref["rt"]), "fp16-ROP render target is expected to be bit-exact (max err %g)" % err.max()


@pytest.mark.parametrize("quality", ["Medium", "VeryHigh", "High"])
def test_cfg1_lattice_1k(g, O, ctx, quality):
    """BASELINE configs[0]: 1k axis-aligned gaussians with deliberate depth ties."""
    asset = g.synthetic_asset(g.SCENE_LATTICE, 1000, 0x5EED0001, quality)
    got, ref = _frame_pair(g, O, ctx, asset, lattice_camera(g, 256, 256))
    assert (np.diff(ref["keys"].astype(np.int64)) == 0).sum() > 10, "the fixture is supposed to contain depth ties"
    _assert_frame(got, ref)


@pytest.mark.parametrize("quality,n,w,h", [("Medium", 50000, 400, 300), ("VeryHigh", 30000, 320, 180), ("High", 30000, 333, 211)])
def test_clustered_scene(g, O, ctx, quality, n, w, h):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0002, quality)
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, w, h))
    _assert_frame(got, ref)


@pytest.mark.parametrize("quality,n,w,h", [("VeryLow", 20000, 333, 211), ("Low", 17000, 320, 180)])
def test_low_presets_bc7_and_clustered_sh(g, O, ctx, quality, n, w, h):
    """SURVEY 8f N4: BC7 colour (single-texel decode in k_calc_view) and Cluster4k/16k SH palettes (u16 index in `other`)."""
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0031, quality)
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, w, h))
    _assert_frame(got, ref)


def test_bc7_all_modes_through_the_view_kernel(g, O, ctx):
    """A VeryLow asset whose colour blob is replaced by the golden random blocks of all eight BC7 modes."""
    d = np.load(__import__("pathlib").Path(__file__).with_name("golden") / "bc7_blocks.npz")
    n = 20000
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, n, 0x5EED0032, "VeryLow")
    blocks = d["blocks"].reshape(-1)
    reps = -(-asset.colorData.nbytes // blocks.size)
    asset.colorData = np.ascontiguousarray(np.tile(blocks, reps)[:asset.colorData.nbytes])
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, 256, 192))
    _assert_frame(got, ref)


def test_fp32_blend_mode(g, O, ctx):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 40000, 0x5EED0002, "Medium")
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, 320, 240), blend=1)
    _assert_frame(got, ref, exact_rt=True)


def test_tie_order_follows_previous_frame(g, O, ctx):
    """CSCalcDistances gathers through the previous order and the sort is stable (SURVEY 7 'Tie order')."""
    asset = g.synthetic_asset(g.SCENE_LATTICE, 1000, 0x5EED0001, "Medium")
    rng = np.random.default_rng(5)
    prev = rng.permutation(1000).astype(np.uint32)
    got, ref = _frame_pair(g, O, ctx, asset, lattice_camera(g, 128, 128), prev_order=prev)
    _assert_frame(got, ref)
    got2, ref2 = _frame_pair(g, O, ctx, asset, lattice_camera(g, 128, 128))
    assert not np.array_equal(ref["order"], ref2["order"]), "ties must resolve differently for a different history"


def test_second_frame_reuses_order(g, O, ctx):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0003, "Medium")
    r = g.GaussianSplatRenderer(asset, ctx)
    cams = [camera(g, 200, 150), camera(g, 200, 150, pos=(2.0, 1.0, -5.0), forward=(-0.3, -0.1, 1.0))]
    order = np.arange(asset.splatCount, dtype=np.uint32)
    for cam in cams:
        rt = np.zeros((150, 200, 4), np.float16)
        r.SortAndRenderSplats(cam, rt=rt)
        fp, _k = g.make_frame_params(cam)
        ref = O.frame(asset, fp, prev_order=order, threads=O.max_threads())
        order = ref["order"]
        assert np.array_equal(r.readback_order(), order)
        assert np.array_equal(rt.astype(np.float32), ref["rt"])
    r.Dispose()


@pytest.mark.parametrize("knobs", [dict(m_SHOrder=0), dict(m_SHOrder=1), dict(m_SHOrder=2), dict(m_SHOnly=True),
                                   dict(m_SplatScale=0.5, m_OpacityScale=3.0), dict(m_SplatScale=2.0, m_OpacityScale=0.2)])
def test_render_knobs(g, O, ctx, knobs):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0004, "Medium")
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, 256, 160), **knobs)
    _assert_frame(got, ref)


def test_object_transform_cutouts_and_deleted_bits(g, O, ctx):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0005, "Medium")
    # GSTestScene.unity:363-365: rotation quaternion (-0.9925,0,0,0.1219), scale (1,1,-1)
    o2w = g.trs((0.3, -0.2, 0.5), g.quat_to_mat((-0.9925, 0.0, 0.0, 0.1219)), (1, 1, -1)).astype(np.float32)
    cut_e = (g.trs((0, 0, 0), None, (0.25, 0.25, 0.25)).astype(np.float32), 0)            # ellipsoid of radius 4
    cut_b = (g.trs((0, 0, 0), None, (0.5, 0.5, 0.5)).astype(np.float32), 1 | 0x100)       # inverted box
    bits = np.random.default_rng(3).integers(0, 2**32, (asset.splatCount + 31) // 32, dtype=np.uint32)
    got, ref = _frame_pair(g, O, ctx, asset, camera(g, 256, 160), localToWorldMatrix=o2w, m_Cutouts=[cut_e, cut_b, (np.eye(4), 0xFFFFFFFF)],
                           m_DeletedBits=bits)
    _assert_frame(got, ref)
    assert (got["view"][:, 3].view(np.float32) == 0).mean() > 0.3


def test_single_huge_and_degenerate_splats(g, O, ctx):
    cam = camera(g, 200, 120, pos=(0, 0, -3))
    for kw in (dict(scale=(3.0, 3.0, 3.0)), dict(scale=(1e-4, 1e-4, 1e-4)), dict(pos=(0, 0, -10.0)), dict(opacity=0.003),
               dict(scale=(2.0, 0.001, 0.001), quat=(0.1, 0.5, 0.3, 0.8))):
        asset = one_splat(g, n_pad=3, **kw)
        got, ref = _frame_pair(g, O, ctx, asset, cam)
        _assert_frame(got, ref)


def test_composite_matches_oracle(g, O, ctx):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0002, "Medium")
    cam = camera(g, 320, 200)
    r = g.GaussianSplatRenderer(asset, ctx)
    rng = np.random.default_rng(1)
    bg = rng.random((200, 320, 4), np.float32)
    for dt in (np.float32, np.float16):
        rt = np.zeros((200, 320, 4), np.float16)
        tgt = bg.astype(dt).copy()
        r.m_FrameCounter = 0
        r.SortAndRenderSplats(cam, rt=rt, camera_target=tgt)
        want = O.composite(rt.astype(np.float32), bg.astype(dt).astype(np.float32), target_fp16=(dt == np.float16))
        assert np.array_equal(tgt.astype(np.float32), want)
        # stand-alone gs_composite on host images
        tgt2 = bg.astype(dt).copy()
        r.Composite(rt, tgt2)
        assert np.array_equal(tgt2, tgt)
    r.Dispose()


def test_staged_calls_equal_fused_frame(g, O, ctx):
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 30000, 0x5EED0006, "Medium")
    cam = camera(g, 300, 200)
    a, b = g.GaussianSplatRenderer(asset, ctx), g.GaussianSplatRenderer(asset, ctx)
    rt_a, rt_b = np.zeros((200, 300, 4), np.float16), np.zeros((200, 300, 4), np.float16)
    a.SortAndRenderSplats(cam, rt=rt_a)
    b.SortPoints(cam); b.CalcViewData(cam); b.DrawSplats(cam, rt_b)
    assert np.array_equal(rt_a, rt_b) and np.array_equal(a.readback_order(), b.readback_order())
    a.Dispose(); b.Dispose()


def test_error_behaviour(g, ctx):
    asset = g.synthetic_asset(g.SCENE_LATTICE, 1000, 1, "Medium")
    r = g.GaussianSplatRenderer(asset, ctx)
    cam = camera(g, 64, 64)
    with pytest.raises(g.GsError) as e:      # DrawSplats before CalcViewData -> GS_ERR_NOT_READY, nothing crashes
        r.DrawSplats(cam, np.zeros((64, 64, 4), np.float16))
    assert e.value.code == -5
    with pytest.raises(g.GsError):
        r.m_SHOrder = 7
        r.CalcViewData(cam)
    r.Dispose()


@pytest.mark.parametrize("count,band", [(2, 1), (3, 2), (4, 1), (8, 1)])
def test_tile_partition_bands_reassemble_the_full_frame(g, O, ctx, count, band):
    """SURVEY 8e.1 on one GPU: render every partition band-packed, all-gather by hand, gs_unshuffle_bands == full frame."""
    import ctypes as C
    import torch
    from unitygaussiansplatting_b200 import _native as N
    from unitygaussiansplatting_b200.multigpu import BandPartition, TILE, unshuffle
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 30000, 0x5EED0007, "Medium")
    cam = camera(g, 333, 211)
    r = g.GaussianSplatRenderer(asset, ctx)
    full = np.zeros((211, 333, 4), np.float16)
    r.SortAndRenderSplats(cam, rt=full)
    parts = [BandPartition(211, count, i, band) for i in range(count)]
    gathered = torch.zeros((count, parts[0].rows_per_partition, 333, 4), dtype=torch.float16, device="cuda")
    for p in parts:
        r.partition, r.band_packed = p.options(), True
        own_px = p.own_tile_rows() * TILE
        if own_px:
            r.SortAndRenderSplats(cam, rt=gathered[p.index][:own_px])
    ctx.sync()
    out = torch.zeros((211, 333, 4), dtype=torch.float16, device="cuda")
    unshuffle(ctx, gathered, parts[0], out)
    ctx.sync()
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), full)
    # host-image variant of the same call
    host = np.zeros((211, 333, 4), np.float16)
    unshuffle(ctx, gathered, parts[0], host)
    assert np.array_equal(host, full)
    r.Dispose()


def test_async_readback_equals_blocking(g, ctx):
    """GS_FLAG_ASYNC_READBACK: host images are filled by a copy stream while the next frame runs; after gs_sync they hold
    exactly what the blocking path returns, for several frames in rotation over two pinned images."""
    import torch
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 60000, 0x5EED0081, "Medium")
    r = g.GaussianSplatRenderer(asset, ctx)
    cams = [camera(g, 400, 300, pos=(0.2 * k, 0.5, -6.0 + 0.3 * k)) for k in range(5)]
    want = []
    for cam in cams:
        rt = np.zeros((300, 400, 4), np.float16)
        r.SortAndRenderSplats(cam, rt=rt)
        want.append(rt)
    r.ResetOrder()
    r.m_FrameCounter = 0
    pins = [torch.zeros((300, 400, 4), dtype=torch.float16).pin_memory() for _ in range(2)]
    r.async_readback = True
    got = []
    for k, cam in enumerate(cams):
        if k >= 2:
            ctx.sync()                      # the image about to be reused must have landed: keep a copy of it first
            got.append(pins[k & 1].numpy().copy())
        r.SortAndRenderSplats(cam, rt=pins[k & 1].numpy())
    ctx.sync()
    # frames 3 and 4 are still in the two images; frames 0..2 were copied out above
    got.append(pins[1].numpy().copy())      # frame 3
    got.append(pins[0].numpy().copy())      # frame 4
    for k in range(5):
        assert np.array_equal(got[k].view(np.uint16), want[k].view(np.uint16)), "frame %d" % k
    r.Dispose()


@pytest.mark.parametrize("device_rt", [False, True])
def test_two_renderers_share_one_render_target(g, O, ctx, device_rt):
    """GaussianSplatRenderSystem draws every active splat object into ONE _GaussianSplatRT, cleared once
    (R/GaussianSplatRenderer.cs:111-168,196), nearest object first, each with its own sort.  GS_FLAG_LOAD_RT makes the
    second object blend under the first; the oracle draws the concatenated, per-object-sorted list in one go."""
    import torch
    a = g.synthetic_asset(g.SCENE_CLUSTERED, 30000, 0x5EED0091, "Medium")
    b = g.synthetic_asset(g.SCENE_CLUSTERED, 20000, 0x5EED0092, "VeryHigh")
    cam = camera(g, 400, 300)
    ra, rb = g.GaussianSplatRenderer(a, ctx), g.GaussianSplatRenderer(b, ctx)
    ra.localToWorldMatrix = g.trs(position=(1.5, 0.0, 3.0)).astype(np.float32)      # further away: drawn second
    rb.localToWorldMatrix = g.trs(position=(-1.0, 0.2, 0.5), scale=(0.7, 0.7, 0.7)).astype(np.float32)
    rt = torch.zeros((300, 400, 4), dtype=torch.float16, device="cuda") if device_rt else np.zeros((300, 400, 4), np.float16)
    active = g.SortAndRenderSplatsMulti([ra, rb], cam, rt)
    assert active == [rb, ra]
    ctx.sync()
    got = rt.cpu().numpy() if device_rt else rt
    views, orders, base = [], [], 0
    for r in active:
        fp, _keep = g.make_frame_params(cam, r.localToWorldMatrix)
        ref = O.frame(r.m_Asset, fp, threads=O.max_threads())
        assert np.array_equal(r.readback_order(), ref["order"])
        views.append(ref["view"]); orders.append(ref["order"] + np.uint32(base)); base += r.splatCount
    want = O.render(np.concatenate(views), np.concatenate(orders), 400, 300, 0, O.max_threads())
    assert got.any()
    assert np.array_equal(got.astype(np.float32), want)
    # and the flag matters: drawing the second object from a cleared target gives something else
    solo = np.zeros((300, 400, 4), np.float16)
    ra.SortAndRenderSplats(cam, rt=solo)
    assert not np.array_equal(solo, got)
    ra.Dispose(); rb.Dispose()


def test_selected_splats(g, O, ctx):
    """_SplatSelectedBits (S/RenderGaussianSplats.shader:63-73,87-101): the fused frame, the staged draw and an emulated group of 3
    all reproduce the oracle's picture of a scene with every 5th splat selected (plus some that are also deleted)."""
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 40000, 0x5EED0093, "Medium")
    n = asset.splatCount
    rng = np.random.default_rng(5)
    sel = np.zeros((n + 31) // 32, np.uint32)
    ids = np.arange(0, n, 5)
    np.bitwise_or.at(sel, ids >> 5, np.uint32(1) << (ids & 31).astype(np.uint32))
    dele = rng.integers(0, 2 ** 32, sel.size, dtype=np.uint64).astype(np.uint32) & rng.integers(0, 2 ** 32, sel.size, dtype=np.uint64).astype(np.uint32)
    cam = camera(g, 400, 300)
    r = g.GaussianSplatRenderer(asset, ctx)
    r.m_SelectedBits, r.m_DeletedBits = sel, dele
    rt = np.zeros((300, 400, 4), np.float16)
    r.SortAndRenderSplats(cam, rt=rt)
    fp, _keep = g.make_frame_params(cam, deleted_bits=dele, selected_bits=sel, splat_count=n)
    ref = O.frame(asset, fp, threads=O.max_threads())
    plain_fp, _k2 = g.make_frame_params(cam, deleted_bits=dele, splat_count=n)
    plain = O.frame(asset, plain_fp, threads=O.max_threads())
    assert not np.array_equal(plain["rt"], ref["rt"])
    assert np.array_equal(rt.astype(np.float32), ref["rt"])
    r.CalcViewData(cam)
    assert np.array_equal(r.readback_view(), ref["view"])          # the selection does not touch _SplatViewData
    rt2 = np.zeros_like(rt)
    r.DrawSplats(cam, rt2)
    assert np.array_equal(rt2, rt)
    r.Dispose()
    from unitygaussiansplatting_b200.multigpu import GaussianSplatGroup
    grp = GaussianSplatGroup.create(asset, [0, 0, 0], emulate=True)
    grp.m_SelectedBits, grp.m_DeletedBits = sel, dele
    rts = [np.zeros_like(rt) for _ in range(3)]
    grp.SortAndRenderSplats(cam, rts=rts)
    for i in range(3):
        assert np.array_equal(rts[i], rt)
    grp.close()


def test_orthographic_projection(g, O, ctx):
    """gs_frame accepts any GPU projection matrix.  With an orthographic one clip.w == 1, so the fused kernel's chunk / splat
    culls must take the view depth from the model-view matrix (not from clip.w): the fused frame has to equal both the staged
    path (gs_calc_view + gs_render, which culls nothing) and the oracle."""
    import ctypes as C
    from unitygaussiansplatting_b200 import _native as N
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 40000, 0x5EED0094, "Medium")
    cam = camera(g, 400, 300)
    r = g.GaussianSplatRenderer(asset, ctx)
    fp = r.frame_params(cam)
    half_h, n_, f_ = 4.0, 0.3, 100.0
    half_w = half_h * 400 / 300
    ortho = np.array([[1 / half_w, 0, 0, 0], [0, 1 / half_h, 0, 0], [0, 0, -2 / (f_ - n_), -(f_ + n_) / (f_ - n_)], [0, 0, 0, 1]], np.float64)
    ortho[1, :] *= -1.0                                  # render-texture flip, as GL.GetGPUProjectionMatrix(.., true) does
    ortho[2, :] = ortho[2, :] * -0.5 + ortho[3, :] * 0.5  # reversed z
    C.memmove(C.addressof(fp) + N.GsFrameParams.mat_proj_gpu.offset, g.camera.colmajor(ortho).ctypes.data, 64)
    rt = np.zeros((300, 400, 4), np.float16)
    r.SortAndRenderSplats(cam, rt=rt, fp=fp)
    ref = O.frame(asset, fp, threads=O.max_threads())
    assert rt.any()
    assert np.array_equal(r.readback_order(), ref["order"])
    assert np.array_equal(rt.astype(np.float32), ref["rt"])
    lib = N.native()
    N.check(ctx.handle, lib.gs_calc_view(ctx.handle, r._asset, C.byref(fp)))
    assert np.array_equal(r.readback_view(), ref["view"])
    rt2 = np.zeros_like(rt)
    opt = r._options()
    im = g.renderer._image(rt2, 400, 300)
    N.check(ctx.handle, lib.gs_render(ctx.handle, r._asset, C.byref(fp), C.byref(opt), C.byref(im)))
    assert np.array_equal(rt2, rt)
    r.Dispose()


def test_scene_depth_buffer(g, O, ctx):
    """GsFrameParams.scene_depth: the pass's ZTest LEqual against the camera's depth buffer (S/RenderGaussianSplats.shader:8-12,
    R/GaussianSplatRenderer.cs:195).  A wall at view distance 6 over the left 60 % of the screen hides what lies behind it; the fused
    frame, the staged draw, a device-resident depth buffer and an emulated group of 3 all equal the oracle's picture."""
    import torch
    asset = g.synthetic_asset(g.SCENE_CLUSTERED, 40000, 0x5EED0095, "Medium")
    n = asset.splatCount
    cam = camera(g, 400, 300)
    P = cam.gpuProjectionMatrix(True).astype(np.float64)
    clip = P @ np.array([0.0, 0.0, -6.0, 1.0])                 # view space looks down -z
    z_wall = np.float32(clip[2] / clip[3])
    assert 0.0 < z_wall < 1.0
    depth = np.zeros((300, 400), np.float32)
    depth[:, :240] = z_wall
    r = g.GaussianSplatRenderer(asset, ctx)
    r.sceneDepth = depth
    rt = np.zeros((300, 400, 4), np.float16)
    r.SortAndRenderSplats(cam, rt=rt)
    fp, _keep = g.make_frame_params(cam, splat_count=n, scene_depth=depth)
    ref = O.frame(asset, fp, threads=O.max_threads())
    free_fp, _k2 = g.make_frame_params(cam, splat_count=n)
    free = O.frame(asset, free_fp, threads=O.max_threads())
    assert np.array_equal(ref["rt"][:, 240:], free["rt"][:, 240:]) and not np.array_equal(ref["rt"][:, :240], free["rt"][:, :240])
    assert np.array_equal(rt.astype(np.float32), ref["rt"])
    assert np.array_equal(r.readback_order(), ref["order"])
    r.CalcViewData(cam)                                         # staged: view data (with the quad depths), then the draw
    assert np.array_equal(r.readback_view(), ref["view"])
    rt2 = np.zeros_like(rt)
    r.DrawSplats(cam, rt2)
    assert np.array_equal(rt2, rt)
    r.sceneDepth = torch.from_numpy(depth).cuda()               # device-resident depth buffer: used in place
    rt3 = np.zeros_like(rt)
    r.SortAndRenderSplats(cam, rt=rt3)
    assert np.array_equal(rt3, rt)
    r.sceneDepth = None                                         # and without one the wall is gone
    rt4 = np.zeros_like(rt)
    r.SortAndRenderSplats(cam, rt=rt4)
    assert np.array_equal(rt4.astype(np.float32), free["rt"])
    r.Dispose()
    from unitygaussiansplatting_b200.multigpu import GaussianSplatGroup
    grp = GaussianSplatGroup.create(asset, [0, 0, 0], emulate=True)
    grp.sceneDepth = depth
    rts = [np.zeros_like(rt) for _ in range(3)]
    grp.SortAndRenderSplats(cam, rts=rts)
    for i in range(3):
        assert np.array_equal(rts[i], rt)
    grp.close()
