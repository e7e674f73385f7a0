/* gsplat_b200.h -- C ABI of the B200-native Gaussian-splat render path.
 *
 * This is the drop-in boundary for the hot path of aras-p/UnityGaussianSplatting
 * (view-calc -> depth sort -> rasterise/blend -> composite).  The reference has no
 * native plugin (SURVEY.md section 0, F3): all GPU work is recorded by C# into a Unity
 * CommandBuffer.  Every entry point below therefore replaces a *C# call site* and
 * the compute/raster work it dispatches; the citation next to each symbol names it
 * (paths relative to the reference repo, R/ = package/Runtime, S/ = package/Shaders).
 *
 * Rules of the ABI:
 *   - plain C: pointers, sizes, PODs.  No C++/torch types.
 *   - every function returns a GsStatus (0 = ok, <0 = error) and never throws or
 *     aborts; gs_last_error() gives the text.  This mirrors the reference's
 *     "log and skip" behaviour (R/GaussianSplatRenderer.cs:361-369,447-448,655).
 *   - one GsContext per CUDA device; calls on one context are serialised by the caller.
 *     All work is enqueued on the context's stream; only gs_sync/gs_readback_* /
 *     host-memory images block.
 *   - matrices are float[16], column-major exactly like UnityEngine.Matrix4x4
 *     (element (row r, col c) at [c*4 + r]).
 */
#ifndef GSPLAT_B200_H
#define GSPLAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define GS_API __declspec(dllexport)
#else
#define GS_API __attribute__((visibility("default")))
#endif

typedef struct GsContext GsContext;
typedef struct GsAsset GsAsset;

typedef enum GsStatus {
  GS_OK = 0,
  GS_ERR_INVALID_ARGUMENT = -1,
  GS_ERR_CUDA = -2,
  GS_ERR_OUT_OF_MEMORY = -3,
  GS_ERR_UNSUPPORTED_FORMAT = -4, /* a format enum outside R/GaussianSplatAsset.cs:31-81 */
  GS_ERR_NOT_READY = -5,          /* e.g. gs_render before gs_calc_view */
  GS_ERR_NO_DEVICE = -6
} GsStatus;

/* R/GaussianSplatAsset.cs:31-37 (VectorFormat), S/GaussianSplatting.hlsl:319-323 */
typedef enum GsVectorFormat { GS_VEC_FLOAT32 = 0, GS_VEC_NORM16 = 1, GS_VEC_NORM11 = 2, GS_VEC_NORM6 = 3 } GsVectorFormat;
/* R/GaussianSplatAsset.cs:51-57 (ColorFormat) */
typedef enum GsColorFormat { GS_COL_FLOAT32X4 = 0, GS_COL_FLOAT16X4 = 1, GS_COL_NORM8X4 = 2, GS_COL_BC7 = 3 } GsColorFormat;
/* R/GaussianSplatAsset.cs:70-81 (SHFormat); values >= 4 are clustered palettes */
typedef enum GsSHFormat { GS_SH_FLOAT32 = 0, GS_SH_FLOAT16 = 1, GS_SH_NORM11 = 2, GS_SH_NORM6 = 3, GS_SH_CLUSTER64K = 4,
                          GS_SH_CLUSTER32K = 5, GS_SH_CLUSTER16K = 6, GS_SH_CLUSTER8K = 7, GS_SH_CLUSTER4K = 8 } GsSHFormat;

/* The asset blobs exactly as GaussianSplatAsset exposes them
 * (R/GaussianSplatAsset.cs:219-237; uploaded by CreateResourcesForAsset,
 * R/GaussianSplatRenderer.cs:373-421).  Pointers are HOST memory, borrowed for the
 * duration of gs_asset_upload; the library copies everything to HBM.
 * `color` is the 2048-wide, 16x16-Morton-swizzled texture image
 * (R/GaussianSplatAsset.cs:152-160, S/GaussianSplatting.hlsl:181-194), row-major.
 * `chunks` may be NULL / chunk_bytes 0 (fully-float32 assets,
 * R/GaussianSplatRenderer.cs:391-405). */
typedef struct GsAssetDesc {
  uint32_t splat_count;
  uint32_t pos_format, scale_format, sh_format, color_format;
  const void *pos, *other, *sh, *color, *chunks;
  uint64_t pos_bytes, other_bytes, sh_bytes, color_bytes, chunk_bytes;
} GsAssetDesc;

/* R/GaussianCutout.cs:20-40, S/SplatUtilities.compute:96-100 (68 bytes) */
typedef struct GsCutout {
  float mat[16];            /* cutout worldToLocal * renderer localToWorld */
  uint32_t type_and_flags;  /* low byte: 0 ellipsoid, 1 box, 0xFF ignore; 0x100: invert */
} GsCutout;

/* Per-frame uniforms.  Field-by-field these are the values C# binds in
 * CalcViewData (R/GaussianSplatRenderer.cs:579-610), SortPoints (:612-639) and
 * SortAndRenderSplats (:137-149). */
typedef struct GsFrameParams {
  float mat_object_to_world[16];  /* tr.localToWorldMatrix            (:587) */
  float mat_world_to_object[16];  /* tr.worldToLocalMatrix            (:588) */
  float mat_view[16];             /* cam.worldToCameraMatrix, -z fwd  (:586,:617) */
  float mat_proj_gpu[16];         /* UNITY_MATRIX_P = GL.GetGPUProjectionMatrix(cam.projectionMatrix, true);
                                     an engine global in the reference (S/SplatUtilities.compute:200,236) */
  float screen_w, screen_h;       /* _VecScreenParams.xy              (:591) */
  float cam_pos_world[3];         /* _VecWorldSpaceCameraPos          (:592) */
  float splat_scale;              /* m_SplatScale   [0.1,2]           (:599) */
  float opacity_scale;            /* m_OpacityScale [0.05,20]         (:600) */
  uint32_t sh_order;              /* m_SHOrder 0..3                   (:601) */
  uint32_t sh_only;               /* m_SHOnly                         (:602) */
  uint32_t cutout_count;          /* _SplatCutoutsCount (R/GaussianSplatRenderer.cs:506-508) */
  uint32_t reserved0;
  const GsCutout *cutouts;        /* host pointer, cutout_count entries, may be NULL */
  const uint32_t *deleted_bits;   /* host pointer, ceil(N/32) words or NULL == _SplatBitsValid 0 (:496-501) */
  const uint32_t *selected_bits;  /* host pointer, ceil(N/32) words or NULL: the edit selection (_SplatSelectedBits, :496).  A
                                     selected splat is drawn by the pixel shader's "selected" branch: magenta outline + tint,
                                     opacity from the gaussian alone (S/RenderGaussianSplats.shader:63-73,87-101) */
  const float *scene_depth;       /* optional: the camera's depth buffer the splat pass tests against.  The reference binds the
                                     current depth target beside _GaussianSplatRT (R/GaussianSplatRenderer.cs:195) and keeps
                                     ShaderLab's default ZTest LEqual with ZWrite Off (S/RenderGaussianSplats.shader:8-12), so
                                     splats behind opaque scene geometry are not drawn.  screen_w x screen_h float32, rows
                                     tightly packed, in mat_proj_gpu's convention (reversed Z: 1 = near plane), where LEqual is
                                     evaluated as "fragment depth >= stored depth"; every fragment of a splat has the depth
                                     clip.z / clip.w of its centre (the quad is flat).  NULL = no depth test. */
  uint32_t scene_depth_on_device; /* 0: scene_depth is host memory (uploaded per frame), 1: device memory (used in place) */
  uint32_t reserved1;
} GsFrameParams;

typedef enum GsPixelFormat {
  GS_PIX_RGBA16F = 0,   /* _GaussianSplatRT: R16G16B16A16_SFloat (R/GaussianSplatRenderer.cs:194) */
  GS_PIX_RGBA32F = 1
} GsPixelFormat;

typedef enum GsMemory { GS_MEM_HOST = 0, GS_MEM_DEVICE = 1 } GsMemory;

typedef struct GsImage {
  void *data;
  uint32_t width, height;
  uint32_t row_pitch_bytes;  /* 0 = tightly packed */
  uint32_t format;           /* GsPixelFormat */
  uint32_t memory;           /* GsMemory: where `data` lives */
} GsImage;

/* How the render-target blend is evaluated.
 * GS_BLEND_FP16_ROP reproduces the reference: the RT is RGBA16F, so the fixed-function
 * blender (Blend OneMinusDstAlpha One, S/RenderGaussianSplats.shader:11) rounds dst to
 * half after EVERY splat.  GS_BLEND_FP32 keeps dst in float32 registers and rounds once. */
typedef enum GsBlendMode { GS_BLEND_FP16_ROP = 0, GS_BLEND_FP32 = 1 } GsBlendMode;

#define GS_BAND_PIXELS 64u /* height of one partition row = edge of a binning cell (csrc/gs_common.cuh kBin) */
#define GS_TILE_PIXELS 16u /* edge of a raster tile = granularity of row_begin/row_end (csrc/gs_common.cuh kTile) */

typedef struct GsRenderOptions {
  uint32_t blend_mode;        /* GsBlendMode */
  uint32_t band_packed;       /* 1: rt holds only this partition's rows, packed: own 64-pixel row k -> pixel rows
                                 [64k, 64k+64); rt->height must be 64 * (number of own rows).  This is the
                                 send buffer of the all-gather. */
  /* Screen-tile partition for multi-GPU (SURVEY 8e.1): this context composites only
   * 64-pixel rows (GS_BAND_PIXELS, the binning cell) r with (r / band_rows) % partition_count == partition_index.
   * partition_count 0 or 1 = whole image. */
  uint32_t partition_index, partition_count, band_rows;
  uint32_t flags;             /* GsRenderFlags */
  /* Contiguous partition (what gs_group_frame uses): when row_end > row_begin this context composites only the 16-pixel
   * raster-tile rows [row_begin, row_end) (GS_TILE_PIXELS), straight into their natural place of a full-size target;
   * partition_* and band_packed are then ignored.  0,0 = not used. */
  uint32_t row_begin, row_end;
} GsRenderOptions;

typedef enum GsRenderFlags {
  /* gs_frame with a HOST render target returns as soon as the read-back is ENQUEUED (on a second stream, double-buffered
   * device staging): frame k's copy overlaps frame k+1's kernels.  The image must be pinned (cudaHostRegister /
   * cudaMallocHost) and must not be read, nor handed to another frame, until gs_sync (or two later frames) -- the
   * managed-side analogue is AsyncGPUReadback.  Errors of the frame (e.g. a truncated bin list) surface at gs_sync. */
  GS_FLAG_ASYNC_READBACK = 1u,
  /* Do not start from a cleared target: read `rt` and blend this asset UNDER what is already there.  The reference
   * clears _GaussianSplatRT once per camera (R/GaussianSplatRenderer.cs:196) and then draws every active splat object
   * into it, nearest object first (GatherSplatsForCamera :73-105, loop :111-168): render the first object without this
   * flag and each further one with it.  A host `rt` is uploaded first. */
  GS_FLAG_LOAD_RT = 2u
} GsRenderFlags;

/* Per-stage device times of the last gs_frame/gs_sort/gs_calc_view/gs_render call with
 * timing enabled (GaussianSplat.Sort / CalcView / Draw / Compose profiler markers,
 * R/GaussianSplatRenderer.cs:20-22,287).  Milliseconds, CUDA events on the context stream. */
typedef struct GsStageTimes {
  float distances_ms, sort_ms, view_ms, bin_ms, raster_ms, composite_ms, total_ms;
  float sort_pass_ms[4];
  uint64_t tile_entries;      /* (tile, splat) pairs produced by binning */
  uint32_t kernel_launches;   /* kernels of this library launched by the call */
  uint32_t reserved;
} GsStageTimes;

/* ---- lifetime ---------------------------------------------------------------- */
/* EnsureSorterAndRegister + resource setup, R/GaussianSplatRenderer.cs:450-475.
 * stream_handle: an existing cudaStream_t to enqueue on (0 = create a private stream). */
GS_API int gs_create(int cuda_device, void *stream_handle, GsContext **out);
GS_API void gs_destroy(GsContext *ctx);
GS_API const char *gs_last_error(GsContext *ctx); /* ctx may be NULL: last global error */
GS_API int gs_sync(GsContext *ctx);
GS_API int gs_set_timing(GsContext *ctx, int enabled);
GS_API int gs_get_stage_times(GsContext *ctx, GsStageTimes *out);
GS_API const char *gs_version(void);

/* ---- asset --------------------------------------------------------------------- */
/* CreateResourcesForAsset + InitSortBuffers + CSSetIndices,
 * R/GaussianSplatRenderer.cs:373-445, S/SplatUtilities.compute:59-67 */
GS_API int gs_asset_upload(GsContext *ctx, const GsAssetDesc *desc, GsAsset **out);
/* DisposeResourcesForAsset / OnDisable, R/GaussianSplatRenderer.cs:533-577 */
GS_API void gs_asset_destroy(GsAsset *asset);
/* CSSetIndices: order[i] = i (S/SplatUtilities.compute:59-67) */
GS_API int gs_asset_reset_order(GsAsset *asset);
GS_API uint32_t gs_asset_splat_count(const GsAsset *asset);

/* ---- the hot path -------------------------------------------------------------- */
/* SortPoints: CSCalcDistances + GpuSorting.Dispatch
 * (R/GaussianSplatRenderer.cs:612-639, S/SplatUtilities.compute:69-82,
 *  R/GpuSorting.cs:142-198).  The order buffer persists across calls: distances are
 * gathered through the previous order and the sort is stable, exactly as the reference. */
GS_API int gs_sort(GsContext *ctx, GsAsset *asset, const GsFrameParams *fp);
/* CalcViewData: CSCalcViewData (R/GaussianSplatRenderer.cs:579-610,
 * S/SplatUtilities.compute:189-252) */
GS_API int gs_calc_view(GsContext *ctx, GsAsset *asset, const GsFrameParams *fp);
/* cmb.DrawProcedural(matSplats, 6 idx, N instances) into the cleared _GaussianSplatRT
 * (R/GaussianSplatRenderer.cs:156-165,194-196; S/RenderGaussianSplats.shader).
 * Output: premultiplied RGBA (format/memory per `rt`).  Requires gs_calc_view first. */
GS_API int gs_render(GsContext *ctx, GsAsset *asset, const GsFrameParams *fp,
                     const GsRenderOptions *opt, GsImage *rt);
/* Composite pass: GaussianComposite.shader:35-39 with Blend SrcAlpha OneMinusSrcAlpha
 * (R/GaussianSplatRenderer.cs:206-210).  `camera_target` is read-modify-write. */
GS_API int gs_composite(GsContext *ctx, const GsImage *rt, GsImage *camera_target);
/* SortAndRenderSplats for one renderer, one stream, no host round trips:
 * (do_sort ? gs_sort : nothing) -> gs_calc_view -> gs_render [-> gs_composite if
 * camera_target != NULL].  do_sort == (m_FrameCounter % m_SortNthFrame == 0),
 * R/GaussianSplatRenderer.cs:120-121.  rt may be NULL when camera_target is given
 * (the RT then lives only in library scratch).
 * In the reference _SplatViewData only carries CSCalcViewData's results to the draw call; the fused
 * path hands them to its compositor directly and does NOT materialise that buffer (nor the colour of
 * splats that cannot produce a fragment).  Pixels are unaffected; gs_readback_view after gs_frame
 * returns GS_ERR_NOT_READY -- call gs_calc_view when the buffer itself is wanted. */
GS_API int gs_frame(GsContext *ctx, GsAsset *asset, const GsFrameParams *fp,
                    const GsRenderOptions *opt, int do_sort, GsImage *rt, GsImage *camera_target);

/* Multi-GPU epilogue (SURVEY 8e.1): `gathered` is the all-gather of every partition's band-packed
 * render target, [partition_count][rows_per_partition][width] pixels in DEVICE memory, where
 * rows_per_partition = 64 * max over partitions of own 64-pixel rows.  Writes the assembled width x height
 * image (device or host) in normal row order. */
GS_API int gs_unshuffle_bands(GsContext *ctx, const void *gathered, uint32_t partition_count, uint32_t band_rows,
                              uint32_t rows_per_partition, uint32_t pixel_format, GsImage *out);

/* ---- several GPUs of one box (SURVEY 8e; the reference itself is single-GPU) ----------------------------------
 * A group renders ONE frame on G GPUs and leaves, on every GPU, exactly what gs_frame leaves on one: the same draw order
 * (bit for bit: the persistent _SplatSortKeys contract of R/GpuSorting.cs:142-198 seeded by last frame's order,
 * R/GaussianSplatRenderer.cs:612-639) and the same render target.  Per frame and GPU:
 *   - the depth sort is sharded by KEY RANGE: every GPU computes the (cheap) key table, takes the splats whose key lies
 *     between two shared splitters -- in last frame's order, so ties keep the reference's order -- sorts only those, and one
 *     exchange of the id slabs gives every GPU the whole order (SURVEY 8e.2).  After gs_group_join the slabs travel as
 *     peer-to-peer stores over NVLink into CUDA-IPC mappings of the peers' order buffers (no collective call); groups made
 *     by gs_group_create, and boxes without IPC, use one ncclAllGather;
 *   - view-calc, binning and compositing are sharded by SCREEN ROWS: a contiguous range of 16-pixel rows per GPU
 *     (GsRenderOptions.row_begin/row_end), rebalanced every frame from the measured per-row cost, composited straight
 *     into place, then one NCCL exchange of the row ranges (SURVEY 8e.1: "a single all-gather of the composited tile buffers";
 *     grouped broadcasts of the exact sizes, in place, on a transfer stream that overlaps the next frame's sort).
 * Two ways to form a group:
 *   gs_group_join    one process per GPU (torchrun-style): every process passes its own context, the group size, its rank
 *                    and the 128-byte id rank 0 got from gs_group_unique_id (sent over any host channel);
 *   gs_group_create  one process driving n GPUs (what a Unity host would do): the library creates the n contexts.
 *                    GS_GROUP_EMULATE lets device indices repeat: the "GPUs" are then n contexts on the same device and the
 *                    exchanges are device-to-device copies -- the whole sharded path on a single-GPU box, for tests.
 * NCCL is bound at run time (libnccl.so.2; a copy already loaded into the process, e.g. PyTorch's, is reused). */
typedef struct GsGroup GsGroup;
#define GS_GROUP_ID_BYTES 128u
#define GS_GROUP_MAX_GPUS 16u
typedef enum GsGroupFlags { GS_GROUP_EMULATE = 1u } GsGroupFlags;

typedef struct GsGroupStats {      /* of the first local member, last gs_group_frame with timing enabled (gs_set_timing) */
  float distances_ms, slab_sort_ms, order_exchange_ms, view_ms, bin_ms, raster_ms, image_exchange_ms, total_ms;
  uint32_t group_size, rank;
  uint32_t row_bounds[GS_GROUP_MAX_GPUS + 1];   /* 16-pixel row ranges of this frame: GPU g composites [row_bounds[g], row_bounds[g+1]) */
  uint32_t slab_counts[GS_GROUP_MAX_GPUS];      /* splats each GPU sorted this frame */
} GsGroupStats;

GS_API int gs_group_unique_id(void *id_out /* GS_GROUP_ID_BYTES */);
GS_API int gs_group_join(GsContext *ctx, uint32_t group_size, uint32_t rank, const void *id, GsGroup **out);
GS_API int gs_group_create(const int *cuda_devices, uint32_t n, uint32_t flags, GsGroup **out);
GS_API void gs_group_destroy(GsGroup *group);
GS_API uint32_t gs_group_size(const GsGroup *group);
GS_API uint32_t gs_group_local_count(const GsGroup *group);          /* members driven by this process: 1 after join, n after create */
GS_API GsContext *gs_group_context(GsGroup *group, uint32_t local_index);
/* CreateResourcesForAsset on every local member (R/GaussianSplatRenderer.cs:373-445): assets_out[local_count]. */
GS_API int gs_group_asset_upload(GsGroup *group, const GsAssetDesc *desc, GsAsset **assets_out);
/* SortAndRenderSplats (R/GaussianSplatRenderer.cs:108-169) on the group.  assets[i] / rts[i] belong to local member i;
 * rts[i] is a full-size image (device or host memory; NULL = this member keeps the frame in library scratch only).  Every
 * non-NULL rts[i] ends up holding the COMPLETE render target.  `opt`: blend_mode, and GS_FLAG_ASYNC_READBACK for host images
 * (the call returns with the read-back enqueued; gs_group_sync completes it).  Collective: every process of the
 * group must call it with the same parameters. */
GS_API int gs_group_frame(GsGroup *group, GsAsset *const *assets, const GsFrameParams *fp, const GsRenderOptions *opt, int do_sort,
                          GsImage *const *rts);
GS_API int gs_group_sync(GsGroup *group);
GS_API int gs_group_get_stats(GsGroup *group, GsGroupStats *out);
/* The row balancer by itself (host arithmetic, no GPU): splits `rows` 16-pixel rows with the given measured costs into
 * `parts` contiguous ranges of near-equal cost; bounds_out[parts + 1], bounds_out[0] = 0, bounds_out[parts] = rows. */
GS_API int gs_group_balance_rows(const uint32_t *row_cost, uint32_t rows, uint32_t parts, uint32_t *bounds_out);

/* ---- stand-alone sorter (GpuSorting.Dispatch, R/GpuSorting.cs:142-198) ----------- */
/* Stable ascending sort of `count` (uint32 key, uint32 payload) pairs in place in DEVICE
 * buffers keys/payload (KEY_UINT PAYLOAD_UINT SHOULD_ASCEND SORT_PAIRS, R/GpuSorting.cs:115-128). */
GS_API int gs_sort_pairs_device(GsContext *ctx, uint32_t *d_keys, uint32_t *d_payload, uint32_t count);
/* Same through HOST buffers (copies in, sorts, copies out, blocks). */
GS_API int gs_sort_pairs_host(GsContext *ctx, uint32_t *keys, uint32_t *payload, uint32_t count);

/* ---- export (EditExportData, R/GaussianSplatRenderer.cs:936-958 -> CSExportData, S/SplatUtilities.compute:616-669) ---- */
/* Decodes every splat of the uploaded asset back to the INRIA .ply attribute record: n x 62 floats in HOST memory `dst`
 * (pos, nor, f_dc, f_rest channel-major, opacity as logit, log scale, rot wxyz -- the InputSplatData layout,
 * E/Utils/GaussianFileReader.cs:17-26).  nor = (1,1,1) marks a splat the cutouts remove (`cutouts` as in GsFrameParams;
 * may be NULL).  gsa_ply_write (gsplat_asset.h) then writes the file ExportPlyFile writes
 * (E/GaussianSplatRendererEditor.cs:394-445).  The baked variant (bake_transform != 0) is a host pass over these records,
 * gsa_bake_transform (gsplat_asset.h); the device entry point itself returns GS_ERR_UNSUPPORTED_FORMAT for the flag.  Blocks. */
GS_API int gs_export_splats(GsContext *ctx, GsAsset *asset, const GsCutout *cutouts, uint32_t cutout_count,
                            uint32_t bake_transform, void *dst);

/* ---- test hooks (blocking device->host reads) ----------------------------------- */
GS_API int gs_readback_order(GsAsset *asset, uint32_t *dst);      /* _SplatSortKeys, N words */
GS_API int gs_readback_keys(GsAsset *asset, uint32_t *dst);       /* _SplatSortDistances, N words (sorted after gs_sort) */
GS_API int gs_readback_view(GsAsset *asset, void *dst);           /* _SplatViewData, N x 40 bytes (S/GaussianSplatting.hlsl:610-615) */
GS_API int gs_upload_order(GsAsset *asset, const uint32_t *src);  /* seed a previous-frame order */

/* ---- Unity render-thread entry (SURVEY 8f N2) -------------------------------------- */
/* Unity executes native GPU work on its render thread through CommandBuffer.IssuePluginEventAndData(func, eventId, data)
 * (the reference records everything into CommandBuffers, R/GaussianSplatRenderer.cs:108-211).  `func` is what
 * gs_unity_get_render_event_func returns (signature of Unity's UnityRenderingEventAndData); `data` points to a
 * GsUnityFrameEvent the managed side keeps alive (pinned) until the command buffer has executed.  The callback runs
 * the requested entry point and stores its GsStatus in `status` -- "log and skip", never a throw across the boundary. */
typedef enum GsUnityEvent {
  GS_UNITY_EVENT_FRAME = 1,   /* gs_frame(ctx, asset, &params, &options, do_sort, has_rt ? &rt : NULL, has_camera_target ? &camera_target : NULL) */
  GS_UNITY_EVENT_SYNC = 2     /* gs_sync(ctx) */
} GsUnityEvent;

typedef struct GsUnityFrameEvent {
  GsContext *ctx;
  GsAsset *asset;
  GsFrameParams params;
  GsRenderOptions options;
  int32_t do_sort;            /* m_FrameCounter % m_SortNthFrame == 0 */
  int32_t status;             /* out: GsStatus of the call (GS_ERR_NOT_READY until the event has run) */
  uint32_t has_rt, has_camera_target;
  GsImage rt, camera_target;
} GsUnityFrameEvent;

typedef void (*GsUnityRenderEventAndDataFunc)(int event_id, void *data);
GS_API GsUnityRenderEventAndDataFunc gs_unity_get_render_event_func(void);
GS_API uint32_t gs_unity_frame_event_size(void);   /* sizeof(GsUnityFrameEvent), for the managed side's layout check */

/* ---- device-pointer access for zero-copy hosts (torch / CUDA-Vulkan interop) ----- */
GS_API void *gs_context_stream(GsContext *ctx);
GS_API void *gs_asset_device_ptr(GsAsset *asset, int which); /* 0 order, 1 keys, 2 view */

#ifdef __cplusplus
}
#endif
#endif /* GSPLAT_B200_H */
