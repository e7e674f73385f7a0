// gs_api.cu -- the C ABI of libgsplat_b200.so (include/gsplat_b200.h): context, asset
// residency in HBM, per-frame uniform derivation and stage sequencing on one CUDA stream.
//
// This file is the native counterpart of the C# frame driver: CreateResourcesForAsset /
// InitSortBuffers (R/GaussianSplatRenderer.cs:373-445), CalcViewData (:579-610), SortPoints
// (:612-639) and SortAndRenderSplats (:108-169).  There is no CPU fallback anywhere: without
// a CUDA device gs_create fails with GS_ERR_NO_DEVICE.
#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "gs_internal.cuh"

namespace gs {
static thread_local std::string g_last_error;
}  // namespace gs

namespace gs {

int fail(GsContext *ctx, int code, const std::string &msg) {
  g_last_error = msg;
  if (ctx) ctx->err = msg;
  return code;
}
int fail_cuda(GsContext *ctx, cudaError_t e, const char *expr, const char *file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, expr);
  return fail(ctx, e == cudaErrorMemoryAllocation ? GS_ERR_OUT_OF_MEMORY : GS_ERR_CUDA, buf);
}

#define M_(m, r, c) ((m)[(c)*4 + (r)])
// Matrix4x4 operator* as Unity evaluates it (plain float ops, no contraction: this TU is
// compiled with -Xcompiler -ffp-contract=off).
static void mat_mul(const float *a, const float *b, float *o) {
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r)
      M_(o, r, c) = M_(a, r, 0) * M_(b, 0, c) + M_(a, r, 1) * M_(b, 1, c) + M_(a, r, 2) * M_(b, 2, c) + M_(a, r, 3) * M_(b, 3, c);
}

// Uniform derivation of CalcViewData (R/GaussianSplatRenderer.cs:586-606) and SortPoints (:617-629),
// plus the CalcCovariance2D constants that depend only on the camera (S/GaussianSplatting.hlsl:62-70).
FrameConsts make_frame_consts(const GsFrameParams *fp) {
  FrameConsts fc;
  memset(&fc, 0, sizeof(fc));
  float mv[16], vp[16], w2c[16], mvs[16];
  mat_mul(fp->mat_view, fp->mat_object_to_world, mv);
  mat_mul(fp->mat_proj_gpu, fp->mat_view, vp);
  memcpy(w2c, fp->mat_view, 64);
  M_(w2c, 2, 0) *= -1.0f; M_(w2c, 2, 1) *= -1.0f; M_(w2c, 2, 2) *= -1.0f;
  mat_mul(w2c, fp->mat_object_to_world, mvs);
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) {
      fc.o2w[r * 4 + c] = M_(fp->mat_object_to_world, r, c);
      fc.mv[r * 4 + c] = M_(mv, r, c);
    }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) fc.w2o[r * 3 + c] = M_(fp->mat_world_to_object, r, c);
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) fc.vp[r * 4 + c] = M_(vp, r, c);
  for (int c = 0; c < 4; ++c) fc.sort_row[c] = M_(mvs, 2, c);
  for (int k = 0; k < 3; ++k) fc.cam_pos[k] = fp->cam_pos_world[k];
  const float p00 = M_(fp->mat_proj_gpu, 0, 0), p11 = M_(fp->mat_proj_gpu, 1, 1);
  const float aspect = p00 / p11;
  const float tanFovX = 1.0f / p00;
  const float tanFovY = 1.0f / (p11 * aspect);  // == tanFovX: reference quirk, kept
  fc.limX = 1.3f * tanFovX;
  fc.limY = 1.3f * tanFovY;
  fc.focal = fp->screen_w * p00 / 2.0f;
  fc.splatScale2 = fp->splat_scale * fp->splat_scale;
  fc.opacityScale = fp->opacity_scale;
  {
    // Bound behind the fused kernel's cheap culls.  CalcCovariance2D (S/GaussianSplatting.hlsl:56-90): cov2d = T S T^t + 0.3 I with
    // T = J W, J = (focal/tz) [I2 | -u], |u|^2 <= limX^2 + limY^2 (the clamp), W = MV 3x3, S = R diag(s^2) R^t splatScale^2.
    // So lambda1 <= |J|_2^2 |W|_2^2 smax^2 splatScale^2 + 0.3 with |J|_2^2 = (focal/tz)^2 (1 + |u|^2); the quad reaches at most
    // 2 (|a1x| + |a2x|) <= 2 sqrt(2) sqrt(2 lambda1) pixels from its centre.  |W|_2^2 is bounded by the smaller of the Frobenius
    // norm and the Gershgorin bound of W^t W (exact for rotation x uniform scale, the usual transform).
    double a[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, fro = 0.0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        for (int k = 0; k < 3; ++k) a[i][j] += (double)M_(mv, k, i) * (double)M_(mv, k, j);
        fro += (double)M_(mv, i, j) * (double)M_(mv, i, j);
      }
    double gersh = 0.0;
    for (int i = 0; i < 3; ++i) {
      double row = 0.0;
      for (int j = 0; j < 3; ++j) row += a[i][j] < 0 ? -a[i][j] : a[i][j];
      if (row > gersh) gersh = row;
    }
    const double w2 = (gersh < fro ? gersh : fro) * 1.0001;
    fc.extentK = (float)((double)fc.focal * fc.focal * (1.0 + (double)fc.limX * fc.limX + (double)fc.limY * fc.limY) * w2 * fc.splatScale2);
  }
  fc.screenW = fp->screen_w;
  fc.screenH = fp->screen_h;
  fc.shOrder = fp->sh_order;
  fc.shOnly = fp->sh_only;
  fc.cutoutCount = fp->cutouts ? fp->cutout_count : 0;
  fc.bitsValid = fp->deleted_bits ? 1u : 0u;
  fc.selValid = fp->selected_bits ? 1u : 0u;
  fc.binsX = ((uint32_t)fp->screen_w + kBin - 1) / kBin;
  fc.binsY = ((uint32_t)fp->screen_h + kBin - 1) / kBin;
  return fc;
}

static int grow(GsContext *ctx, void **p, size_t *cur, size_t need) {
  if (*cur >= need && *p) return GS_OK;
  if (*p) { cudaStreamSynchronize(ctx->stream); cudaFree(*p); *p = nullptr; *cur = 0; }
  GS_CUDA_TRY(ctx, cudaMalloc(p, need));
  *cur = need;
  return GS_OK;
}

int ensure_sort_scratch(GsContext *ctx, uint32_t capacity) {
  if (capacity <= ctx->sort_capacity) return GS_OK;
  cudaStreamSynchronize(ctx->stream);
  cudaFree(ctx->sort.alt_keys); cudaFree(ctx->sort.alt_vals); cudaFree(ctx->sort.lookback);
  ctx->sort.alt_keys = ctx->sort.alt_vals = ctx->sort.lookback = nullptr;
  ctx->sort_capacity = 0;
  GS_CUDA_TRY(ctx, cudaMalloc(&ctx->sort.alt_keys, (size_t)capacity * 4));
  GS_CUDA_TRY(ctx, cudaMalloc(&ctx->sort.alt_vals, (size_t)capacity * 4));
  ctx->lookback_words = sort_lookback_words(capacity, 4);
  GS_CUDA_TRY(ctx, cudaMalloc(&ctx->sort.lookback, ctx->lookback_words * 4));
  ctx->sort.max_tiles = (capacity + kSortTileItems - 1) / kSortTileItems;
  ctx->sort_capacity = capacity;
  return GS_OK;
}

static int ensure_bin_scratch(GsContext *ctx, uint32_t n, uint32_t tiles, uint32_t min_capacity) {
  uint64_t want = (uint64_t)n * 8;
  if (want < (4u << 20)) want = 4u << 20;
  if (want > (768u << 20)) want = 768u << 20;
  if (want < min_capacity) want = min_capacity;
  if ((uint32_t)want > ctx->bin.capacity) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->bin.tile_keys); cudaFree(ctx->bin.tile_vals);
    ctx->bin.tile_keys = ctx->bin.tile_vals = nullptr;
    ctx->bin.capacity = 0;
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.tile_keys, want * 4));
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.tile_vals, want * 4));
    ctx->bin.capacity = (uint32_t)want;
  }
  int rc = ensure_sort_scratch(ctx, ctx->bin.capacity > n ? ctx->bin.capacity : n);
  if (rc) return rc;
  const uint32_t blocks = n / 1024 + 2 < 1024u ? 1024u : n / 1024 + 2;   // the binner's ticket + range totals (<= 593 words) fit too
  if (blocks > ctx->bin_blocks_cap) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->bin.block_sums);
    ctx->bin.block_sums = nullptr;
    ctx->bin_blocks_cap = 0;
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.block_sums, (size_t)blocks * 4));
    ctx->bin_blocks_cap = blocks;
  }
  if (tiles > ctx->tiles_cap) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->bin.bin_ranges);
    ctx->bin.bin_ranges = nullptr;
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.bin_ranges, (size_t)tiles * 8));
    ctx->tiles_cap = tiles;
  }
  return GS_OK;
}

void rec(GsContext *ctx, int e) {
  if (ctx->timing) { cudaEventRecord(ctx->ev[e], ctx->stream); ctx->ev_valid[e] = true; }
}
static float ev_ms(GsContext *ctx, int a, int b) {
  if (!ctx->ev_valid[a] || !ctx->ev_valid[b]) return 0.0f;
  float ms = 0.0f;
  if (cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]) != cudaSuccess) { cudaGetLastError(); return 0.0f; }
  return ms;
}

// GS_FLAG_ASYNC_READBACK plumbing, created on first use
static int ensure_async_readback(GsContext *ctx) {
  if (ctx->copy_stream) return GS_OK;
  GS_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    GS_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_rt_ready[i], cudaEventDisableTiming));
    GS_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_copy_done[i], cudaEventDisableTiming));
  }
  return GS_OK;
}

uint32_t pix_bytes(uint32_t fmt) { return fmt == GS_PIX_RGBA16F ? 8u : 16u; }

int upload_frame_inputs(GsContext *ctx, GsAsset *as, const GsFrameParams *fp, cudaStream_t stream) {
  if (fp->cutouts && fp->cutout_count) {
    if (fp->cutout_count > ctx->cutout_cap) {
      cudaStreamSynchronize(ctx->stream);
      cudaFree(ctx->d_cutouts);
      ctx->d_cutouts = nullptr;
      GS_CUDA_TRY(ctx, cudaMalloc(&ctx->d_cutouts, sizeof(GsCutout) * fp->cutout_count));
      ctx->cutout_cap = fp->cutout_count;
    }
    GS_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_cutouts, fp->cutouts, sizeof(GsCutout) * fp->cutout_count, cudaMemcpyHostToDevice, stream));
  }
  if (fp->deleted_bits) {
    size_t words = ((size_t)as->av.n + 31) / 32;
    if (words > ctx->deleted_words) {
      cudaStreamSynchronize(ctx->stream);
      cudaFree(ctx->d_deleted);
      ctx->d_deleted = nullptr;
      GS_CUDA_TRY(ctx, cudaMalloc(&ctx->d_deleted, words * 4));
      ctx->deleted_words = words;
    }
    GS_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_deleted, fp->deleted_bits, words * 4, cudaMemcpyHostToDevice, stream));
  }
  if (fp->selected_bits) {
    size_t words = ((size_t)as->av.n + 31) / 32;
    if (words > ctx->selected_words) {
      cudaStreamSynchronize(ctx->stream);
      cudaFree(ctx->d_selected);
      ctx->d_selected = nullptr;
      GS_CUDA_TRY(ctx, cudaMalloc(&ctx->d_selected, words * 4));
      ctx->selected_words = words;
    }
    GS_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_selected, fp->selected_bits, words * 4, cudaMemcpyHostToDevice, stream));
  }
  return GS_OK;
}

// The scene depth buffer the splat pass is tested against (GsFrameParams.scene_depth): used in place when it is device
// memory, uploaded on `stream` when it is host memory.
int bind_depth(GsContext *ctx, const GsFrameParams *fp, cudaStream_t stream) {
  ctx->cur_depth = nullptr;
  if (!fp->scene_depth) return GS_OK;
  if (fp->scene_depth_on_device) { ctx->cur_depth = fp->scene_depth; return GS_OK; }
  const size_t bytes = (size_t)(uint32_t)fp->screen_w * (uint32_t)fp->screen_h * sizeof(float);
  if (bytes > ctx->depth_bytes) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_depth);
    ctx->d_depth = nullptr; ctx->depth_bytes = 0;
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->d_depth, bytes));
    ctx->depth_bytes = bytes;
  }
  GS_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_depth, fp->scene_depth, bytes, cudaMemcpyHostToDevice, stream));
  ctx->cur_depth = ctx->d_depth;
  return GS_OK;
}

int check_params(GsContext *ctx, GsAsset *as, const GsFrameParams *fp) {
  if (!ctx || !as || !fp) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null context/asset/params");
  if (as->ctx != ctx) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "asset belongs to another context");
  GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));   // the caller's current device may be another one
  if (!(fp->screen_w >= 1.0f) || !(fp->screen_h >= 1.0f) || fp->screen_w > 8160.0f || fp->screen_h > 8160.0f)
    return fail(ctx, GS_ERR_INVALID_ARGUMENT, "screen size must be in [1,8160] (8-bit bin indices)");
  if (fp->sh_order > 3) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "sh_order must be 0..3");
  return GS_OK;
}

static int do_sort(GsContext *ctx, GsAsset *as, const FrameConsts &fc) {
  GsNvtxRange nvtx("GaussianSplat.Sort");
  int rc = ensure_sort_scratch(ctx, as->av.n);
  if (rc) return rc;
  rec(ctx, EV_BEGIN);
  GS_CUDA_TRY(ctx, cudaMemsetAsync(ctx->sort.ghist, 0, 4 * 256 * 4, ctx->stream));
  launch_calc_distances(as->av, fc, as->key_table, ctx->sort.ghist, ctx->stream);
  rec(ctx, EV_DIST);
  cudaEvent_t pe[5] = {ctx->ev[EV_SORT0], ctx->ev[EV_SORT1], ctx->ev[EV_SORT2], ctx->ev[EV_SORT3], ctx->ev[EV_SORT4]};
  launch_sort_pairs(as->keys, as->order, as->d_n, as->av.n, 4, 8, true, ctx->sort, ctx->stream, ctx->timing ? pe : nullptr,
                    as->key_table);
  if (ctx->timing) for (int e = EV_SORT0; e <= EV_SORT4; ++e) ctx->ev_valid[e] = true;
  ctx->launches += 1 + 4;
  GS_CUDA_TRY(ctx, cudaGetLastError());
  return GS_OK;
}

static GsRenderOptions default_opts() {
  GsRenderOptions o;
  memset(&o, 0, sizeof(o));
  return o;
}

int do_view(GsContext *ctx, GsAsset *as, const GsFrameParams *fp, const FrameConsts &fc, bool cull, const GsRenderOptions &opt,
            cudaStream_t stream) {
  GsNvtxRange nvtx("GaussianSplat.CalcView");
  int rc = upload_frame_inputs(ctx, as, fp, stream);
  if (rc) return rc;
  const bool own = stream == ctx->stream;   // the group path runs view-calc beside the sort on a second stream and times it itself
  if (own) rec(ctx, EV_VIEW0);
  if (fp->scene_depth && !as->zndc) GS_CUDA_TRY(ctx, cudaMalloc(&as->zndc, (size_t)as->av.n * sizeof(float) + 16));
  as->zndc_valid = fp->scene_depth != nullptr;
  launch_calc_view(as->av, fc, ctx->d_cutouts, ctx->d_deleted, ctx->d_selected, as->view, as->rect, as->draw, as->block_bits,
                   as->zndc_valid ? as->zndc : nullptr, cull, make_partition(opt), stream);
  if (own) rec(ctx, EV_VIEW1);
  ctx->launches += 1;
  as->view_valid = !cull;
  as->draw_valid = true;
  {
    const gs::Partition p = make_partition(opt);
    as->draw_part[0] = p.range ? p.t0 : p.index; as->draw_part[1] = cull ? (p.range ? 0xFFFFFFFFu : p.count) : 0; as->draw_part[2] = p.range ? p.t1 : p.band;
  }
  as->view_w = (uint32_t)fp->screen_w;
  as->view_h = (uint32_t)fp->screen_h;
  GS_CUDA_TRY(ctx, cudaGetLastError());
  return GS_OK;
}

// binning + raster into a device image
int do_render(GsContext *ctx, GsAsset *as, const FrameConsts &fc, const GsRenderOptions &opt, void *d_rt, uint32_t pitch,
                     uint32_t fmt) {
  GsNvtxRange nvtx("GaussianSplat.Draw");
  const uint32_t tiles = fc.binsX * fc.binsY;
  int rc = ensure_bin_scratch(ctx, as->av.n, tiles, 0);
  if (rc) return rc;
  {  // raster-tile cost history (launch order); invalidated when the tile grid changes
    // per-tile state is indexed by the tile's id in the whole image, whatever part of it this context composites
    const uint32_t rtiles = (((uint32_t)fc.screenW + kTile - 1) / kTile) * fc.binsY * (kBin / kTile);
    if (rtiles > ctx->raster_tiles_cap) {
      cudaStreamSynchronize(ctx->stream);
      cudaFree(ctx->bin.tile_cost); cudaFree(ctx->bin.tile_order);
      ctx->bin.tile_cost = ctx->bin.tile_order = nullptr;
      GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.tile_cost, (size_t)rtiles * 4));
      GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.tile_order, (size_t)rtiles * 4));
      ctx->raster_tiles_cap = rtiles;
      ctx->raster_tiles_cur = 0;
    }
    if (rtiles != ctx->raster_tiles_cur) {
      GS_CUDA_TRY(ctx, cudaMemsetAsync(ctx->bin.tile_cost, 0, (size_t)rtiles * 4, ctx->stream));
      ctx->raster_tiles_cur = rtiles;
    }
  }
  int bin_launches = 0;
  const BinScratch lists = launch_binning(fc, opt, as->av.n, as->order, as->rect, as->block_bits, ctx->bin, ctx->sort, ctx->stream, &bin_launches);
  rec(ctx, EV_BIN1);
  launch_raster(fc, opt, as->draw, lists, d_rt, pitch, fmt, ctx->stream, ctx->cur_depth ? as->zndc : nullptr, ctx->cur_depth);
  rec(ctx, EV_RASTER1);
  ctx->launches += bin_launches + 3;  // bin_emit, look-back clear, 1-2 sort passes; bin_ranges, tile_order, raster
  GS_CUDA_TRY(ctx, cudaGetLastError());
  return GS_OK;
}


int image_ok(GsContext *ctx, const GsImage *im, uint32_t W, uint32_t H, uint32_t *pitch) {
  if (!im || !im->data) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "image is null");
  if (im->format > GS_PIX_RGBA32F) return fail(ctx, GS_ERR_UNSUPPORTED_FORMAT, "unsupported pixel format");
  if (im->width != W || im->height != H) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "image size does not match screen size");
  uint32_t p = im->row_pitch_bytes ? im->row_pitch_bytes : W * pix_bytes(im->format);
  if (p < W * pix_bytes(im->format) || (p % pix_bytes(im->format)) != 0) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "bad row pitch");
  *pitch = p;
  return GS_OK;
}

// options shared by gs_render / gs_frame: validated copy
int check_options(GsContext *ctx, const FrameConsts &fc, GsRenderOptions &opt) {
  if (opt.blend_mode > GS_BLEND_FP32) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "bad blend mode");
  if (opt.row_end > opt.row_begin) {
    const uint32_t rows = ((uint32_t)fc.screenH + kTile - 1) / kTile;
    if (opt.row_end > rows) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "row_end beyond the last 16-pixel row of the screen");
    opt.band_packed = 0; opt.partition_count = 0; opt.partition_index = 0;
  } else {
    opt.row_begin = opt.row_end = 0;
  }
  return GS_OK;
}

// what the compositor starts from in a device staging image: the host image's content (GS_FLAG_LOAD_RT), or zeros where a
// partition leaves rows untouched
static int init_staging(GsContext *ctx, const GsRenderOptions &opt, void *d_rt, uint32_t d_pitch, uint32_t W, uint32_t H, uint32_t fmt,
                        const GsImage *host_rt, uint32_t host_pitch) {
  if (opt.flags & GS_FLAG_LOAD_RT) {
    if (host_rt) GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(d_rt, d_pitch, host_rt->data, host_pitch, (size_t)W * pix_bytes(fmt), H, cudaMemcpyHostToDevice, ctx->stream));
    else GS_CUDA_TRY(ctx, cudaMemsetAsync(d_rt, 0, (size_t)d_pitch * H, ctx->stream));
  } else if (opt.partition_count > 1 || opt.row_end > opt.row_begin) {
    GS_CUDA_TRY(ctx, cudaMemsetAsync(d_rt, 0, (size_t)d_pitch * H, ctx->stream));
  }
  return GS_OK;
}

static int check_bin_overflow(GsContext *ctx) {
  uint32_t ec[2] = {0, 0};
  GS_CUDA_TRY(ctx, cudaMemcpyAsync(ec, ctx->bin.entry_count, 8, cudaMemcpyDeviceToHost, ctx->stream));
  GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->times.tile_entries = ec[0];
  if (ec[1]) return fail(ctx, GS_ERR_OUT_OF_MEMORY, "tile-list capacity exceeded (splat footprints cover too many tiles)");
  return GS_OK;
}

}  // namespace gs

using namespace gs;

extern "C" {

const char *gs_version(void) { return "gsplat_b200 0.1 (sm_100a)"; }

const char *gs_last_error(GsContext *ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int gs_create(int cuda_device, void *stream_handle, GsContext **out) {
  if (!out) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "out is null");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    return fail(nullptr, GS_ERR_NO_DEVICE, "no CUDA device: libgsplat_b200 has no CPU fallback");
  }
  if (cuda_device < 0 || cuda_device >= count) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "bad device index");
  GsContext *ctx = new (std::nothrow) GsContext();
  if (!ctx) return fail(nullptr, GS_ERR_OUT_OF_MEMORY, "host allocation failed");
  ctx->device = cuda_device;
  auto init = [&]() -> int {
    GS_CUDA_TRY(ctx, cudaSetDevice(cuda_device));
    if (stream_handle) ctx->stream = (cudaStream_t)stream_handle;
    else {
      // own stream: highest priority, so that the group path's helper stream (view-calc, lowest priority) only fills what the
      // sort / compositing chain on this stream leaves idle
      int least = 0, greatest = 0;
      GS_CUDA_TRY(ctx, cudaDeviceGetStreamPriorityRange(&least, &greatest));
      GS_CUDA_TRY(ctx, cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, greatest));
      ctx->own_stream = true;
    }
    for (int i = 0; i < EV_COUNT; ++i) GS_CUDA_TRY(ctx, cudaEventCreate(&ctx->ev[i]));
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->sort.ghist, 4 * 256 * 4));
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->sort.tickets, 4 * 4));
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->d_scalar, 16 * 4));
    GS_CUDA_TRY(ctx, cudaMalloc(&ctx->bin.entry_count, 4 * 4));
    GS_CUDA_TRY(ctx, cudaMemsetAsync(ctx->bin.entry_count, 0, 16, ctx->stream));
    return GS_OK;
  };
  const int rc = init();
  if (rc != GS_OK) {
    g_last_error = ctx->err;   // keep the text reachable through gs_last_error(NULL)
    gs_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return GS_OK;
}

void gs_destroy(GsContext *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  cudaFree(ctx->sort.alt_keys); cudaFree(ctx->sort.alt_vals); cudaFree(ctx->sort.lookback);
  cudaFree(ctx->sort.ghist); cudaFree(ctx->sort.tickets); cudaFree(ctx->d_scalar);
  cudaFree(ctx->bin.bin_ranges); cudaFree(ctx->bin.tile_cost); cudaFree(ctx->bin.tile_order); cudaFree(ctx->bin.block_sums); cudaFree(ctx->bin.entry_count); cudaFree(ctx->bin.tile_keys); cudaFree(ctx->bin.tile_vals);
  cudaFree(ctx->rt_scratch); cudaFree(ctx->tgt_scratch); cudaFree(ctx->d_cutouts); cudaFree(ctx->d_deleted); cudaFree(ctx->d_selected); cudaFree(ctx->d_depth);
  if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  for (int i = 0; i < 2; ++i) {
    cudaFree(ctx->rt_async[i]);
    if (ctx->ev_rt_ready[i]) cudaEventDestroy(ctx->ev_rt_ready[i]);
    if (ctx->ev_copy_done[i]) cudaEventDestroy(ctx->ev_copy_done[i]);
  }
  for (int i = 0; i < EV_COUNT; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int gs_sync(GsContext *ctx) {
  if (!ctx) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null context");
  GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  // frames rendered into device images are not checked when they are enqueued: surface a truncated bin list here
  const int rc = check_bin_overflow(ctx);
  if (ctx->copy_stream) {   // asynchronous read-backs in flight complete here
    GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    ctx->copy_pending[0] = ctx->copy_pending[1] = false;
  }
  return rc;
}

int gs_set_timing(GsContext *ctx, int enabled) {
  if (!ctx) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null context");
  ctx->timing = enabled != 0;
  return GS_OK;
}

int gs_get_stage_times(GsContext *ctx, GsStageTimes *out) {
  if (!ctx || !out) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  GsStageTimes t = ctx->times;
  t.distances_ms = ev_ms(ctx, EV_BEGIN, EV_DIST);
  t.sort_ms = ev_ms(ctx, EV_SORT0, EV_SORT4);
  for (int p = 0; p < 4; ++p) t.sort_pass_ms[p] = ev_ms(ctx, EV_SORT0 + p, EV_SORT1 + p);
  t.view_ms = ev_ms(ctx, EV_VIEW0, EV_VIEW1);
  t.bin_ms = ev_ms(ctx, EV_VIEW1, EV_BIN1);
  t.raster_ms = ev_ms(ctx, EV_BIN1, EV_RASTER1);
  t.composite_ms = ev_ms(ctx, EV_RASTER1, EV_COMP1);
  int first = ctx->ev_valid[EV_BEGIN] ? EV_BEGIN : EV_VIEW0, last = EV_VIEW1;
  for (int e = EV_VIEW1; e < EV_COUNT; ++e) if (ctx->ev_valid[e]) last = e;
  t.total_ms = ev_ms(ctx, first, last);
  uint32_t ec[2] = {0, 0};
  if (ctx->bin.entry_count) cudaMemcpy(ec, ctx->bin.entry_count, 8, cudaMemcpyDeviceToHost);
  t.tile_entries = ec[0];
  t.kernel_launches = ctx->launches;
  *out = t;
  return GS_OK;
}

int gs_asset_upload(GsContext *ctx, const GsAssetDesc *d, GsAsset **out) {
  if (!ctx || !d || !out) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  // HasValidAsset, R/GaussianSplatRenderer.cs:361-368
  if (d->splat_count == 0 || !d->pos || !d->other || !d->sh || !d->color) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "asset has no splats or a null blob");
  if (d->pos_format > 3 || d->scale_format > 3) return fail(ctx, GS_ERR_UNSUPPORTED_FORMAT, "unknown vector format");
  if (d->color_format > GS_COL_BC7) return fail(ctx, GS_ERR_UNSUPPORTED_FORMAT, "unknown colour format");
  if (d->sh_format > GS_SH_CLUSTER4K) return fail(ctx, GS_ERR_UNSUPPORTED_FORMAT, "unknown SH format");
  const uint64_t n = d->splat_count;
  // bytes per texel: Float32x4 16, Float16x4 8, Norm8x4 4, BC7 1 (16-byte 4x4 blocks), R/GaussianSplatAsset.cs:58-68
  const uint32_t colsz = d->color_format == 0 ? 16u : d->color_format == 1 ? 8u : d->color_format == 2 ? 4u : 1u;
  // clustered SH (R/GaussianSplatAsset.cs:135-150,187-198): the blob is a palette of 64k..4k Float16 entries and every
  // splat carries a u16 palette index at the end of its `other` record (S/GaussianSplatting.hlsl:447-448,467-470)
  const bool clustered = d->sh_format > GS_SH_NORM6;
  const uint64_t sh_items = clustered ? (uint64_t)(65536u >> (d->sh_format - GS_SH_CLUSTER64K)) : n;
  const uint32_t shst = d->sh_format == 0 ? 192u : (d->sh_format == 1 || clustered) ? 96u : d->sh_format == 2 ? 60u : 32u;
  uint32_t th = (uint32_t)((n + kTexWidth - 1) / kTexWidth);
  th = (th + 15) / 16 * 16;
  if (d->pos_bytes < n * vec_stride(d->pos_format) || d->other_bytes < n * (4 + vec_stride(d->scale_format) + (clustered ? 2u : 0u)) ||
      d->sh_bytes < sh_items * shst || d->color_bytes < (uint64_t)kTexWidth * th * colsz)
    return fail(ctx, GS_ERR_INVALID_ARGUMENT, "asset blob smaller than its format requires");
  const uint32_t chunk_count = (d->chunks && d->chunk_bytes) ? (uint32_t)(d->chunk_bytes / 64) : 0;
  GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GsAsset *as = new (std::nothrow) GsAsset();
  if (!as) return fail(ctx, GS_ERR_OUT_OF_MEMORY, "host allocation failed");
  as->ctx = ctx;
  auto up = [&](void **dst, const void *src, uint64_t bytes, uint64_t min_bytes = 0) -> cudaError_t {
    // +16 bytes of slack: the widest vector load of the last splat may read past a tightly sized blob
    const uint64_t alloc = (bytes > min_bytes ? bytes : min_bytes) + 16;
    cudaError_t e = cudaMalloc(dst, alloc);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync((uint8_t *)*dst + bytes, 0, alloc - bytes, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
  };
  // a u16 palette index can name any of 65536 entries whatever the palette's nominal size: back all of them (zeros)
  const uint64_t sh_min = clustered ? 65536ull * 96ull : 0ull;
  cudaError_t e = cudaSuccess;
  if ((e = up(&as->d_pos, d->pos, d->pos_bytes)) != cudaSuccess || (e = up(&as->d_other, d->other, d->other_bytes)) != cudaSuccess ||
      (e = up(&as->d_sh, d->sh, d->sh_bytes, sh_min)) != cudaSuccess || (e = up(&as->d_color, d->color, d->color_bytes)) != cudaSuccess ||
      (chunk_count && (e = up(&as->d_chunks, d->chunks, (uint64_t)chunk_count * 64)) != cudaSuccess) ||
      (e = cudaMalloc(&as->order, n * 4)) != cudaSuccess || (e = cudaMalloc(&as->keys, n * 4)) != cudaSuccess ||
      (e = cudaMalloc(&as->key_table, n * 4)) != cudaSuccess || (e = cudaMalloc(&as->draw, n * 48)) != cudaSuccess ||
      (e = cudaMalloc(&as->view, n * kViewStride + 16)) != cudaSuccess || (e = cudaMalloc(&as->rect, n * 4)) != cudaSuccess ||
      (e = cudaMalloc(&as->d_n, 4)) != cudaSuccess || (e = cudaMalloc(&as->block_bits, block_bits_words(d->splat_count) * 4 + 64)) != cudaSuccess) {
    gs_asset_destroy(as);
    return fail_cuda(ctx, e, "asset upload", __FILE__, __LINE__);
  }
  uint32_t n32 = d->splat_count;
  GS_CUDA_TRY(ctx, cudaMemcpyAsync(as->d_n, &n32, 4, cudaMemcpyHostToDevice, ctx->stream));
  as->av.n = d->splat_count;
  as->av.posFmt = d->pos_format; as->av.scaleFmt = d->scale_format; as->av.shFmt = d->sh_format; as->av.colFmt = d->color_format;
  as->av.chunkCount = chunk_count;
  as->av.pos = (const uint8_t *)as->d_pos; as->av.other = (const uint8_t *)as->d_other; as->av.sh = (const uint8_t *)as->d_sh;
  as->av.color = (const uint8_t *)as->d_color; as->av.chunks = (const Chunk *)as->d_chunks;
  launch_set_indices(as->order, as->av.n, ctx->stream);  // CSSetIndices
  ctx->launches += 1;
  GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // host blobs are only borrowed for this call
  *out = as;
  return GS_OK;
}

void gs_asset_destroy(GsAsset *as) {
  if (!as) return;
  if (as->ctx) { cudaSetDevice(as->ctx->device); cudaStreamSynchronize(as->ctx->stream); }
  cudaFree(as->d_pos); cudaFree(as->d_other); cudaFree(as->d_sh); cudaFree(as->d_color); cudaFree(as->d_chunks);
  cudaFree(as->order); cudaFree(as->keys); cudaFree(as->key_table); cudaFree(as->draw); cudaFree(as->view); cudaFree(as->rect); cudaFree(as->d_n); cudaFree(as->block_bits); cudaFree(as->zndc); cudaFree(as->slab_mask); cudaFree(as->order_tmp); cudaFree(as->order_alt); cudaFree(as->slab_group_bits);
  delete as;
}

int gs_asset_reset_order(GsAsset *as) {
  if (!as) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null asset");
  launch_set_indices(as->order, as->av.n, as->ctx->stream);
  as->ctx->launches += 1;
  GS_CUDA_TRY(as->ctx, cudaGetLastError());
  return GS_OK;
}

uint32_t gs_asset_splat_count(const GsAsset *as) { return as ? as->av.n : 0; }

int gs_sort(GsContext *ctx, GsAsset *as, const GsFrameParams *fp) {
  int rc = check_params(ctx, as, fp);
  if (rc) return rc;
  for (int e = 0; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
  FrameConsts fc = make_frame_consts(fp);
  return do_sort(ctx, as, fc);
}

int gs_calc_view(GsContext *ctx, GsAsset *as, const GsFrameParams *fp) {
  int rc = check_params(ctx, as, fp);
  if (rc) return rc;
  for (int e = 0; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
  FrameConsts fc = make_frame_consts(fp);
  return do_view(ctx, as, fp, fc, false, default_opts(), ctx->stream);
}

int gs_render(GsContext *ctx, GsAsset *as, const GsFrameParams *fp, const GsRenderOptions *opt_in, GsImage *rt) {
  int rc = check_params(ctx, as, fp);
  if (rc) return rc;
  if (!as->draw_valid || as->view_w != (uint32_t)fp->screen_w || as->view_h != (uint32_t)fp->screen_h)
    return fail(ctx, GS_ERR_NOT_READY, "gs_render needs gs_calc_view for the same screen size first");
  const uint32_t W = (uint32_t)fp->screen_w;
  uint32_t pitch = 0;
  GsRenderOptions opt = opt_in ? *opt_in : default_opts();
  FrameConsts fc = make_frame_consts(fp);
  if ((rc = check_options(ctx, fc, opt))) return rc;
  {
    const gs::Partition p = make_partition(opt);
    const uint32_t want[3] = {p.range ? p.t0 : p.index, p.range ? 0xFFFFFFFFu : p.count, p.range ? p.t1 : p.band};
    if (as->draw_part[1] > 1 && (as->draw_part[0] != want[0] || as->draw_part[1] != want[1] || as->draw_part[2] != want[2]))
      return fail(ctx, GS_ERR_NOT_READY, "the last gs_frame prepared draw records for another tile partition; run gs_calc_view");
  }
  const uint32_t H = opt.band_packed ? partition_own_bin_rows(opt, fc.binsY) * kBin : (uint32_t)fp->screen_h;
  if ((rc = image_ok(ctx, rt, W, H, &pitch))) return rc;
  for (int e = EV_BIN1; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
  if ((rc = bind_depth(ctx, fp, ctx->stream))) return rc;
  if (ctx->cur_depth && !as->zndc_valid) return fail(ctx, GS_ERR_NOT_READY, "a scene depth buffer needs the quad depths: run gs_calc_view with scene_depth set");
  rec(ctx, EV_VIEW1);
  if (rt->memory == GS_MEM_DEVICE) return do_render(ctx, as, fc, opt, rt->data, pitch, rt->format);
  const uint32_t tight = W * pix_bytes(rt->format);
  if ((rc = grow(ctx, &ctx->rt_scratch, &ctx->rt_bytes, (size_t)tight * H))) return rc;
  if ((rc = init_staging(ctx, opt, ctx->rt_scratch, tight, W, H, rt->format, rt, pitch))) return rc;
  if ((rc = do_render(ctx, as, fc, opt, ctx->rt_scratch, tight, rt->format))) return rc;
  GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(rt->data, pitch, ctx->rt_scratch, tight, tight, H, cudaMemcpyDeviceToHost, ctx->stream));
  return check_bin_overflow(ctx);
}

static int composite_impl(GsContext *ctx, const void *d_rt, uint32_t rt_pitch, uint32_t rt_fmt, GsImage *tgt, uint32_t W, uint32_t H) {
  GsNvtxRange nvtx("GaussianSplat.Compose");
  uint32_t tp = 0;
  int rc = image_ok(ctx, tgt, W, H, &tp);
  if (rc) return rc;
  if (tgt->memory == GS_MEM_DEVICE) {
    launch_composite(d_rt, rt_pitch, rt_fmt, tgt->data, tp, tgt->format, W, H, ctx->stream);
  } else {
    const uint32_t tight = W * pix_bytes(tgt->format);
    if ((rc = grow(ctx, &ctx->tgt_scratch, &ctx->tgt_bytes, (size_t)tight * H))) return rc;
    GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->tgt_scratch, tight, tgt->data, tp, tight, H, cudaMemcpyHostToDevice, ctx->stream));
    launch_composite(d_rt, rt_pitch, rt_fmt, ctx->tgt_scratch, tight, tgt->format, W, H, ctx->stream);
    GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(tgt->data, tp, ctx->tgt_scratch, tight, tight, H, cudaMemcpyDeviceToHost, ctx->stream));
  }
  rec(ctx, EV_COMP1);
  ctx->launches += 1;
  GS_CUDA_TRY(ctx, cudaGetLastError());
  if (tgt->memory != GS_MEM_DEVICE) GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

int gs_composite(GsContext *ctx, const GsImage *rt, GsImage *tgt) {
  if (!ctx || !rt || !tgt) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  uint32_t rp = 0;
  int rc = image_ok(ctx, rt, rt->width, rt->height, &rp);
  if (rc) return rc;
  const uint32_t W = rt->width, H = rt->height;
  ctx->ev_valid[EV_COMP1] = false;
  rec(ctx, EV_RASTER1);
  if (rt->memory == GS_MEM_DEVICE) return composite_impl(ctx, rt->data, rp, rt->format, tgt, W, H);
  const uint32_t tight = W * pix_bytes(rt->format);
  if ((rc = grow(ctx, &ctx->rt_scratch, &ctx->rt_bytes, (size_t)tight * H))) return rc;
  GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->rt_scratch, tight, rt->data, rp, tight, H, cudaMemcpyHostToDevice, ctx->stream));
  return composite_impl(ctx, ctx->rt_scratch, tight, rt->format, tgt, W, H);
}

int gs_frame(GsContext *ctx, GsAsset *as, const GsFrameParams *fp, const GsRenderOptions *opt_in, int do_sort_flag, GsImage *rt,
             GsImage *tgt) {
  int rc = check_params(ctx, as, fp);
  if (rc) return rc;
  if (!rt && !tgt) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "gs_frame needs rt and/or camera_target");
  const uint32_t W = (uint32_t)fp->screen_w;
  GsRenderOptions opt = opt_in ? *opt_in : default_opts();
  uint32_t rt_pitch = 0, rt_fmt = GS_PIX_RGBA16F;
  FrameConsts fc = make_frame_consts(fp);
  if ((rc = check_options(ctx, fc, opt))) return rc;
  const uint32_t H = opt.band_packed ? partition_own_bin_rows(opt, fc.binsY) * kBin : (uint32_t)fp->screen_h;
  if (opt.band_packed && tgt) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "band_packed output cannot be composited before the gather");
  if (rt) { if ((rc = image_ok(ctx, rt, W, H, &rt_pitch))) return rc; rt_fmt = rt->format; }
  for (int e = 0; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
  if (do_sort_flag && (rc = do_sort(ctx, as, fc))) return rc;
  if ((rc = do_view(ctx, as, fp, fc, true, opt, ctx->stream))) return rc;   // fused frame: colour of never-drawn splats is dead code
  void *d_rt;
  uint32_t d_pitch;
  const bool rt_dev = rt && rt->memory == GS_MEM_DEVICE;
  const bool async_rb = rt && !rt_dev && !tgt && (opt.flags & GS_FLAG_ASYNC_READBACK) != 0;
  int slot = 0;
  if (rt_dev) { d_rt = rt->data; d_pitch = rt_pitch; }
  else if (async_rb) {
    if ((rc = ensure_async_readback(ctx))) return rc;
    slot = ctx->rt_flip;
    ctx->rt_flip ^= 1;
    d_pitch = W * pix_bytes(rt_fmt);
    // the staging image of two frames ago: its copy must have left the device before this frame's raster overwrites it
    if (ctx->copy_pending[slot]) GS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copy_done[slot], 0));
    if (ctx->rt_async_bytes[slot] < (size_t)d_pitch * H && ctx->copy_pending[slot]) GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));  // about to be freed
    if ((rc = grow(ctx, &ctx->rt_async[slot], &ctx->rt_async_bytes[slot], (size_t)d_pitch * H))) return rc;
    d_rt = ctx->rt_async[slot];
    if ((rc = init_staging(ctx, opt, d_rt, d_pitch, W, H, rt_fmt, rt, rt_pitch))) return rc;
  } else {
    d_pitch = W * pix_bytes(rt_fmt);
    if ((rc = grow(ctx, &ctx->rt_scratch, &ctx->rt_bytes, (size_t)d_pitch * H))) return rc;
    d_rt = ctx->rt_scratch;
    if ((rc = init_staging(ctx, opt, d_rt, d_pitch, W, H, rt_fmt, rt, rt_pitch))) return rc;
  }
  if ((rc = bind_depth(ctx, fp, ctx->stream))) return rc;
  if ((rc = do_render(ctx, as, fc, opt, d_rt, d_pitch, rt_fmt))) return rc;
  bool synced = false;
  if (async_rb) {
    GS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_rt_ready[slot], ctx->stream));
    GS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_rt_ready[slot], 0));
    GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(rt->data, rt_pitch, d_rt, d_pitch, (size_t)W * pix_bytes(rt_fmt), H, cudaMemcpyDeviceToHost, ctx->copy_stream));
    GS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy_done[slot], ctx->copy_stream));
    ctx->copy_pending[slot] = true;
    return GS_OK;   // completion and the bin-list check: gs_sync
  }
  if (rt && !rt_dev) {
    GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(rt->data, rt_pitch, d_rt, d_pitch, (size_t)W * pix_bytes(rt_fmt), H, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (tgt) {
    if ((rc = composite_impl(ctx, d_rt, d_pitch, rt_fmt, tgt, W, H))) return rc;
    synced = tgt->memory != GS_MEM_DEVICE;
  }
  if ((rt && !rt_dev) || synced) return check_bin_overflow(ctx);
  return GS_OK;
}

int gs_unshuffle_bands(GsContext *ctx, const void *gathered, uint32_t parts, uint32_t band_rows, uint32_t rows_pp, uint32_t fmt,
                       GsImage *out) {
  if (!ctx || !gathered || !out || parts == 0) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  uint32_t pitch = 0;
  int rc = image_ok(ctx, out, out->width, out->height, &pitch);
  if (rc) return rc;
  if (out->format != fmt) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "gathered and output pixel formats differ");
  const uint32_t W = out->width, H = out->height;
  if (out->memory == GS_MEM_DEVICE) {
    launch_unshuffle(gathered, parts, band_rows, rows_pp, fmt, out->data, pitch, W, H, ctx->stream);
    ctx->launches += 1;
    GS_CUDA_TRY(ctx, cudaGetLastError());
    return GS_OK;
  }
  const uint32_t tight = W * pix_bytes(fmt);
  if ((rc = grow(ctx, &ctx->rt_scratch, &ctx->rt_bytes, (size_t)tight * H))) return rc;
  launch_unshuffle(gathered, parts, band_rows, rows_pp, fmt, ctx->rt_scratch, tight, W, H, ctx->stream);
  ctx->launches += 1;
  GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(out->data, pitch, ctx->rt_scratch, tight, tight, H, cudaMemcpyDeviceToHost, ctx->stream));
  GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

// ---- stand-alone sorter ---------------------------------------------------------------------------
int gs_sort_pairs_device(GsContext *ctx, uint32_t *d_keys, uint32_t *d_payload, uint32_t count) {
  if (!ctx || (count && (!d_keys || !d_payload))) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  if (count == 0) return GS_OK;
  if (count >= (1u << 30)) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "count must be < 2^30");
  int rc = ensure_sort_scratch(ctx, count);
  if (rc) return rc;
  GS_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scalar, &count, 4, cudaMemcpyHostToDevice, ctx->stream));
  for (int e = 0; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
  cudaEvent_t pe[5] = {ctx->ev[EV_SORT0], ctx->ev[EV_SORT1], ctx->ev[EV_SORT2], ctx->ev[EV_SORT3], ctx->ev[EV_SORT4]};
  rec(ctx, EV_BEGIN);
  launch_sort_pairs(d_keys, d_payload, ctx->d_scalar, count, 4, 8, false, ctx->sort, ctx->stream, ctx->timing ? pe : nullptr);
  if (ctx->timing) for (int e = EV_SORT0; e <= EV_SORT4; ++e) ctx->ev_valid[e] = true;
  ctx->launches += 5;
  GS_CUDA_TRY(ctx, cudaGetLastError());
  return GS_OK;
}

int gs_sort_pairs_host(GsContext *ctx, uint32_t *keys, uint32_t *payload, uint32_t count) {
  if (!ctx || (count && (!keys || !payload))) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  if (count == 0) return GS_OK;
  uint32_t *dk = nullptr, *dv = nullptr;
  GS_CUDA_TRY(ctx, cudaMalloc(&dk, (size_t)count * 4));
  cudaError_t e = cudaMalloc(&dv, (size_t)count * 4);
  if (e != cudaSuccess) { cudaFree(dk); return fail_cuda(ctx, e, "cudaMalloc", __FILE__, __LINE__); }
  cudaMemcpyAsync(dk, keys, (size_t)count * 4, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(dv, payload, (size_t)count * 4, cudaMemcpyHostToDevice, ctx->stream);
  int rc = gs_sort_pairs_device(ctx, dk, dv, count);
  if (rc == GS_OK) {
    cudaMemcpyAsync(keys, dk, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(payload, dv, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream);
    e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) rc = fail_cuda(ctx, e, "sort", __FILE__, __LINE__);
  }
  cudaFree(dk); cudaFree(dv);
  return rc;
}

// ---- test hooks -------------------------------------------------------------------------------------
static int readback(GsAsset *as, void *dst, const void *src, size_t bytes) {
  if (!as || !dst) return fail(as ? as->ctx : nullptr, GS_ERR_INVALID_ARGUMENT, "null argument");
  GsContext *ctx = as->ctx;
  GS_CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  GS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}
int gs_readback_order(GsAsset *as, uint32_t *dst) { return readback(as, dst, as ? as->order : nullptr, as ? (size_t)as->av.n * 4 : 0); }
int gs_readback_keys(GsAsset *as, uint32_t *dst) { return readback(as, dst, as ? as->keys : nullptr, as ? (size_t)as->av.n * 4 : 0); }
int gs_readback_view(GsAsset *as, void *dst) {
  if (as && !as->view_valid) return fail(as->ctx, GS_ERR_NOT_READY, "_SplatViewData is only materialised by gs_calc_view (gs_frame hands the draw its own records)");
  return readback(as, dst, as ? as->view : nullptr, as ? (size_t)as->av.n * kViewStride : 0);
}
int gs_export_splats(GsContext *ctx, GsAsset *as, const GsCutout *cutouts, uint32_t cutout_count, uint32_t bake_transform, void *dst) {
  if (!ctx || !as || !dst || (cutout_count && !cutouts)) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "null argument");
  if (as->ctx != ctx) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "asset belongs to another context");
  if (bake_transform) return fail(ctx, GS_ERR_UNSUPPORTED_FORMAT, "the baked export is a host pass over these records: call with bake_transform = 0, then gsa_bake_transform (gsplat_asset.h)");
  GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GsFrameParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.cutouts = cutouts; fp.cutout_count = cutout_count;
  int rc = upload_frame_inputs(ctx, as, &fp, ctx->stream);
  if (rc != GS_OK) return rc;
  float *d_out = nullptr;
  const size_t bytes = (size_t)as->av.n * 62 * sizeof(float);
  GS_CUDA_TRY(ctx, cudaMalloc(&d_out, bytes));
  launch_export_data(as->av, cutout_count, ctx->d_cutouts, d_out, ctx->stream);
  ctx->launches += 1;
  cudaError_t e = cudaMemcpyAsync(dst, d_out, bytes, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(d_out);
  if (e != cudaSuccess) return fail_cuda(ctx, e, "gs_export_splats", __FILE__, __LINE__);
  return GS_OK;
}

int gs_upload_order(GsAsset *as, const uint32_t *src) {
  if (!as || !src) return fail(as ? as->ctx : nullptr, GS_ERR_INVALID_ARGUMENT, "null argument");
  GS_CUDA_TRY(as->ctx, cudaMemcpyAsync(as->order, src, (size_t)as->av.n * 4, cudaMemcpyHostToDevice, as->ctx->stream));
  GS_CUDA_TRY(as->ctx, cudaStreamSynchronize(as->ctx->stream));
  return GS_OK;
}

// ---- Unity render-thread entry: IssuePluginEventAndData -> gs_frame / gs_sync ----
static void gs_unity_on_render_event(int event_id, void *data) {
  GsUnityFrameEvent *ev = static_cast<GsUnityFrameEvent *>(data);
  if (!ev) return;
  switch (event_id) {
    case GS_UNITY_EVENT_FRAME:
      ev->status = gs_frame(ev->ctx, ev->asset, &ev->params, &ev->options, ev->do_sort, ev->has_rt ? &ev->rt : nullptr,
                            ev->has_camera_target ? &ev->camera_target : nullptr);
      break;
    case GS_UNITY_EVENT_SYNC:
      ev->status = gs_sync(ev->ctx);
      break;
    default:
      ev->status = fail(ev->ctx, GS_ERR_INVALID_ARGUMENT, "unknown render event id");
  }
}
GsUnityRenderEventAndDataFunc gs_unity_get_render_event_func(void) { return gs_unity_on_render_event; }
uint32_t gs_unity_frame_event_size(void) { return (uint32_t)sizeof(GsUnityFrameEvent); }

void *gs_context_stream(GsContext *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
void *gs_asset_device_ptr(GsAsset *as, int which) {
  if (!as) return nullptr;
  return which == 0 ? (void *)as->order : which == 1 ? (void *)as->keys : which == 2 ? (void *)as->view : nullptr;
}

}  // extern "C"
