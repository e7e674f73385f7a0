// gs_kernels.cuh -- declarations shared between the .cu translation units.
#pragma once
#include "gs_common.cuh"

namespace gs {

constexpr uint32_t kRectEmpty = 0xFFFFFFFFu;  // bin rect sentinel (bin indices are < 255)

// Screen-space footprint of one splat, derived from its SplatViewData exactly the way the
// draw stage defines it (S/RenderGaussianSplats.shader:35-77; DESIGN.md "Raster rule").
struct SplatFootprint {
  float cx, cy;              // centre, pixels (D3D viewport: x right, y down)
  float i1x, i1y, i2x, i2y;  // axis / |axis|^2 : quad coordinates q = (dot(d,i1), dot(d,i2))
  float hx, hy;              // conservative half extents of the visible part, pixels
  float ca;                  // opacity (half -> float)
};

// `selected`: the splat's bit is set in _SplatSelectedBits, so the vertex shader hands the pixel shader col.a = -1 (:63-73)
// and the fragment's alpha comes from the gaussian alone (:87-101): the footprint is that of opacity 1, and the record
// carries ca = -1 as the marker.
__device__ __forceinline__ bool splat_footprint(float4 clip, float a1x, float a1y, float a2x, float a2y, float ca, float W,
                                                float H, SplatFootprint &fp, bool selected = false) {
  if (!(clip.w > 0.0f)) return false;  // behindCam -> NaN vertex -> primitive dropped (shader :41-45)
  if (!(ca >= 0.0f)) return false;     // CSCalcViewData never emits a negative opacity; NaN draws nothing
  const float ca_rec = selected ? -1.0f : ca;
  if (selected) ca = 1.0f;
  float ndx = __fdiv_rn(clip.x, clip.w), ndy = __fdiv_rn(clip.y, clip.w);
  float cx = fmaf(ndx, 0.5f, 0.5f) * W, cy = fmaf(ndy, -0.5f, 0.5f) * H;
  float ex = 2.0f * (fabsf(a1x) + fabsf(a2x)), ey = 2.0f * (fabsf(a1y) + fabsf(a2y));
  if (!(ex < 1.0e6f) || !(ey < 1.0e6f) || !(fabsf(cx) < 1.0e7f) || !(fabsf(cy) < 1.0e7f)) return false;
  // alpha = sat(exp(-r2) * ca) can only reach 1/255 if ca does (exp_neg(0) = 1.00000012)
  if (ca < 0.00392f) return false;
  float n1 = a1x * a1x + a1y * a1y, n2 = a2x * a2x + a2y * a2y;
  fp.cx = cx; fp.cy = cy;
  fp.i1x = __fdiv_rn(a1x, n1); fp.i1y = __fdiv_rn(a1y, n1);
  fp.i2x = __fdiv_rn(a2x, n2); fp.i2y = __fdiv_rn(a2y, n2);
  fp.ca = ca_rec;
  // visible part: the +-2 quad intersected with {r2 <= ln(255*ca)} (discard at alpha < 1/255)
  float r2 = fminf(__logf(ca * 255.0f) * 1.001f + 2.0e-3f, 8.0f);
  float rq = sqrtf(fmaxf(r2, 0.0f));
  float exE = rq * sqrtf(a1x * a1x + a2x * a2x), eyE = rq * sqrtf(a1y * a1y + a2y * a2y);
  fp.hx = fminf(ex, exE) * 1.0001f + 0.01f;
  fp.hy = fminf(ey, eyE) * 1.0001f + 0.01f;
  return true;
}

// ---- screen-tile partition helpers (multi-GPU, SURVEY 8e.1) ----------------------------------
// Two ways of giving one GPU a part of the screen:
//   interleaved (count > 1): 64-pixel bin rows r with (r / band) % count == index (GsRenderOptions.partition_*);
//   range       (range != 0): the contiguous 16-pixel raster-tile rows [t0, t1) (GsRenderOptions.row_begin/row_end) --
//                what the group path uses, with boundaries moved every frame by last frame's measured row costs.
struct Partition {
  uint32_t index, count, band;  // interleaved; count <= 1 and !range: everything is ours
  uint32_t range, t0, t1;       // range mode: own raster-tile rows
  __host__ __device__ uint32_t b0() const { return t0 / (kBin / kTile); }                          // first own bin row
  __host__ __device__ uint32_t b1() const { return (t1 + (kBin / kTile) - 1) / (kBin / kTile); }   // one past the last
  __host__ __device__ uint32_t own_rows_below(uint32_t y) const {  // # own bin rows in [0, y)
    if (range) { const uint32_t lo = b0(), hi = b1(); return y <= lo ? 0u : (y < hi ? y : hi) - lo; }
    if (count <= 1) return y;
    uint32_t cyc = band * count, q = y / cyc, r = y % cyc;
    uint32_t lo = index * band;
    uint32_t in = r > lo ? (r - lo < band ? r - lo : band) : 0u;
    return q * band + in;
  }
  __host__ __device__ bool owns(uint32_t y) const {
    if (range) return y >= b0() && y < b1();
    return count <= 1 || (y / band) % count == index;
  }
  __host__ __device__ uint32_t kth_own_row(uint32_t k) const {
    if (range) return b0() + k;
    if (count <= 1) return k;
    return ((k / band) * count + index) * band + (k % band);
  }
  // raster-tile rows: how many are ours, and the k-th of them
  __host__ __device__ uint32_t own_tile_rows(uint32_t binsY) const {
    return range ? t1 - t0 : own_rows_below(binsY) * (kBin / kTile);
  }
  __host__ __device__ uint32_t kth_own_tile_row(uint32_t k) const {
    if (range) return t0 + k;
    return kth_own_row(k / (kBin / kTile)) * (kBin / kTile) + (k % (kBin / kTile));
  }
};
inline Partition make_partition(const GsRenderOptions &o) {
  Partition p;
  p.count = o.partition_count;
  p.index = o.partition_count > 1 ? o.partition_index : 0;
  p.band = o.band_rows ? o.band_rows : 1;
  p.range = o.row_end > o.row_begin ? 1u : 0u;
  p.t0 = o.row_begin; p.t1 = o.row_end;
  if (p.range) { p.count = 0; p.index = 0; }
  return p;
}

// Pixel rows/cols whose centres can be touched -> inclusive rectangle of kBin-pixel bins packed x0|y0<<8|x1<<16|y1<<24.
// Range partitions clip the rows to their own pixel band first, so the rectangle holds own bin rows only.
__device__ __forceinline__ uint32_t footprint_tile_rect(const SplatFootprint &fp, const FrameConsts &fc, const Partition &part) {
  float x0 = fmaxf(ceilf(fp.cx - fp.hx - 0.5f), 0.0f), x1 = fminf(floorf(fp.cx + fp.hx - 0.5f), fc.screenW - 1.0f);
  float y0 = fmaxf(ceilf(fp.cy - fp.hy - 0.5f), 0.0f), y1 = fminf(floorf(fp.cy + fp.hy - 0.5f), fc.screenH - 1.0f);
  if (part.range) {
    y0 = fmaxf(y0, (float)(part.t0 * kTile));
    y1 = fminf(y1, (float)(part.t1 * kTile) - 1.0f);
  }
  if (!(x0 <= x1) || !(y0 <= y1)) return kRectEmpty;
  uint32_t tx0 = (uint32_t)x0 / kBin, tx1 = (uint32_t)x1 / kBin, ty0 = (uint32_t)y0 / kBin, ty1 = (uint32_t)y1 / kBin;
  return tx0 | (ty0 << 8) | (tx1 << 16) | (ty1 << 24);
}

__device__ __forceinline__ uint32_t rect_entries(uint32_t r, const Partition &p) {
  if (r == kRectEmpty) return 0;
  uint32_t x0 = r & 255u, y0 = (r >> 8) & 255u, x1 = (r >> 16) & 255u, y1 = r >> 24;
  uint32_t rows = p.own_rows_below(y1 + 1) - p.own_rows_below(y0);
  return rows * (x1 - x0 + 1);
}


// ---- launchers (each enqueues on `s`, returns nothing; errors surface via cudaGetLastError) ----
void launch_set_indices(uint32_t *order, uint32_t n, cudaStream_t s);
void launch_export_data(const AssetView &a, uint32_t cutoutCount, const GsCutout *cutouts, float *out, cudaStream_t s);  // gs_export.cu

// Key-range sharding of the depth sort over the GPUs of a group (SURVEY 8e.2); see k_calc_distances.
constexpr int kMaxSlabs = 16;
struct SlabArgs {
  uint32_t count, index;          // G slabs, and the one this GPU sorts
  const uint32_t *order_prev;     // last frame's draw order (replicated)
  uint32_t qpos[kMaxSlabs - 1];   // positions in order_prev whose splats' current keys are the G-1 splitters
  uint32_t *mask;                 // out: bit i = splat i belongs to slab `index`
  uint32_t *group_bits;           // out: bit j = some splat of [128 j, 128 j + 128) belongs to slab `index` (group_bits_words(n) words)
  uint32_t *info;                 // out (zeroed by the caller): [0, kMaxSlabs) ascending splitters, [kMaxSlabs, 2 kMaxSlabs) #{key >= splitter j}
};
void launch_calc_distances(const AssetView &a, const FrameConsts &fc, uint32_t *key_table, uint32_t *ghist, cudaStream_t s,
                           const SlabArgs *slabs = nullptr);
// block_bits: block_bits_words(n) words, bit j = some splat of [256 j, 256 j + 256) got a bin rectangle
inline size_t block_bits_words(uint32_t n) { return ((size_t)(n + 255) / 256 + 31) / 32 + 1; }
inline size_t group_bits_words(uint32_t n) { return ((size_t)(n + 127) / 128 + 31) / 32 + 1; }
void launch_calc_view(const AssetView &a, const FrameConsts &fc, const GsCutout *cutouts, const uint32_t *deleted, const uint32_t *selected, uint32_t *view,
                      uint32_t *rect, float4 *draw, uint32_t *block_bits, float *zndc /* per-splat quad depth, or nullptr */, bool cull_undrawable,
                      const Partition &part, cudaStream_t s);

// Radix sort (gs_sort.cu).  Scratch layout is owned by the caller (gs_api.cu).
struct SortScratch {
  uint32_t *alt_keys, *alt_vals;  // ping-pong buffers, >= capacity elements each
  uint32_t *ghist;                // 4*256 digit counts (one row per pass)
  uint32_t *lookback;             // passes * max_tiles * 256 status words
  uint32_t *tickets;              // passes counters
  uint32_t max_tiles;             // capacity / kSortTileItems rounded up
};
constexpr uint32_t kSortTileItems = 4096;  // 256 threads x 16 keys
size_t sort_lookback_words(uint32_t capacity, int passes);
// Stable ascending LSD sort of (key,val) pairs on bits [0, bits*passes), bits in {5..8}.  The count is read from d_count
// (device).  count_is_capacity: the host passes the exact count as `capacity` (exact grid); otherwise `capacity` only bounds
// the buffers and a persistent grid serves whatever d_count holds.
// ghist must already hold the per-pass digit counts when hist_ready, otherwise it is computed.
// After an even number of passes the result is back in keys/vals -- unless final_keys/final_vals name where the last pass
// writes.  key_table != nullptr: the input keys are key_table[vals[i]] (gathered inside pass 0; `keys` is then output only).
void launch_sort_pairs(uint32_t *keys, uint32_t *vals, const uint32_t *d_count, uint32_t capacity, int passes, int bits, bool hist_ready,
                       const SortScratch &sc, cudaStream_t s, cudaEvent_t *pass_events = nullptr, const uint32_t *key_table = nullptr,
                       bool count_is_capacity = true, uint32_t *final_keys = nullptr, uint32_t *final_vals = nullptr);
// (out_ids, out_keys) = (id, key_table[id]) of the ids of order[0..n) whose mask bit is set, order kept; *count_out = how many.
// group_bits (one bit per 128 ids, kept in shared memory) lets whole groups be skipped without reading their mask words.
// status: compact_status_words(n) words of scratch.
size_t compact_status_words(uint32_t n);
void launch_compact_order(const uint32_t *order, uint32_t n, const uint32_t *mask, const uint32_t *group_bits, const uint32_t *key_table,
                          uint32_t *out_ids, uint32_t *out_keys, uint32_t *status, uint32_t *count_out, cudaStream_t s);

// Binning + raster + composite (gs_raster.cu)
struct BinScratch {
  uint32_t *block_sums;    // [0] block ticket, [1..] look-back status of the fused count+scan+emit kernel
  uint32_t *entry_count;   // [0] = (tile,splat) entries clamped to capacity, [1] = overflow flag, [2] = unclamped total
  uint32_t *tile_keys, *tile_vals;  // capacity entries each
  uint32_t *bin_ranges;    // uint2 [start,end) per bin
  uint32_t *tile_cost, *tile_order;   // per raster tile: last frame's cost, this frame's launch order
  uint32_t capacity;
};
// returns the scratch view whose tile_keys / tile_vals hold the bin-sorted lists (launch_raster's input)
BinScratch launch_binning(const FrameConsts &fc, const GsRenderOptions &opt, uint32_t n, const uint32_t *order, const uint32_t *rect,
                          const uint32_t *block_bits, const BinScratch &bs, const SortScratch &sc, cudaStream_t s, int *launches);
// zndc / scene_depth: per-splat quad depth and the W x H depth buffer to test it against (both nullptr: no depth test)
void launch_raster(const FrameConsts &fc, const GsRenderOptions &opt, const float4 *draw, const BinScratch &bs, void *rt,
                   uint32_t rt_pitch_bytes, uint32_t rt_format, cudaStream_t s, const float *zndc = nullptr, const float *scene_depth = nullptr);
uint32_t partition_own_bin_rows(const GsRenderOptions &opt, uint32_t binsY);
uint32_t partition_own_tile_rows(const GsRenderOptions &opt, uint32_t binsY);
void launch_unshuffle(const void *gathered, uint32_t parts, uint32_t band, uint32_t rows_pp, uint32_t fmt, void *out, uint32_t pitch,
                      uint32_t W, uint32_t H, cudaStream_t s);
void launch_composite(const void *rt, uint32_t rt_pitch, uint32_t rt_format, void *target, uint32_t tgt_pitch, uint32_t tgt_format,
                      uint32_t W, uint32_t H, cudaStream_t s);

}  // namespace gs
