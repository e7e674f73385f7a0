// gs_raster.cu -- tile binning, front-to-back compositing and the final composite pass.
//
// The reference draws one instanced quad per splat through the hardware rasteriser with
// fixed-function blending `Blend OneMinusDstAlpha One` into an RGBA16F target
// (S/RenderGaussianSplats.shader:10-12,35-108; draw call R/GaussianSplatRenderer.cs:156-165).
// A CUDA device has neither rasteriser nor ROP, so the same pixels are produced by:
//   1. bin   -- walk the splats in sorted order; each emits one (bin id, splat id) entry per
//               64x64-pixel bin its visible footprint can touch (rect written by k_calc_view).
//               Bins are coarser than the 16x16 raster tiles on purpose: 2.5x fewer entries to
//               emit and sort, and the per-warp ballot cull below makes a foreign entry cost 1/32
//               of an evaluation.  Emission order == depth order, so one STABLE 16-bit radix sort
//               by tile id (2 onesweep passes) yields per-tile lists that are already in
//               draw order.  No 64-bit (tile|depth) re-sort of duplicated keys.
//   2. raster-- one CTA per tile, one pixel per thread.  The tile's list is consumed in
//               batches of 256 raster-ready records (written by k_calc_view) that land in shared
//               memory by cp.async, double buffered; every warp owns an 8x4 pixel block and
//               first culls a batch against that block with one ballot per 32 splats, so
//               small splats cost 1/32 of a pixel evaluation where they do not land.
//               Blending reproduces the ROP: dst = src*(1-dst.a) + dst, rounded to half after
//               every splat (GS_BLEND_FP16_ROP) -- or kept in float32 (GS_BLEND_FP32).
//   3. composite (S/GaussianComposite.shader:35-39).
#include <cstdlib>

#include "gs_kernels.cuh"

namespace gs {

constexpr int kBinItems = 8;                  // ranks per thread
constexpr int kBinBlock = 256 * kBinItems;    // ranks per block

// ---- 1. count + scan + emit in ONE pass ---------------------------------------------------------
// Blocks take their index by atomic ticket, publish their entry total with a LOCAL flag, resolve
// their exclusive offset by a warp-parallel decoupled look-back (32 predecessors per probe, gs_common.cuh), then
// emit (tile id, splat id) entries in depth order.
enum : uint32_t { kBinFlagLocal = kLbLocal, kBinFlagIncl = kLbIncl, kBinValMask = kLbMask };

__device__ __forceinline__ uint32_t entry_tile(uint32_t e, uint32_t r, const Partition &p, uint32_t tilesX) {
  const uint32_t x0 = r & 255u, y0 = (r >> 8) & 255u, x1 = (r >> 16) & 255u;
  const uint32_t w = x1 - x0 + 1;
  uint32_t krow = 0, col = e;
  if (e >= w) { krow = e / w; col = e - krow * w; }
  const uint32_t ty = p.count <= 1 ? y0 + krow : p.kth_own_row(p.own_rows_below(y0) + krow);
  return ty * tilesX + x0 + col;
}

__global__ void __launch_bounds__(256) k_bin_emit(const uint32_t *__restrict__ order, const uint32_t *__restrict__ rect,
                                                  const uint32_t *__restrict__ block_bits, uint32_t bits_words, uint32_t n, Partition part,
                                                  uint32_t tilesX, volatile uint32_t *status,
                                                  uint32_t *ticket, uint32_t capacity, uint32_t *__restrict__ keys,
                                                  uint32_t *__restrict__ vals, uint32_t *__restrict__ entry_count,
                                                  uint32_t *__restrict__ ghist, uint32_t digit_bits, bool two_pass) {
  extern __shared__ uint32_t s_bits[];   // the view kernel's block bitmap (bits_words words), or nothing when it is too large to hold
  __shared__ uint32_t s_w[8];
  __shared__ uint32_t s_block, s_excl;
  __shared__ uint32_t s_dh[512];   // digit histograms of the two sort passes over the tile ids we emit
  __shared__ uint2 s_items[kBinBlock];     // per warp: its drawable ranks, squeezed together in order
  __shared__ uint32_t s_pre[kBinBlock];
  const uint32_t nblocks = (n + kBinBlock - 1) / kBinBlock;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_block = atomicAdd(ticket, 1u);
  for (uint32_t i = threadIdx.x; i < bits_words; i += 256) s_bits[i] = __ldg(block_bits + i);
  s_dh[threadIdx.x] = 0; s_dh[threadIdx.x + 256] = 0;
  const uint32_t dmask = (1u << digit_bits) - 1u;
  __syncthreads();
  const uint32_t b = s_block;
  // warp-striped ranks: item i of lane l is rank wbase + i*32 + l (coalesced loads; the warp's 256 ranks are consecutive)
  const uint32_t wbase = b * kBinBlock + warp * (32 * kBinItems) + lane;
  uint32_t id[kBinItems], rc[kBinItems];
#pragma unroll
  for (int i = 0; i < kBinItems; ++i) {
    const uint32_t r = wbase + i * 32;
    id[i] = (r < n) ? __ldg(order + r) : 0xFFFFFFFFu;
  }
  // the rectangle of a splat is a random 4-byte gather; the view kernel's per-block bits (in shared memory) say where there
  // is nothing to fetch
#pragma unroll
  for (int i = 0; i < kBinItems; ++i) {
    rc[i] = kRectEmpty;
    if (id[i] != 0xFFFFFFFFu) {
      const uint32_t bw = bits_words ? s_bits[id[i] >> 13] : __ldg(block_bits + (id[i] >> 13));
      if ((bw >> ((id[i] >> 8) & 31u)) & 1u) rc[i] = __ldg(rect + id[i]);
    }
  }
  // Most ranks have nothing to emit (70 % of cfg2's splats draw nothing; in a group of G only 1/G of the rest is ours).
  // The warp first squeezes its drawable ranks, in order, into shared memory, and everything below -- entry counts, prefix
  // scans, the emission loop -- runs over those K <= 256 items in chunks of 32 instead of over 8 sparse slots.
  uint2 *w_items = s_items + warp * (32 * kBinItems);     // (splat id, rect)
  uint32_t *w_pre = s_pre + warp * (32 * kBinItems);      // exclusive prefix of the item's entries inside its chunk
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t K = 0;
#pragma unroll
  for (int i = 0; i < kBinItems; ++i) {
    const bool has = rect_entries(rc[i], part) != 0;
    const uint32_t bal = __ballot_sync(0xffffffffu, has);
    if (has) w_items[K + __popc(bal & lt)] = make_uint2(id[i], rc[i]);
    K += __popc(bal);
  }
  __syncwarp();
  const uint32_t nchunks = (K + 31) >> 5;
  uint32_t ctot[kBinItems];   // entries of chunk j (warp-uniform)
  uint32_t wsum = 0;
#pragma unroll
  for (int j = 0; j < kBinItems; ++j) {
    ctot[j] = 0;
    if ((uint32_t)j < nchunks) {
      const uint32_t k = j * 32 + lane;
      const uint32_t c = k < K ? rect_entries(w_items[k].y, part) : 0u;
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
      }
      w_pre[k] = inc - c;
      ctot[j] = __shfl_sync(0xffffffffu, inc, 31);
      wsum += ctot[j];
    }
  }
  if (lane == 0) s_w[warp] = wsum;
  __syncthreads();
  uint32_t woff = 0, total = 0;
#pragma unroll
  for (uint32_t w = 0; w < 8; ++w) {
    const uint32_t c = s_w[w];
    if (w < warp) woff += c;
    total += c;
  }
  if (warp == 0) {
    if (lane == 0) status[b] = (b == 0 ? kBinFlagIncl : kBinFlagLocal) | total;
    uint32_t excl = 0;
    if (b > 0) {
      excl = lookback_exclusive(status, b);
      // prefixes saturate instead of wrapping at 2^30: a saturated total is > any capacity, so it is reported as overflow
      if (lane == 0) status[b] = kBinFlagIncl | min(excl + total, (uint32_t)kBinValMask);
    }
    if (lane == 0) {
      s_excl = excl;
      if (b == nblocks - 1) {
        const uint32_t all = min(excl + total, (uint32_t)kBinValMask);
        entry_count[1] = all > capacity ? 1u : 0u;   // overflow: lists are truncated, the API reports it
        entry_count[0] = all > capacity ? capacity : all;
        entry_count[2] = all;
      }
    }
  }
  __syncthreads();
  // Emission is warp-cooperative: the 32 items of a chunk own one contiguous output range; lane x of the warp writes entry x
  // of that range (owner found by a 5-step shuffle search over the lanes' prefix sums), so every store is a full coalesced
  // line regardless of how many bins each splat touches.
  uint32_t off = s_excl + woff;
#pragma unroll
  for (int j = 0; j < kBinItems; ++j) {
    if ((uint32_t)j >= nchunks) break;
    const uint32_t k = j * 32 + lane;
    const uint2 it = k < K ? w_items[k] : make_uint2(0xFFFFFFFFu, kRectEmpty);
    const uint32_t pre = k < K ? w_pre[k] : 0xFFFFFFFFu;   // lanes past the end never own an entry
    const uint32_t T = ctot[j];
    for (uint32_t e0 = 0; e0 < T; e0 += 32) {
      const uint32_t x = e0 + lane;
      // owner = last lane whose exclusive prefix is <= x
      uint32_t lo = 0, hi = 31;
#pragma unroll
      for (int step = 0; step < 5; ++step) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        const uint32_t pm = __shfl_sync(0xffffffffu, pre, mid);
        if (pm <= x) lo = mid; else hi = mid - 1;
      }
      const uint32_t opre = __shfl_sync(0xffffffffu, pre, lo);
      const uint32_t orc = __shfl_sync(0xffffffffu, it.y, lo);
      const uint32_t oid = __shfl_sync(0xffffffffu, it.x, lo);
      const uint32_t o = off + x;
      if (x < T && o < capacity) {
        const uint32_t tile = entry_tile(x - opre, orc, part, tilesX);
        keys[o] = tile;
        vals[o] = oid;
        atomicAdd(&s_dh[tile & dmask], 1u);
        if (two_pass) atomicAdd(&s_dh[256 + ((tile >> digit_bits) & dmask)], 1u);
      }
    }
    off += T;
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < 512; i += 256) {
    const uint32_t c = s_dh[i];
    if (c) atomicAdd(&ghist[i], c);
  }
}

// digit width and pass count of the stable sort by bin id: one pass while the bin count fits a digit (<= 256 bins, e.g.
// 1200x797 = 19x13), else two passes of the narrowest digit that covers it
static void bin_sort_plan(uint32_t bins, int *bits, int *passes) {
  if (bins <= 256u) { *passes = 1; *bits = bins <= 32u ? 5 : bins <= 64u ? 6 : bins <= 128u ? 7 : 8; return; }
  *passes = 2;
  *bits = bins <= 1024u ? 5 : bins <= 4096u ? 6 : bins <= 16384u ? 7 : 8;
}

BinScratch launch_binning(const FrameConsts &fc, const GsRenderOptions &opt, uint32_t n, const uint32_t *order, const uint32_t *rect,
                          const uint32_t *block_bits, const BinScratch &bs, const SortScratch &sc, cudaStream_t s, int *launches) {
  const Partition part = make_partition(opt);
  const uint32_t tiles = fc.binsX * fc.binsY;
  if (launches) *launches = 0;
  if (!n) { cudaMemsetAsync(bs.entry_count, 0, 16, s); return bs; }
  const uint32_t nblocks = (n + kBinBlock - 1) / kBinBlock;
  cudaMemsetAsync(bs.block_sums, 0, ((size_t)nblocks + 1) * sizeof(uint32_t), s);   // [0] ticket, [1..] look-back status
  int bits, passes;
  bin_sort_plan(tiles, &bits, &passes);
  if (launches) *launches = 2 + passes;   // bin_emit, look-back clear, sort passes
  cudaMemsetAsync(sc.ghist, 0, 4 * 256 * sizeof(uint32_t), s);
  uint32_t words = (uint32_t)block_bits_words(n);
  static int bits_global = -1;   // GS_WALK_BITS_GLOBAL=1 forces the large-asset path (bitmap read through L1) for tests
  if (bits_global < 0) { const char *e = getenv("GS_WALK_BITS_GLOBAL"); bits_global = (e && e[0] == '1') ? 1 : 0; }
  if (bits_global) words = 0;
  if (words * 4u > 16u * 1024u) words = 0;   // beside the kernel's 28 KB of static shared memory only 20 KB of the default 48 remain:
                                              // a larger bitmap (> 33 M splats) is read through L1 instead
  k_bin_emit<<<nblocks, 256, words * 4u, s>>>(order, rect, block_bits, words, n, part, fc.binsX, bs.block_sums + 1, bs.block_sums, bs.capacity,
                                     bs.tile_keys, bs.tile_vals, bs.entry_count, sc.ghist, (uint32_t)bits, passes == 2);
  // the entry count lives on the device: a persistent grid sorts whatever it is (no capacity-sized grid or memset)
  launch_sort_pairs(bs.tile_keys, bs.tile_vals, bs.entry_count, bs.capacity, passes, bits, true, sc, s, nullptr, nullptr,
                    /*count_is_capacity=*/false);
  BinScratch sorted = bs;   // an odd number of passes leaves the sorted lists in the sorter's ping-pong buffers
  if (passes & 1) { sorted.tile_keys = sc.alt_keys; sorted.tile_vals = sc.alt_vals; }
  return sorted;
}

// ---- 2. raster ---------------------------------------------------------------------------------
__device__ __forceinline__ float round_half(float v) { return __half2float(__float2half_rn(v)); }

// first index in sorted keys[0,m) whose key is >= target; all 32 lanes of a warp cooperate
__device__ __forceinline__ uint32_t lower_bound32(const uint32_t *__restrict__ keys, uint32_t m, uint32_t target, uint32_t lane) {
  uint32_t lo = 0, hi = m;
  while (hi - lo > 32) {
    const uint32_t len = hi - lo;
    const uint32_t p = lo + (uint32_t)(((uint64_t)len * (lane + 1)) / 33);   // lo < p < hi, increasing with lane
    const uint32_t below = __ballot_sync(0xffffffffu, __ldg(keys + p) < target);
    const int c = __popc(below);                                             // predicate is monotone over lanes
    const uint32_t p_lo = __shfl_sync(0xffffffffu, p, c > 0 ? c - 1 : 0), p_hi = __shfl_sync(0xffffffffu, p, c < 32 ? c : 31);
    if (c > 0) lo = p_lo + 1;
    if (c < 32) hi = p_hi;
  }
  const uint32_t p = lo + lane;
  const uint32_t below = __ballot_sync(0xffffffffu, p < hi && __ldg(keys + p) < target);
  return lo + __popc(below);
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// one warp per bin: [start,end) of the bin's entries in the sorted list, by two 32-ary searches (5 probes for 10M entries)
__global__ void __launch_bounds__(256) k_bin_ranges(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ entry_count,
                                                    uint32_t bins, uint2 *__restrict__ ranges) {
  const uint32_t bin = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (bin >= bins) return;
  const uint32_t m = __ldg(entry_count);
  const uint32_t a = lower_bound32(keys, m, bin, lane), b = lower_bound32(keys, m, bin + 1, lane);
  if (lane == 0) ranges[bin] = make_uint2(a, b);
}

// Launch order of the raster tiles: longest-processing-time first, from the cost each tile measured last frame
// (counting sort over 64 log-scale buckets, one CTA).  Pixels do not depend on the order; only the tail does.
__global__ void __launch_bounds__(1024) k_tile_order(const uint32_t *__restrict__ cost, uint32_t ntiles, uint32_t ntx, Partition part,
                                                     uint32_t *__restrict__ order) {
  // `cost` is indexed by the tile's id in the whole image (ty * ntx + tx) so that a moving partition keeps its history;
  // `order` receives the ids of OUR ntiles tiles (own tile row k = kth_own_tile_row(k)), most expensive first
  __shared__ uint32_t s_hist[64], s_base[64];
  __shared__ uint32_t s_any;
  if (threadIdx.x < 64) s_hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_any = 0;
  __syncthreads();
  auto bucket = [](uint32_t c) -> uint32_t {   // 0 for cost 0, else 2*log2 resolution, descending order wanted
    if (c == 0) return 0u;
    const uint32_t l = 31u - (uint32_t)__clz(c);
    const uint32_t half = l ? ((c >> (l - 1)) & 1u) : 0u;
    return min(63u, 1u + 2u * l + half);
  };
  auto global_id = [&](uint32_t t) -> uint32_t { const uint32_t k = t / ntx; return part.kth_own_tile_row(k) * ntx + (t - k * ntx); };
  for (uint32_t t = threadIdx.x; t < ntiles; t += 1024) {
    const uint32_t c = cost[global_id(t)];
    if (c) s_any = 1;
    atomicAdd(&s_hist[63u - bucket(c)], 1u);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int b = 0; b < 64; ++b) { s_base[b] = run; run += s_hist[b]; }
  }
  __syncthreads();
  if (!s_any) {   // no history (first frame / new resolution): a stride permutation spreads spatial clusters
    for (uint32_t t = threadIdx.x; t < ntiles; t += 1024) order[t] = global_id((ntiles % 1031u) ? (uint32_t)(((uint64_t)t * 1031u) % ntiles) : t);
    return;
  }
  for (uint32_t t = threadIdx.x; t < ntiles; t += 1024) {
    const uint32_t gid = global_id(t);
    order[atomicAdd(&s_base[63u - bucket(cost[gid])], 1u)] = gid;
  }
}

// per raster-tile row: the sum of its tiles' costs (what the group path balances its row ranges with)
__global__ void __launch_bounds__(256) k_row_costs(const uint32_t *__restrict__ cost, uint32_t ntx, uint32_t t0, uint32_t t1,
                                                   uint32_t *__restrict__ row_cost) {
  const uint32_t row = t0 + blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= t1) return;
  uint32_t acc = 0;
  for (uint32_t x = lane; x < ntx; x += 32) acc += cost[row * ntx + x];
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) row_cost[row] = acc;
}
void launch_row_costs(const uint32_t *cost, uint32_t ntx, uint32_t t0, uint32_t t1, uint32_t *row_cost, cudaStream_t s) {
  if (t1 > t0) k_row_costs<<<(t1 - t0 + 7) / 8, 256, 0, s>>>(cost, ntx, t0, t1, row_cost);
}

// SEL ("extras"): a separate instantiation for frames with an edit selection and / or a scene depth buffer bound, so that
// ordinary frames pay nothing.  Selected splats (records with opacity -1) take the pixel shader's other branch
// (S/RenderGaussianSplats.shader:87-101); with `scene_depth` every fragment is depth-tested like the pass's ZTest LEqual
// (reversed Z: quad depth >= stored depth), the per-splat quad depths being staged beside the records.
template <bool FP16_ROP, int OUT_FMT, bool SEL>
__global__ void __launch_bounds__(256)
k_raster(FrameConsts fc, Partition part, const float4 *__restrict__ draw, const uint2 *__restrict__ bin_ranges,
         const uint32_t *__restrict__ tile_vals, const uint32_t *__restrict__ tile_order, uint32_t *__restrict__ tile_cost, uint32_t ntx,
         uint8_t *__restrict__ rt, uint32_t pitch, uint32_t band_packed, uint32_t load_rt,
         const float *__restrict__ zndc, const float *__restrict__ scene_depth) {
  uint32_t st_batches = 0, st_eval = 0;   // this warp's work, for the tile's cost below
  // two staging buffers of 256 raster records (3 x float4 each), planar [buf][plane][entry]: batch k+1 lands asynchronously
  // while batch k is composited
  __shared__ __align__(128) float4 s_rec[2][3][256];  // plane 0: cx, cy, i1x, i1y   1: i2x, i2y, opacity, hx   2: r, g, b, hy
  __shared__ float s_z[SEL ? 2 : 1][SEL ? 256 : 1];   // quad depths of the staged batch (depth test only)
  const bool depth_test = SEL && scene_depth != nullptr;

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // 1-D grid over raster tiles: tile = (16-pixel column, R * own 64-pixel bin row + tile row inside that bin row)
  constexpr uint32_t R = kBin / kTile;   // raster tiles per bin edge
  // launch order != raster order: CTA i takes tile order[i] (k_tile_order: most expensive first, by last frame's cost),
  // so the expensive tiles start early instead of forming the tail
  const uint32_t lin = __ldg(tile_order + blockIdx.x);   // tile id in the whole image: ty * ntx + tx
  const uint32_t ty = lin / ntx;
  const uint32_t tx = lin - ty * ntx, brow = ty / R;
  if (ty * kTile >= (uint32_t)fc.screenH) { if (threadIdx.x == 0) tile_cost[lin] = 0; return; }
  __shared__ uint32_t s_cost;
  if (threadIdx.x == 0) s_cost = 0;
  // [start,end) of this tile's bin in the bin-sorted entry list (k_bin_ranges); R*R tiles share one list
  const uint2 range = __ldg(bin_ranges + brow * fc.binsX + (tx / R));
  const uint32_t bx = tx * kTile + (warp & 1) * 8, by = ty * kTile + (warp >> 1) * 4;
  const uint32_t px = bx + (lane & 7), py = by + (lane >> 3);
  const float pxc = (float)px + 0.5f, pyc = (float)py + 0.5f;
  const float bcx = (float)bx + 4.0f, bcy = (float)by + 2.0f;
  const bool in_image = px < (uint32_t)fc.screenW && py < (uint32_t)fc.screenH;

  float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;  // ClearRenderTarget(0,0,0,0), R/GaussianSplatRenderer.cs:196
  // the scene's depth at this pixel (depth target bound at R/GaussianSplatRenderer.cs:195; ZTest LEqual, ZWrite Off)
  float zscene = 0.0f;
  if (SEL && depth_test && in_image) zscene = __ldg(scene_depth + (size_t)py * (uint32_t)fc.screenW + px);
  // where this pixel lives in the target (band-packed: own bin row k of an interleaved partition -> rows [64k, 64k+64))
  const uint32_t out_row = band_packed ? part.own_rows_below(brow) * kBin + (py - brow * kBin) : py;
  if (load_rt && in_image) {
    // GS_FLAG_LOAD_RT: the target was cleared once and earlier renderers of this camera already drew into it
    // (R/GaussianSplatRenderer.cs:111-168 loops the active splat objects over ONE _GaussianSplatRT); blend under what is there
    const uint8_t *row = rt + (size_t)out_row * pitch;
    if (OUT_FMT == GS_PIX_RGBA16F) {
      const uint2 v = reinterpret_cast<const uint2 *>(row)[px];
      d0 = f16lo(v.x); d1 = f16hi(v.x); d2 = f16lo(v.y); d3 = f16hi(v.y);
    } else {
      const float4 v = reinterpret_cast<const float4 *>(row)[px];
      d0 = v.x; d1 = v.y; d2 = v.z; d3 = v.w;
    }
  }

  // three-deep pipeline: splat ids of batch k+2 (register) -> records of batch k+1 (cp.async in flight) -> batch k (composited)
  auto load_id = [&](uint32_t e) -> uint32_t { return e < range.y ? __ldg(tile_vals + e) : 0xFFFFFFFFu; };
  auto stage = [&](int buf, uint32_t id) {
    if (id != 0xFFFFFFFFu) {
      const float4 *src = draw + (size_t)id * 3;
      cp_async16(&s_rec[buf][0][tid], src);
      cp_async16(&s_rec[buf][1][tid], src + 1);
      cp_async16(&s_rec[buf][2][tid], src + 2);
      if (SEL && depth_test) cp_async4(&s_z[SEL ? buf : 0][SEL ? tid : 0], zndc + id);
    }
    cp_async_commit();
  };
  uint32_t id_next = load_id(range.x + tid);
  stage(0, id_next);
  id_next = load_id(range.x + 256 + tid);

  int buf = 0;
  for (uint32_t base = range.x; base < range.y; base += 256, buf ^= 1) {
    stage(buf ^ 1, id_next);              // batch k+1 -> other buffer (free since the barrier that ended batch k-1)
    id_next = load_id(base + 512 + tid);  // ids of batch k+2
    cp_async_wait<1>();                   // batch k has landed (this thread's copies) ...
    __syncthreads();                      // ... and everyone else's
    const float4 *s_a = s_rec[buf][0], *s_b = s_rec[buf][1], *s_c = s_rec[buf][2];

    const uint32_t cnt = min(256u, range.y - base);
    ++st_batches;
    for (uint32_t c0 = 0; c0 < cnt; c0 += 32) {
      // a warp whose 32 pixels all reached dst.a == 1 ignores everything behind exactly: skip the batch remainder
      if (__all_sync(0xffffffffu, d3 == 1.0f || !in_image)) break;
      // one ballot culls 32 splats against this warp's 8x4 pixel block
      const uint32_t e = c0 + lane;
      bool hit = false;
      if (e < cnt) {
        const float4 A = s_a[e];
        const float hx = s_b[e].w, hy = s_c[e].w;
        hit = (fabsf(A.x - bcx) <= hx + 3.5f) && (fabsf(A.y - bcy) <= hy + 1.5f);
      }
      uint32_t mask = __ballot_sync(0xffffffffu, hit);
      while (mask) {
        const uint32_t j = c0 + __ffs(mask) - 1;
        mask &= mask - 1;
        const float4 A = s_a[j], B = s_b[j];
        const float dx = pxc - A.x, dy = A.y - pyc;  // pixel y grows down, NDC y up
        const float qa = fmaf(dy, A.w, dx * A.z), qb = fmaf(dy, B.y, dx * B.x);
        const bool inside = (fabsf(qa) <= 2.0f) && (fabsf(qb) <= 2.0f);  // quad corners at +-2 (:54-55)
        if (!__any_sync(0xffffffffu, inside)) continue;
        ++st_eval;
        const float power = -fmaf(qb, qb, qa * qa);                       // -dot(i.pos, i.pos) (:81)
        float alpha = exp_neg(power);                                     // half alpha = exp(power) (:82)
        bool tint = false, outline = false;
        if (SEL && B.z < 0.0f) {                                          // "selected": outline, more opacity, magenta tint (:87-101)
          tint = true;
          if (alpha > 7.0f / 255.0f) {
            if (alpha < 10.0f / 255.0f) { alpha = 1.0f; outline = true; }
            alpha = __saturatef(alpha + 0.3f);
          }
        } else {
          alpha = __saturatef(alpha * B.z);                               // :83-86 (saturate: NaN -> 0, one instruction)
        }
        bool pass = inside && alpha >= 0.003921569f;                      // discard below 1/255 (:103-104)
        if (SEL && depth_test) pass = pass && (s_z[SEL ? buf : 0][SEL ? j : 0] >= zscene);   // ZTest LEqual, reversed Z
        if (pass) {
          float4 C = s_c[j];
          if (SEL && tint) {
            if (outline) { C.x = 1.0f; C.y = 0.0f; C.z = 1.0f; }
            C.x = lerpf(C.x, 1.0f, 0.5f); C.y = lerpf(C.y, 0.0f, 0.5f); C.z = lerpf(C.z, 1.0f, 0.5f);
          }
          const float om = 1.0f - d3;                                     // Blend OneMinusDstAlpha One (:11)
          float n0 = fmaf(C.x * alpha, om, d0), n1 = fmaf(C.y * alpha, om, d1), n2 = fmaf(C.z * alpha, om, d2),
                n3 = fmaf(alpha, om, d3);
          if (FP16_ROP) {  // the ROP stores half: round every channel (two packed f32x2 -> f16x2 conversions)
            const float2 lo = __half22float2(__floats2half2_rn(n0, n1)), hi = __half22float2(__floats2half2_rn(n2, n3));
            n0 = lo.x; n1 = lo.y; n2 = hi.x; n3 = hi.y;
          }
          d0 = n0; d1 = n1; d2 = n2; d3 = n3;
        }
      }
    }
    // a pixel whose dst.a == 1 ignores every later splat exactly (src*0 + dst): safe early out.  The barrier also
    // frees this batch's buffer for the copies issued at the top of the next-but-one iteration.
    if (__syncthreads_and(d3 == 1.0f || !in_image)) break;
  }
  cp_async_wait<0>();
  // this tile's cost for next frame's launch order: the slowest warp's work (evaluations dominate, culls and batches add)
  if (lane == 0) atomicMax(&s_cost, st_eval * 4 + st_batches * 16 + 1);
  __syncthreads();
  if (threadIdx.x == 0) tile_cost[lin] = s_cost;
  if (in_image) {
    uint8_t *row = rt + (size_t)out_row * pitch;
    if (OUT_FMT == GS_PIX_RGBA16F) {
      uint2 o;
      o.x = f32tof16(d0) | (f32tof16(d1) << 16);
      o.y = f32tof16(d2) | (f32tof16(d3) << 16);
      reinterpret_cast<uint2 *>(row)[px] = o;
    } else {
      reinterpret_cast<float4 *>(row)[px] = make_float4(d0, d1, d2, d3);
    }
  }
}

void launch_raster(const FrameConsts &fc, const GsRenderOptions &opt, const float4 *draw, const BinScratch &bs, void *rt,
                   uint32_t rt_pitch_bytes, uint32_t rt_format, cudaStream_t s, const float *zndc, const float *scene_depth) {
  const Partition part = make_partition(opt);
  const uint32_t rows = part.own_tile_rows(fc.binsY);
  if (!rows || !fc.binsX) return;
  const uint32_t ntx = ((uint32_t)fc.screenW + kTile - 1) / kTile, ntiles = ntx * rows;
  const uint32_t grid = ntiles;
  k_tile_order<<<1, 1024, 0, s>>>(bs.tile_cost, ntiles, ntx, part, bs.tile_order);
  const bool rop = opt.blend_mode == GS_BLEND_FP16_ROP;
  uint8_t *out = reinterpret_cast<uint8_t *>(rt);
  const uint32_t bins = fc.binsX * fc.binsY;
  uint2 *ranges = reinterpret_cast<uint2 *>(bs.bin_ranges);
  const uint32_t packed = part.range ? 0u : opt.band_packed, load = (opt.flags & GS_FLAG_LOAD_RT) ? 1u : 0u;
  k_bin_ranges<<<(bins + 7) / 8, 256, 0, s>>>(bs.tile_keys, bs.entry_count, bins, ranges);
#define GS_LAUNCH_RASTER(ROP, FMT)                                                                                              \
  do {                                                                                                                         \
    if (fc.selValid || scene_depth) k_raster<ROP, FMT, true><<<grid, 256, 0, s>>>(fc, part, draw, ranges, bs.tile_vals, bs.tile_order, bs.tile_cost, ntx, out, rt_pitch_bytes, packed, load, zndc, scene_depth); \
    else k_raster<ROP, FMT, false><<<grid, 256, 0, s>>>(fc, part, draw, ranges, bs.tile_vals, bs.tile_order, bs.tile_cost, ntx, out, rt_pitch_bytes, packed, load, nullptr, nullptr); \
  } while (0)
  if (rt_format == GS_PIX_RGBA16F) {
    if (rop) GS_LAUNCH_RASTER(true, GS_PIX_RGBA16F); else GS_LAUNCH_RASTER(false, GS_PIX_RGBA16F);
  } else {
    if (rop) GS_LAUNCH_RASTER(true, GS_PIX_RGBA32F); else GS_LAUNCH_RASTER(false, GS_PIX_RGBA32F);
  }
#undef GS_LAUNCH_RASTER
}

uint32_t partition_own_bin_rows(const GsRenderOptions &opt, uint32_t binsY) { return make_partition(opt).own_rows_below(binsY); }
uint32_t partition_own_tile_rows(const GsRenderOptions &opt, uint32_t binsY) { return make_partition(opt).own_tile_rows(binsY); }

// ---- 2b. multi-GPU epilogue: gathered band-packed targets -> one image ---------------------------
__global__ void __launch_bounds__(256) k_unshuffle(const uint8_t *__restrict__ gathered, Partition part, uint32_t rows_pp, uint32_t px_bytes,
                                                   uint8_t *__restrict__ out, uint32_t pitch, uint32_t W, uint32_t H) {
  const uint32_t x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  const uint32_t ty = y / kBin;
  Partition owner = part;
  owner.index = part.count > 1 ? (ty / part.band) % part.count : 0;
  const uint32_t k = owner.own_rows_below(ty);
  const uint8_t *src = gathered + ((size_t)owner.index * rows_pp + (size_t)k * kBin + (y - ty * kBin)) * W * px_bytes;
  if (px_bytes == 8) reinterpret_cast<uint2 *>(out + (size_t)y * pitch)[x] = reinterpret_cast<const uint2 *>(src)[x];
  else reinterpret_cast<uint4 *>(out + (size_t)y * pitch)[x] = reinterpret_cast<const uint4 *>(src)[x];
}

void launch_unshuffle(const void *gathered, uint32_t parts, uint32_t band, uint32_t rows_pp, uint32_t fmt, void *out, uint32_t pitch,
                      uint32_t W, uint32_t H, cudaStream_t s) {
  Partition p{};
  p.count = parts; p.index = 0; p.band = band ? band : 1;
  dim3 grid((W + 31) / 32, (H + 7) / 8);
  k_unshuffle<<<grid, 256, 0, s>>>(reinterpret_cast<const uint8_t *>(gathered), p, rows_pp, fmt == GS_PIX_RGBA16F ? 8u : 16u,
                                   reinterpret_cast<uint8_t *>(out), pitch, W, H);
}

// ---- 3. composite (S/GaussianComposite.shader:35-39, Blend SrcAlpha OneMinusSrcAlpha :11) ------
__device__ __forceinline__ float gamma_to_linear(float x) {  // UnityCG.cginc GammaToLinearSpace (not vendored)
  return x * fmaf(x, fmaf(x, 0.305306011f, 0.682171111f), 0.012522878f);
}

__global__ void __launch_bounds__(256) k_composite(const uint8_t *__restrict__ rt, uint32_t rt_pitch, uint32_t rt_fmt,
                                                   uint8_t *__restrict__ tgt, uint32_t tgt_pitch, uint32_t tgt_fmt, uint32_t W,
                                                   uint32_t H) {
  const uint32_t x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  float4 c;
  if (rt_fmt == GS_PIX_RGBA16F) {
    uint2 v = reinterpret_cast<const uint2 *>(rt + (size_t)y * rt_pitch)[x];
    c = make_float4(f16lo(v.x), f16hi(v.x), f16lo(v.y), f16hi(v.y));
  } else {
    c = reinterpret_cast<const float4 *>(rt + (size_t)y * rt_pitch)[x];
  }
  if (!(c.w > 0.0f)) return;  // SrcAlpha == 0 leaves the target untouched
  float4 d;
  if (tgt_fmt == GS_PIX_RGBA16F) {
    uint2 v = reinterpret_cast<const uint2 *>(tgt + (size_t)y * tgt_pitch)[x];
    d = make_float4(f16lo(v.x), f16hi(v.x), f16lo(v.y), f16hi(v.y));
  } else {
    d = reinterpret_cast<const float4 *>(tgt + (size_t)y * tgt_pitch)[x];
  }
  const float a = c.w, om = 1.0f - a;
  float4 o;
  o.x = fmaf(gamma_to_linear(__fdiv_rn(c.x, a)), a, d.x * om);
  o.y = fmaf(gamma_to_linear(__fdiv_rn(c.y, a)), a, d.y * om);
  o.z = fmaf(gamma_to_linear(__fdiv_rn(c.z, a)), a, d.z * om);
  o.w = fmaf(a, a, d.w * om);
  if (tgt_fmt == GS_PIX_RGBA16F) {
    uint2 v;
    v.x = f32tof16(o.x) | (f32tof16(o.y) << 16);
    v.y = f32tof16(o.z) | (f32tof16(o.w) << 16);
    reinterpret_cast<uint2 *>(tgt + (size_t)y * tgt_pitch)[x] = v;
  } else {
    reinterpret_cast<float4 *>(tgt + (size_t)y * tgt_pitch)[x] = o;
  }
}

void launch_composite(const void *rt, uint32_t rt_pitch, uint32_t rt_format, void *target, uint32_t tgt_pitch, uint32_t tgt_format,
                      uint32_t W, uint32_t H, cudaStream_t s) {
  if (!W || !H) return;
  dim3 grid((W + 31) / 32, (H + 7) / 8);
  k_composite<<<grid, 256, 0, s>>>(reinterpret_cast<const uint8_t *>(rt), rt_pitch, rt_format, reinterpret_cast<uint8_t *>(target),
                                   tgt_pitch, tgt_format, W, H);
}

}  // namespace gs
