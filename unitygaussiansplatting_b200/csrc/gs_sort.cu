// gs_sort.cu -- stable LSD radix sort of (uint32 key, uint32 payload) pairs for sm_100a.
//
// Replaces GpuSorting.Dispatch (R/GpuSorting.cs:142-198) and the DeviceRadixSort kernels
// (S/DeviceRadixSort.hlsl: Init/Upsweep/Scan/Downsweep; 13 dispatches, 80 B/pair of traffic).
// Same contract -- ascending, stable, 8-bit digits, 4 passes, key+payload, result back in the
// input buffers -- different algorithm: a single-pass-per-digit "onesweep" with decoupled
// look-back, so a sort is 4 data passes + one histogram read (68 B/pair) instead of
// reduce-then-scan's two reads per pass:
//   * digit histograms for all passes come from one read of the keys (or for free from
//     k_calc_distances, which wrote the keys in the first place);
//   * each CTA takes a 4096-pair tile by atomic ticket (so a tile's predecessors are
//     always resident: look-back cannot deadlock), ranks its keys with warp-level digit
//     matching (the match mask of equal digits gives the stable rank as a popc of the lower
//     lanes; one lane bumps the warp-private shared histogram), publishes the tile's
//     per-digit count with a LOCAL flag, walks back over predecessors' status words until
//     it meets an INCLUSIVE one, then publishes its own inclusive prefix;
//   * keys and payloads are first scattered inside shared memory into digit order, then
//     written out in runs, so global stores are coalesced per digit run;
//   * payloads are fetched only after ranking (their latency hides behind the look-back),
//     which keeps the kernel at <= 64 registers and 4 CTAs/SM.
// The digit width is a template parameter: depth keys use 4 x 8 bits, the tile binner sorts
// 12..16-bit tile ids in 2 passes of 6..8 bits.
// No tensor-core path: there is no contraction here, only byte/integer traffic.
#include <cstdlib>

#include "gs_kernels.cuh"

namespace gs {

enum : uint32_t { kFlagLocal = 1u << 30, kFlagIncl = 2u << 30, kValMask = (1u << 30) - 1u };

size_t sort_lookback_words(uint32_t capacity, int passes) {
  size_t tiles = ((size_t)capacity + kSortTileItems - 1) / kSortTileItems;
  return tiles * 256 * (size_t)passes;
}

// ---- digit histograms of all passes in one read -------------------------------------------
template <int PASSES, int BITS>
__global__ void __launch_bounds__(256) k_sort_hist(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ d_count,
                                                   uint32_t *__restrict__ ghist) {
  constexpr uint32_t NB = 1u << BITS;
  __shared__ uint32_t sh[PASSES * 256];
  for (int i = threadIdx.x; i < PASSES * 256; i += 256) sh[i] = 0;
  __syncthreads();
  const uint32_t n = *d_count;
  const uint32_t nvec = n >> 2;
  const uint4 *k4 = reinterpret_cast<const uint4 *>(keys);
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < nvec; i += gridDim.x * 256) {
    uint4 v = __ldg(k4 + i);
    const uint32_t kk[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int p = 0; p < PASSES; ++p) atomicAdd(&sh[p * 256 + ((kk[q] >> (BITS * p)) & (NB - 1))], 1u);
  }
  if (blockIdx.x == 0) {
    for (uint32_t i = (nvec << 2) + threadIdx.x; i < n; i += 256) {
      uint32_t k = keys[i];
#pragma unroll
      for (int p = 0; p < PASSES; ++p) atomicAdd(&sh[p * 256 + ((k >> (BITS * p)) & (NB - 1))], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < PASSES * 256; i += 256) {
    uint32_t c = sh[i];
    if (c) atomicAdd(&ghist[i], c);
  }
}

// ---- block-wide exclusive scan of one value per thread (256 threads) ------------------------
template <int WARPS>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *s_warp /*WARPS*/) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  uint32_t wsum = (lane < WARPS) ? s_warp[lane] : 0u;
  uint32_t winc = wsum;
#pragma unroll
  for (int o = 1; o < WARPS; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
    if (lane >= (uint32_t)o) winc += t;
  }
  uint32_t wexcl = __shfl_sync(0xffffffffu, winc - wsum, warp);
  __syncthreads();  // s_warp reusable afterwards
  return wexcl + inc - v;
}

// Equal-digit mask by BITS ballots.  (__match_any_sync was measured 2.4x slower than 8 ballots on B200:
// tools/mb/mb_match.cu, 1953 vs 812 ns per warp-op at 64 resident warps/SM.)
template <int BITS>
__device__ __forceinline__ uint32_t match_digit(uint32_t d) {
  uint32_t m = 0xffffffffu;
#pragma unroll
  for (int b = 0; b < BITS; ++b) {
    const bool bit = (d >> b) & 1u;
    const uint32_t bal = __ballot_sync(0xffffffffu, bit);
    m &= bit ? bal : ~bal;
  }
  return m;
}

// ---- one digit pass -------------------------------------------------------------------------
// GATHER: the keys of this pass are keys_src[payload] (pass 0 of the depth sort reads the per-splat key
// table through last frame's order, S/SplatUtilities.compute:76-81, without a separate gather pass).
// PERSIST: a fixed grid whose CTAs keep taking tiles until the (device-side) count is exhausted -- for lists whose length
// the host does not know when it launches (the binner's entry list): no capacity-sized grid of idle CTAs.
template <int BITS, bool GATHER, bool PERSIST>
__global__ void __launch_bounds__(256, 4)
k_onesweep(const uint32_t *__restrict__ src_k, const uint32_t *__restrict__ src_v, uint32_t *__restrict__ dst_k,
           uint32_t *__restrict__ dst_v, const uint32_t *__restrict__ d_count, int shift, const uint32_t *__restrict__ ghist,
           volatile uint32_t *lookback, uint32_t *ticket) {
  constexpr uint32_t NB = 1u << BITS;
  constexpr int KPT = 16;   // keys per thread
  constexpr uint32_t kTileItems = kSortTileItems;   // 256 threads x KPT
  constexpr int kSortWarps = 8;
  constexpr int kSortThreads = 256;
  extern __shared__ __align__(16) uint8_t s_dyn[];
  uint2 *s_kv = reinterpret_cast<uint2 *>(s_dyn);                                         // [kTileItems]
  uint32_t (*s_whist)[NB] = reinterpret_cast<uint32_t (*)[NB]>(s_dyn + kTileItems * 8);    // [kSortWarps][NB]
  __shared__ uint32_t s_hist[NB];
  __shared__ uint32_t s_dig_start[NB];
  __shared__ uint32_t s_off[NB];
  __shared__ uint32_t s_scan[kSortWarps];
  __shared__ uint32_t s_tile;

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t n = *d_count;
  const uint32_t num_tiles = (n + kTileItems - 1) / kTileItems;
  do {   // one tile per iteration (a single iteration unless PERSIST; every shared array written below was last read
         // before a barrier of the previous iteration, so no extra barrier is needed between tiles)
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  for (uint32_t d = tid; d < NB; d += kSortThreads) s_hist[d] = 0;
#pragma unroll
  for (uint32_t d = lane; d < NB; d += 32) s_whist[warp][d] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  if (tile >= num_tiles) return;
  const uint32_t tile_base = tile * kTileItems;
  const bool full_tile = tile_base + kTileItems <= n;

  // warp-striped load: warp w owns 512 consecutive pairs, item i of lane l is base + i*32 + l
  uint32_t key[KPT], val[KPT];
  const uint32_t wbase = tile_base + warp * (32 * KPT) + lane;
  if (GATHER) {
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      const uint32_t idx = wbase + i * 32;
      val[i] = (idx < n) ? __ldg(src_v + idx) : 0xFFFFFFFFu;
    }
#pragma unroll
    for (int i = 0; i < KPT; ++i) key[i] = (val[i] != 0xFFFFFFFFu) ? __ldg(src_k + val[i]) : 0xFFFFFFFFu;
  } else if (full_tile) {
#pragma unroll
    for (int i = 0; i < KPT; ++i) key[i] = __ldg(src_k + wbase + i * 32);
  } else {
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      const uint32_t idx = wbase + i * 32;
      key[i] = (idx < n) ? __ldg(src_k + idx) : 0xFFFFFFFFu;  // pads sort last (S/SortCommon.hlsl:244-247 does the same)
    }
  }

  // 1. tile digit histogram (cheap, before ranking) so that the LOCAL count is published as early as possible
#pragma unroll
  for (int i = 0; i < KPT; ++i) {
    const uint32_t d = (key[i] >> shift) & (NB - 1);
    const uint32_t d0 = __shfl_sync(0xffffffffu, d, 0);
    if (__all_sync(0xffffffffu, d == d0)) {   // skewed digits (high bytes of depth keys): one add per warp
      if (lane == 0) atomicAdd(&s_hist[d0], 32u);
    } else {
      atomicAdd(&s_hist[d], 1u);
    }
  }
  __syncthreads();

  // 2. publish, then resolve the exclusive prefix over earlier tiles with 4 status probes in flight
  uint32_t prefix = 0, tile_total = 0;
  if (tid < NB) {
    tile_total = s_hist[tid];  // includes pads (only the last digit of the last tile)
    uint32_t pub = tile_total;
    if (tid == NB - 1 && !full_tile) pub -= (tile_base + kTileItems - n);
    volatile uint32_t *lb = lookback + (size_t)tile * NB + tid;
    if (tile == 0) {
      *lb = kFlagIncl | pub;
    } else {
      *lb = kFlagLocal | pub;
      int t = (int)tile - 1;
      bool done = false;
      constexpr int kProbe = 4;   // status probes in flight per round (8 measured slower: more polling traffic, same wait)
      while (!done) {
        uint32_t v[kProbe];
#pragma unroll
        for (int q = 0; q < kProbe; ++q) v[q] = (t - q >= 0) ? lookback[(size_t)(t - q) * NB + tid] : (uint32_t)kFlagIncl;
        int used = 0;
#pragma unroll
        for (int q = 0; q < kProbe; ++q) {
          if (!done && used == q) {
            if (v[q] != 0) {
              prefix += v[q] & kValMask;
              used = q + 1;
              if (v[q] & kFlagIncl) done = true;
            }
          }
        }
        t -= used;
      }
      *lb = kFlagIncl | (prefix + pub);
    }
  }
  __syncwarp();   // the spin loop above ends per thread: tell the compiler the warp is whole again before the ballots
  if (!GATHER) {  // payloads: issued now, consumed at the scatter
    if (full_tile) {
#pragma unroll
      for (int i = 0; i < KPT; ++i) val[i] = __ldg(src_v + wbase + i * 32);
    } else {
#pragma unroll
      for (int i = 0; i < KPT; ++i) {
        const uint32_t idx = wbase + i * 32;
        val[i] = (idx < n) ? __ldg(src_v + idx) : 0u;
      }
    }
  }

  // 3. stable in-warp ranking; ranks (< 4096) are packed two per register
  uint32_t rank2[KPT / 2];
  const uint32_t lt_mask = (1u << lane) - 1u;
#pragma unroll
  for (int i = 0; i < KPT; ++i) {
    const uint32_t d = (key[i] >> shift) & (NB - 1);
    const uint32_t m = match_digit<BITS>(d);
    // every lane reads its digit's running count (lanes of one digit read one word: a broadcast), then the lowest lane of
    // each digit group -- the one with no equal-digit lane below it -- stores the new count: a predicated store, no
    // branch, no shuffle.  The __syncwarp() orders round i's store before round i+1's loads for the memory model (and for
    // compute-sanitizer's racecheck, which flagged the version without it); it costs nothing measurable.
    const uint32_t below = __popc(m & lt_mask);
    const uint32_t prev = s_whist[warp][d];
    __syncwarp();
    if (below == 0) s_whist[warp][d] = prev + __popc(m);
    const uint32_t r = prev + below;
    if (i & 1) rank2[i >> 1] |= r << 16; else rank2[i >> 1] = r;
    __syncwarp();
  }
  __syncthreads();

  // 4. thread `tid` < NB owns digit `tid`: exclusive prefix over warps, tile/global digit bases
  if (tid < NB) {
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
      uint32_t c = s_whist[w][tid];
      s_whist[w][tid] = run;
      run += c;
    }
  }
  const uint32_t dig_start = block_excl_scan<kSortWarps>(tile_total, s_scan);
  const uint32_t gbase = block_excl_scan<kSortWarps>(tid < NB ? __ldg(ghist + tid) : 0u, s_scan);
  if (tid < NB) {
    s_dig_start[tid] = dig_start;
    s_off[tid] = gbase + prefix - dig_start;
  }
  __syncthreads();

  // 5. scatter into digit order inside shared memory
#pragma unroll
  for (int i = 0; i < KPT; ++i) {
    const uint32_t d = (key[i] >> shift) & (NB - 1);
    const uint32_t r = (i & 1) ? (rank2[i >> 1] >> 16) : (rank2[i >> 1] & 0xffffu);
    const uint32_t pos = s_dig_start[d] + s_whist[warp][d] + r;
    s_kv[pos] = make_uint2(key[i], val[i]);
  }
  __syncthreads();

  const uint32_t valid = full_tile ? kTileItems : n - tile_base;
#pragma unroll 4
  for (uint32_t j = tid; j < valid; j += kSortThreads) {
    const uint2 kv = s_kv[j];
    const uint32_t dst = j + s_off[(kv.x >> shift) & (NB - 1)];
    dst_k[dst] = kv.x;
    dst_v[dst] = kv.y;
  }
  } while (PERSIST);
}

// zero `per_item_words * ceil(count / items)` words, count read on the device: clears exactly the look-back rows a sort of a
// device-sized list will use (instead of a capacity-sized cudaMemset)
__global__ void __launch_bounds__(256) k_zero_rows(uint32_t *__restrict__ buf, const uint32_t *__restrict__ d_count, uint32_t items,
                                                   uint32_t words_per_row, uint32_t row_stride_words, uint32_t reps, uint32_t rep_stride_words) {
  const uint32_t rows = (*d_count + items - 1) / items;
  const size_t per_rep = (size_t)rows * words_per_row;
  for (size_t i = blockIdx.x * 256 + threadIdx.x; i < per_rep * reps; i += (size_t)gridDim.x * 256) {
    const uint32_t rep = (uint32_t)(i / per_rep);
    const size_t j = i - (size_t)rep * per_rep;
    buf[(size_t)rep * rep_stride_words + (j / words_per_row) * row_stride_words + (j % words_per_row)] = 0u;
  }
}

// ---- ordered compaction of a draw order by a membership mask ------------------------------------------
// (out_ids, out_keys) = (id, key_table[id]) of the ids of order[0..n) whose bit is set in `mask`, in the order they stand in: the
// input of a slab's radix sort, compacted out of last frame's draw order.  One status word per 4096-item block, decoupled
// look-back 32 predecessors wide (gs_common.cuh).  The walk reads the order once (coalesced); per id it first looks at one bit per 128 ids in
// a bitmap held in shared memory (a random lookup per draw-order entry through L1 costs ~22 us per 6.1 M entries on B200 however
// small the table: 32 distinct lines per warp load) and touches the mask word -- a random L2 access -- only where that
// group has members at all.
constexpr int kCmpItems = 16;
constexpr int kCmpBlock = 256 * kCmpItems;
enum : uint32_t { kCmpFlagLocal = kLbLocal, kCmpFlagIncl = kLbIncl, kCmpValMask = kLbMask };

__global__ void __launch_bounds__(256) k_compact_order(const uint32_t *__restrict__ order, uint32_t n, const uint32_t *__restrict__ mask,
                                                       const uint32_t *__restrict__ group_bits, uint32_t bits_words,
                                                       const uint32_t *__restrict__ key_table, uint32_t *__restrict__ out_ids,
                                                       uint32_t *__restrict__ out_keys, volatile uint32_t *status, uint32_t *ticket,
                                                       uint32_t *__restrict__ count_out) {
  extern __shared__ uint32_t s_bits[];   // the group bitmap (bits_words words), or nothing when it is too large to hold
  __shared__ uint32_t s_w[8];
  __shared__ uint32_t s_block, s_excl;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_block = atomicAdd(ticket, 1u);
  for (uint32_t i = threadIdx.x; i < bits_words; i += 256) s_bits[i] = __ldg(group_bits + i);
  __syncthreads();
  const uint32_t b = s_block;
  const uint32_t nblocks = (n + kCmpBlock - 1) / kCmpBlock;
  const uint32_t wbase = b * kCmpBlock + warp * (32 * kCmpItems) + lane;
  uint32_t id[kCmpItems];
#pragma unroll
  for (int i = 0; i < kCmpItems; ++i) {
    const uint32_t r = wbase + i * 32;
    id[i] = (r < n) ? __ldg(order + r) : 0xFFFFFFFFu;
  }
  uint32_t keepbits = 0;
#pragma unroll
  for (int i = 0; i < kCmpItems; ++i) {
    bool keep = id[i] != 0xFFFFFFFFu;
    if (keep) {
      const uint32_t gw = bits_words ? s_bits[id[i] >> 12] : __ldg(group_bits + (id[i] >> 12));
      keep = ((gw >> ((id[i] >> 7) & 31u)) & 1u) && ((__ldg(mask + (id[i] >> 5)) >> (id[i] & 31u)) & 1u);
    }
    keepbits |= keep ? (1u << i) : 0u;
  }
  // ranks: slot i of a warp holds 32 consecutive order positions -> ballot prefix inside the slot, running sum over slots
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t pos[kCmpItems], wsum = 0;
#pragma unroll
  for (int i = 0; i < kCmpItems; ++i) {
    const uint32_t bal = __ballot_sync(0xffffffffu, (keepbits >> i) & 1u);
    pos[i] = wsum + __popc(bal & lt);
    wsum += __popc(bal);
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
    if (lane == 0) status[b] = (b == 0 ? kCmpFlagIncl : kCmpFlagLocal) | total;
    uint32_t excl = 0;
    if (b > 0) {
      excl = lookback_exclusive(status, b);
      if (lane == 0) status[b] = kCmpFlagIncl | (excl + total);
    }
    if (lane == 0) {
      s_excl = excl;
      if (b == nblocks - 1) *count_out = excl + total;
    }
  }
  __syncthreads();
  const uint32_t base = s_excl + woff;
#pragma unroll
  for (int i = 0; i < kCmpItems; ++i) {
    if ((keepbits >> i) & 1u) {
      out_ids[base + pos[i]] = id[i];
      out_keys[base + pos[i]] = __ldg(key_table + id[i]);
    }
  }
}

size_t compact_status_words(uint32_t n) { return (size_t)(n + kCmpBlock - 1) / kCmpBlock + 1; }

void launch_compact_order(const uint32_t *order, uint32_t n, const uint32_t *mask, const uint32_t *group_bits, const uint32_t *key_table,
                          uint32_t *out_ids, uint32_t *out_keys, uint32_t *status /* compact_status_words(n) */, uint32_t *count_out, cudaStream_t s) {
  if (!n) { cudaMemsetAsync(count_out, 0, 4, s); return; }
  const uint32_t nblocks = (n + kCmpBlock - 1) / kCmpBlock;
  cudaMemsetAsync(status, 0, ((size_t)nblocks + 1) * sizeof(uint32_t), s);   // [0] ticket, [1..] look-back status
  uint32_t words = (uint32_t)group_bits_words(n);
  static int bits_global = -1;   // GS_WALK_BITS_GLOBAL=1 forces the large-asset path (bitmap read through L1) for tests
  if (bits_global < 0) { const char *e = getenv("GS_WALK_BITS_GLOBAL"); bits_global = (e && e[0] == '1') ? 1 : 0; }
  if (bits_global) words = 0;
  if (words * 4u > 40u * 1024u) words = 0;   // a bitmap that does not fit the default shared memory is read through L1 instead
  k_compact_order<<<nblocks, 256, words * 4u, s>>>(order, n, mask, group_bits, words, key_table, out_ids, out_keys, status + 1, status, count_out);
}

template <int BITS>
static void launch_pass(uint32_t count_bound, bool persist, cudaStream_t s, const uint32_t *sk, const uint32_t *sv, uint32_t *dk,
                        uint32_t *dv, const uint32_t *d_count, int shift, const uint32_t *ghist, uint32_t *lookback, uint32_t *ticket,
                        bool gather) {
  // 32 KB of pairs + 8 KB of warp histograms at BITS = 8, plus 3 KB of static shared memory: within the default 48 KB
  const size_t smem = (size_t)kSortTileItems * 8 + 8 * (1u << BITS) * 4;
  uint32_t grid = (uint32_t)(((uint64_t)count_bound + kSortTileItems - 1) / kSortTileItems);
  auto go = [&](auto kern) { kern<<<grid, 256, smem, s>>>(sk, sv, dk, dv, d_count, shift, ghist, lookback, ticket); };
  if (persist) {
    grid = min(grid, 148u * 4u);
    if (gather) go(k_onesweep<BITS, true, true>); else go(k_onesweep<BITS, false, true>);
  } else {
    if (gather) go(k_onesweep<BITS, true, false>); else go(k_onesweep<BITS, false, false>);
  }
}

void launch_sort_pairs(uint32_t *keys, uint32_t *vals, const uint32_t *d_count, uint32_t capacity, int passes, int bits,
                       bool hist_ready, const SortScratch &sc, cudaStream_t s, cudaEvent_t *pass_events, const uint32_t *key_table,
                       bool count_is_capacity, uint32_t *final_keys, uint32_t *final_vals) {
  if (capacity == 0) return;
  const uint32_t tiles = (capacity + kSortTileItems - 1) / kSortTileItems;
  const uint32_t nb = 1u << bits;
  // count_is_capacity: the host knows the exact count (depth sort, slab sort) -> exact grid, exact memset.  Otherwise the list
  // length lives on the device only (the binner's entries): a persistent grid, and the look-back rows actually needed are
  // cleared by a kernel that reads the count.
  const bool persist = !count_is_capacity;
  // Half-size tiles for a slab's exact, smallish count were measured slower on B200 (24.0 vs 22 us per pass of 1.5 M pairs):
  // a pass is bound by its fixed per-tile work, not by the tile count.
  if (persist) k_zero_rows<<<148, 256, 0, s>>>(sc.lookback, d_count, kSortTileItems, nb, nb, (uint32_t)passes, tiles * nb);
  else cudaMemsetAsync(sc.lookback, 0, (size_t)tiles * nb * passes * sizeof(uint32_t), s);
  cudaMemsetAsync(sc.tickets, 0, 4 * sizeof(uint32_t), s);
  if (!hist_ready) {
    cudaMemsetAsync(sc.ghist, 0, 4 * 256 * sizeof(uint32_t), s);
    const uint32_t grid = min(tiles, 148u * 8u);
    if (passes == 4) k_sort_hist<4, 8><<<grid, 256, 0, s>>>(keys, d_count, sc.ghist);
    else if (bits == 5) k_sort_hist<2, 5><<<grid, 256, 0, s>>>(keys, d_count, sc.ghist);
    else if (bits == 6) k_sort_hist<2, 6><<<grid, 256, 0, s>>>(keys, d_count, sc.ghist);
    else if (bits == 7) k_sort_hist<2, 7><<<grid, 256, 0, s>>>(keys, d_count, sc.ghist);
    else k_sort_hist<2, 8><<<grid, 256, 0, s>>>(keys, d_count, sc.ghist);
  }
  uint32_t *sk = keys, *sv = vals, *dk = sc.alt_keys, *dv = sc.alt_vals;
  for (int p = 0; p < passes; ++p) {
    if (pass_events) cudaEventRecord(pass_events[p], s);
    uint32_t *lb = sc.lookback + (size_t)p * tiles * nb;
    const bool gather = key_table != nullptr && p == 0;   // pass 0 reads key_table[vals[i]] instead of keys[i]
    const uint32_t *src_keys = gather ? key_table : sk;
    if (p == passes - 1 && final_keys && final_vals) { dk = final_keys; dv = final_vals; }   // the last pass lands where the caller wants it
    if (bits == 5) launch_pass<5>(capacity, persist, s, src_keys, sv, dk, dv, d_count, bits * p, sc.ghist + 256 * p, lb, sc.tickets + p, gather);
    else if (bits == 6) launch_pass<6>(capacity, persist, s, src_keys, sv, dk, dv, d_count, bits * p, sc.ghist + 256 * p, lb, sc.tickets + p, gather);
    else if (bits == 7) launch_pass<7>(capacity, persist, s, src_keys, sv, dk, dv, d_count, bits * p, sc.ghist + 256 * p, lb, sc.tickets + p, gather);
    else launch_pass<8>(capacity, persist, s, src_keys, sv, dk, dv, d_count, bits * p, sc.ghist + 256 * p, lb, sc.tickets + p, gather);
    uint32_t *t = sk; sk = dk; dk = t;
    t = sv; sv = dv; dv = t;
  }
  if (pass_events) cudaEventRecord(pass_events[passes], s);
}

}  // namespace gs
