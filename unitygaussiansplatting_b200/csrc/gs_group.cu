// gs_group.cu -- one frame on the G GPUs of one box (include/gsplat_b200.h, "several GPUs"; SURVEY 8e.1 + 8e.2).
//
// The reference is single-GPU; what a group must reproduce is its per-frame contract: after SortPoints the persistent order
// buffer holds the stable ascending sort of the depth keys taken through last frame's order (R/GaussianSplatRenderer.cs:612-639,
// R/GpuSorting.cs:142-198), and the render target holds the front-to-back blend of every splat in that order
// (S/RenderGaussianSplats.shader:10-12,79-108).  Both come out bit-identical to gs_frame on one GPU, because
//   * the sort is sharded by KEY RANGE.  Splitters are the current keys of the splats at the quantile positions of last
//     frame's order (replicated data -> the same values on every GPU).  GPU g compacts, out of last frame's order, the
//     splats of slab g -- keys in [splitter g-1, splitter g) -- and radix-sorts only those.  A stable sort of a
//     subsequence is the subsequence of the stable sort, ties never straddle a splitter, so the slabs concatenated ARE
//     the single-GPU order.  Slab sizes fall out of the distance kernel on every GPU (counts of keys >= each splitter),
//     so every GPU knows every offset and the exchange needs no size negotiation;
//   * every pixel is composited by exactly one GPU, from the same per-bin list in the same order.  Each GPU owns a
//     contiguous range of 16-pixel rows, culls view-calc / binning to it, composites straight into place; the ranges are
//     re-cut every frame from the per-row cost measured two frames earlier (exchanged with the pixels), which is the
//     same on every GPU, so the cuts agree without a negotiation either.
// Streams: the sort chain and the compositing chain run on the context stream, view-calc beside the sort on a second
// (lowest-priority) stream, the exchange of composited rows / row costs and the host read-back on a third, overlapping the
// next frame; the only host wait inside a frame is for the 128-byte slab table (the GPU is busy with view-calc meanwhile).
// Order exchange, fastest available first: one process per GPU -> remote stores into the peers' order buffers mapped through
// CUDA IPC (k_push_slab / k_wait_slabs, no NCCL call in the frame); several members in one process, or IPC unavailable ->
// one ncclAllGather of equal slots + G device copies; badly unbalanced slabs -> grouped NCCL broadcasts of the exact sizes in
// place.  Row exchange: grouped NCCL broadcasts in place.  In GS_GROUP_EMULATE, or without NCCL in a single process, plain
// device-to-device copies ordered by events stand in for every exchange.
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "gs_internal.cuh"
#include "gs_nccl.h"

using namespace gs;

namespace {

enum { GT_BEGIN = 0, GT_DIST, GT_SORT, GT_ORDER, GT_VIEWWAIT, GT_RASTER, GT_IMAGE, GT_V0, GT_V1, GT_COUNT };

struct Member {
  GsContext *ctx = nullptr;
  bool own_ctx = false;
  uint32_t rank = 0;
  ncclComm_t comm = nullptr;
  cudaStream_t aux = nullptr;   // view-calc runs here, beside the sort chain (lowest priority: it fills what the sort chain leaves idle)
  cudaStream_t xfer = nullptr;  // the exchange of the composited rows runs here and overlaps the NEXT frame's sort chain
  cudaEvent_t ev_raster = nullptr, ev_image = nullptr;   // rows composited / rows of every GPU in place (and read back)
  bool image_pending = false;
  cudaEvent_t ev_begin = nullptr, ev_view = nullptr, ev_info = nullptr, ev_cost[2] = {nullptr, nullptr};
  cudaEvent_t ev_produced = nullptr, ev_consumed = nullptr;   // emulated exchange
  cudaEvent_t tev[GT_COUNT]{};
  uint32_t *d_info = nullptr, *d_slab_count = nullptr, *d_cmp_status = nullptr, *d_row_cost = nullptr;
  uint32_t *d_gather = nullptr;   // staging of the order exchange: G slabs of `cap` ids each (the all-gather's buffer)
  size_t gather_words = 0;
  size_t cmp_words = 0;
  uint32_t rows_cap = 0;
  uint32_t *h_info = nullptr, *h_row_cost[2] = {nullptr, nullptr};   // pinned
  void *rt_scratch = nullptr;
  size_t rt_bytes = 0;
};

}  // namespace

// Peer-to-peer order exchange (one process per GPU): every process maps every peer's two order buffers and flag words
// through CUDA IPC; after its slab sort a GPU stores its slab straight into all peers' NEW order buffer over NVLink and
// raises a flag there; nobody calls into NCCL, nothing is staged or unpacked.
struct PeerLink {
  bool tried = false, ready = false;
  GsAsset *asset = nullptr;
  uint32_t *buf[2] = {nullptr, nullptr};                       // local: the asset's two order buffers, by fixed index
  uint32_t *peer_buf[2][GS_GROUP_MAX_GPUS] = {};               // the same two buffers of every rank (own rank: local)
  uint32_t *flags = nullptr, *peer_flags[GS_GROUP_MAX_GPUS] = {};   // flags[c] = last sort frame whose slab rank c delivered here
  uint32_t *d_done = nullptr;                                   // block counter of the push kernel
  void *opened[3 * GS_GROUP_MAX_GPUS] = {};
  int n_opened = 0;
  uint32_t sort_frames = 0;
};

struct GsGroup {
  PeerLink link;
  uint32_t size = 0;
  std::vector<Member> m;
  bool emulate = false, use_nccl = false;
  uint64_t frame = 0;
  uint32_t hist_w = 0, hist_h = 0;
  uint64_t hist_frames = 0;   // frames rendered at (hist_w, hist_h): the cost of frame k is usable from frame k+2 on
  uint32_t bounds[GS_GROUP_MAX_GPUS + 1]{};
  uint32_t slab_off[GS_GROUP_MAX_GPUS + 1]{}, slab_cnt[GS_GROUP_MAX_GPUS]{};
  bool timed = false;
};

namespace {

int fail_nccl(GsContext *ctx, ncclResult_t r, const char *what) {
  char buf[256];
  snprintf(buf, sizeof(buf), "NCCL error %d (%s) in %s", (int)r, nccl_api().GetErrorString ? nccl_api().GetErrorString(r) : "?", what);
  return fail(ctx, GS_ERR_CUDA, buf);
}
#define GS_NCCL_TRY(ctx, expr)                                   \
  do {                                                           \
    ncclResult_t _r = (expr);                                    \
    if (_r != ncclSuccess) return fail_nccl((ctx), _r, #expr);   \
  } while (0)

// inside ncclGroupStart ... ncclGroupEnd: a failed call closes the group before the error is returned
#define GS_NCCL_TRY_G(ctx, expr)                                                   \
  do {                                                                             \
    ncclResult_t _r = (expr);                                                      \
    if (_r != ncclSuccess) { nccl_api().GroupEnd(); return fail_nccl((ctx), _r, #expr); } \
  } while (0)

int member_init(Member &mb) {
  GsContext *ctx = mb.ctx;
  GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int least = 0, greatest = 0;
  GS_CUDA_TRY(ctx, cudaDeviceGetStreamPriorityRange(&least, &greatest));
  GS_CUDA_TRY(ctx, cudaStreamCreateWithPriority(&mb.aux, cudaStreamNonBlocking, least));
  GS_CUDA_TRY(ctx, cudaStreamCreateWithPriority(&mb.xfer, cudaStreamNonBlocking, greatest));
  cudaEvent_t *evs[] = {&mb.ev_begin, &mb.ev_view, &mb.ev_info, &mb.ev_cost[0], &mb.ev_cost[1], &mb.ev_produced, &mb.ev_consumed, &mb.ev_raster, &mb.ev_image};
  for (cudaEvent_t *e : evs) GS_CUDA_TRY(ctx, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  for (int i = 0; i < GT_COUNT; ++i) GS_CUDA_TRY(ctx, cudaEventCreate(&mb.tev[i]));
  GS_CUDA_TRY(ctx, cudaMalloc(&mb.d_info, 2 * kMaxSlabs * 4));
  GS_CUDA_TRY(ctx, cudaMalloc(&mb.d_slab_count, 16));
  GS_CUDA_TRY(ctx, cudaMallocHost(&mb.h_info, 2 * kMaxSlabs * 4));
  return GS_OK;
}

void member_free(Member &mb) {
  if (!mb.ctx) return;
  cudaSetDevice(mb.ctx->device);
  cudaStreamSynchronize(mb.ctx->stream);
  if (mb.aux) { cudaStreamSynchronize(mb.aux); cudaStreamDestroy(mb.aux); }
  if (mb.xfer) { cudaStreamSynchronize(mb.xfer); cudaStreamDestroy(mb.xfer); }
  cudaEvent_t evs[] = {mb.ev_begin, mb.ev_view, mb.ev_info, mb.ev_cost[0], mb.ev_cost[1], mb.ev_produced, mb.ev_consumed, mb.ev_raster, mb.ev_image};
  for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
  for (int i = 0; i < GT_COUNT; ++i) if (mb.tev[i]) cudaEventDestroy(mb.tev[i]);
  cudaFree(mb.d_info); cudaFree(mb.d_slab_count); cudaFree(mb.d_cmp_status); cudaFree(mb.d_row_cost); cudaFree(mb.rt_scratch); cudaFree(mb.d_gather);
  cudaFreeHost(mb.h_info); cudaFreeHost(mb.h_row_cost[0]); cudaFreeHost(mb.h_row_cost[1]);
  if (mb.comm && nccl_api().ok()) nccl_api().CommDestroy(mb.comm);
  if (mb.own_ctx) gs_destroy(mb.ctx);
  mb.ctx = nullptr;
}

int member_rows(Member &mb, uint32_t rows) {   // row-cost vectors for a screen of `rows` 16-pixel rows
  if (rows <= mb.rows_cap) return GS_OK;
  GsContext *ctx = mb.ctx;
  cudaStreamSynchronize(ctx->stream);
  cudaFree(mb.d_row_cost); cudaFreeHost(mb.h_row_cost[0]); cudaFreeHost(mb.h_row_cost[1]);
  mb.d_row_cost = nullptr; mb.h_row_cost[0] = mb.h_row_cost[1] = nullptr; mb.rows_cap = 0;
  GS_CUDA_TRY(ctx, cudaMalloc(&mb.d_row_cost, (size_t)rows * 4));
  GS_CUDA_TRY(ctx, cudaMallocHost(&mb.h_row_cost[0], (size_t)rows * 4));
  GS_CUDA_TRY(ctx, cudaMallocHost(&mb.h_row_cost[1], (size_t)rows * 4));
  mb.rows_cap = rows;
  return GS_OK;
}

int member_asset(Member &mb, GsAsset *as) {   // per-asset buffers only the group path needs
  GsContext *ctx = mb.ctx;
  const uint32_t n = as->av.n;
  if (!as->slab_mask) GS_CUDA_TRY(ctx, cudaMalloc(&as->slab_mask, ((size_t)(n + 1023) / 1024) * 128 + 64));
  if (!as->order_tmp) GS_CUDA_TRY(ctx, cudaMalloc(&as->order_tmp, (size_t)n * 4 + 16));
  if (!as->slab_group_bits) GS_CUDA_TRY(ctx, cudaMalloc(&as->slab_group_bits, group_bits_words(n) * 4 + 64));
  const size_t words = compact_status_words(n);
  if (words > mb.cmp_words) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(mb.d_cmp_status);
    mb.d_cmp_status = nullptr; mb.cmp_words = 0;
    GS_CUDA_TRY(ctx, cudaMalloc(&mb.d_cmp_status, words * 4));
    mb.cmp_words = words;
  }
  return ensure_sort_scratch(ctx, n);
}

// ---- the exchange: every member ends up with every segment ------------------------------------------------------------
// bufs[i]: local member i's copy of the whole buffer; segment c = bytes [off[c], off[c] + cnt[c]) is produced by rank c.
int exchange_begin(GsGroup *g) {
  if (g->use_nccl) GS_NCCL_TRY(g->m[0].ctx, nccl_api().GroupStart());
  return GS_OK;
}
// on_xfer: use the members' transfer streams instead of their context streams
int exchange_add(GsGroup *g, uint8_t *const *bufs, const size_t *off, const size_t *cnt, bool on_xfer = false) {
  const uint32_t G = g->size;
  auto st = [&](Member &m) -> cudaStream_t { return on_xfer ? m.xfer : m.ctx->stream; };
  if (g->use_nccl) {
    const NcclApi &nc = nccl_api();
    for (size_t i = 0; i < g->m.size(); ++i) {
      Member &mb = g->m[i];
      for (uint32_t c = 0; c < G; ++c)
        if (cnt[c]) GS_NCCL_TRY_G(mb.ctx, nc.Broadcast(bufs[i] + off[c], bufs[i] + off[c], cnt[c], ncclUint8, (int)c, mb.comm, st(mb)));
    }
    return GS_OK;
  }
  // all ranks are local members (member i == rank i): copies ordered by events, with barrier semantics like a collective
  for (Member &mb : g->m) { cudaSetDevice(mb.ctx->device); GS_CUDA_TRY(mb.ctx, cudaEventRecord(mb.ev_produced, st(mb))); }
  for (uint32_t d = 0; d < G; ++d) {
    Member &dst = g->m[d];
    cudaSetDevice(dst.ctx->device);
    for (uint32_t c = 0; c < G; ++c) {
      if (c == d || !cnt[c]) continue;
      GS_CUDA_TRY(dst.ctx, cudaStreamWaitEvent(st(dst), g->m[c].ev_produced, 0));
      GS_CUDA_TRY(dst.ctx, cudaMemcpyAsync(bufs[d] + off[c], bufs[c] + off[c], cnt[c], cudaMemcpyDefault, st(dst)));
    }
    GS_CUDA_TRY(dst.ctx, cudaEventRecord(dst.ev_consumed, st(dst)));
  }
  for (uint32_t c = 0; c < G; ++c) {
    cudaSetDevice(g->m[c].ctx->device);
    for (uint32_t d = 0; d < G; ++d)
      if (d != c) GS_CUDA_TRY(g->m[c].ctx, cudaStreamWaitEvent(st(g->m[c]), g->m[d].ev_consumed, 0));
  }
  return GS_OK;
}
int exchange_end(GsGroup *g) {
  if (g->use_nccl) GS_NCCL_TRY(g->m[0].ctx, nccl_api().GroupEnd());
  return GS_OK;
}

// The order exchange as ONE ncclAllGather: NCCL's all-gather moves the 24.5 MB of cfg2 in 60 us on two B200s where grouped
// broadcasts / send-recv of the exact slab sizes take 97 (tools/mb_exchange.py), so every GPU sorts its slab into slot `rank`
// of a staging buffer of G equal slots (cap = the largest slab), the slots are gathered in place, and G device copies move
// slot c's first cnt[c] ids to their place off[c] of the order.
int exchange_allgather(GsGroup *g, uint8_t *const *bufs, size_t slot_bytes, const size_t *cnt) {
  const uint32_t G = g->size;
  if (g->use_nccl) {
    const NcclApi &nc = nccl_api();
    GS_NCCL_TRY(g->m[0].ctx, nc.GroupStart());
    for (size_t i = 0; i < g->m.size(); ++i) {
      Member &mb = g->m[i];
      GS_NCCL_TRY_G(mb.ctx, nc.AllGather(bufs[i] + (size_t)mb.rank * slot_bytes, bufs[i], slot_bytes, ncclUint8, mb.comm, mb.ctx->stream));
    }
    GS_NCCL_TRY(g->m[0].ctx, nc.GroupEnd());
    return GS_OK;
  }
  size_t off[GS_GROUP_MAX_GPUS];
  for (uint32_t c = 0; c < G; ++c) off[c] = (size_t)c * slot_bytes;
  return exchange_add(g, bufs, off, cnt);   // device copies of the filled part of every slot
}

struct PushArgs { uint32_t *dst[GS_GROUP_MAX_GPUS]; uint32_t *flag[GS_GROUP_MAX_GPUS]; uint32_t npeers; };

// Stores this GPU's sorted slab into every peer's order buffer (remote stores over NVLink, coalesced 4-byte lanes), then --
// once every block's stores are fenced system-wide -- the last block raises this rank's flag on every peer.
__global__ void __launch_bounds__(512) k_push_slab(const uint32_t *__restrict__ src, uint32_t cnt, PushArgs a, uint32_t tag, uint32_t *done) {
  for (uint32_t p = 0; p < a.npeers; ++p) {
    uint32_t *dst = a.dst[p];
    for (uint32_t i = blockIdx.x * 512 + threadIdx.x; i < cnt; i += gridDim.x * 512) dst[i] = __ldg(src + i);
  }
  __threadfence_system();
  __syncthreads();
  __shared__ uint32_t s_last;
  if (threadIdx.x == 0) s_last = atomicAdd(done, 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  if (s_last) {
    __threadfence_system();
    if (threadIdx.x < a.npeers) *reinterpret_cast<volatile uint32_t *>(a.flag[threadIdx.x]) = tag;
    if (threadIdx.x == 0) *done = 0;
  }
}

// Waits until every other rank's flag here has reached `tag` (their slabs are in this GPU's order buffer).  A peer that never
// delivers would hang the stream: after ~2 s the kernel gives up and records it (flags[count] != 0 -> the frame is void).
__global__ void k_wait_slabs(volatile uint32_t *flags, uint32_t count, uint32_t self, uint32_t tag) {
  const uint32_t c = threadIdx.x;
  if (c < count && c != self) {
    const long long t0 = clock64();
    while ((int32_t)(flags[c] - tag) < 0) {
      __nanosleep(200);
      if (clock64() - t0 > 4000000000ll) { flags[count] = 1u; break; }
    }
  }
  __threadfence_system();
}

// Collective (every process of the group, same call sequence).  On any failure anywhere the link stays off and the NCCL
// exchange is used.
int peer_link_setup(GsGroup *g, GsAsset *as) {
  PeerLink &k = g->link;
  k.tried = true;
  Member &mb = g->m[0];
  GsContext *ctx = mb.ctx;
  const uint32_t G = g->size, n = as->av.n;
  const NcclApi &nc = nccl_api();
  struct Pack { cudaIpcMemHandle_t h[3]; uint32_t ok; uint32_t pad[15]; };
  static_assert(sizeof(Pack) == 3 * 64 + 64, "pack layout");
  Pack mine;
  memset(&mine, 0, sizeof(mine));
  bool ok = true;
  if (!as->order_alt) ok = cudaMalloc(&as->order_alt, (size_t)n * 4 + 16) == cudaSuccess;
  if (ok && !k.flags) ok = cudaMalloc(&k.flags, 64 * 4) == cudaSuccess && cudaMalloc(&k.d_done, 16) == cudaSuccess;
  if (ok) {
    cudaMemsetAsync(k.flags, 0, 64 * 4, ctx->stream);
    cudaMemsetAsync(k.d_done, 0, 16, ctx->stream);
    cudaMemsetAsync(as->order_alt, 0, (size_t)n * 4, ctx->stream);
    ok = cudaIpcGetMemHandle(&mine.h[0], as->order) == cudaSuccess && cudaIpcGetMemHandle(&mine.h[1], as->order_alt) == cudaSuccess &&
         cudaIpcGetMemHandle(&mine.h[2], k.flags) == cudaSuccess;
  }
  cudaGetLastError();
  mine.ok = ok ? 1u : 0u;
  Pack *d_all = nullptr;
  std::vector<Pack> all(G);
  if (cudaMalloc(&d_all, sizeof(Pack) * G) != cudaSuccess) return fail(ctx, GS_ERR_OUT_OF_MEMORY, "peer link: device allocation failed");
  cudaMemcpyAsync(d_all + mb.rank, &mine, sizeof(Pack), cudaMemcpyHostToDevice, ctx->stream);
  ncclResult_t r = nc.AllGather(d_all + mb.rank, d_all, sizeof(Pack), ncclUint8, mb.comm, ctx->stream);
  if (r != ncclSuccess) { cudaFree(d_all); return fail_nccl(ctx, r, "ncclAllGather(peer handles)"); }
  cudaMemcpyAsync(all.data(), d_all, sizeof(Pack) * G, cudaMemcpyDeviceToHost, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { cudaFree(d_all); return fail(ctx, GS_ERR_CUDA, "peer link: handle exchange failed"); }
  bool everyone = true;
  for (uint32_t c = 0; c < G; ++c) everyone &= all[c].ok != 0;
  uint32_t opened_ok = everyone ? 1u : 0u;
  if (everyone) {
    k.buf[0] = as->order; k.buf[1] = as->order_alt;
    for (uint32_t c = 0; c < G && opened_ok; ++c) {
      if (c == mb.rank) { k.peer_buf[0][c] = k.buf[0]; k.peer_buf[1][c] = k.buf[1]; k.peer_flags[c] = k.flags; continue; }
      void *ptr[3] = {nullptr, nullptr, nullptr};
      for (int j = 0; j < 3 && opened_ok; ++j) {
        if (cudaIpcOpenMemHandle(&ptr[j], all[c].h[j], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { opened_ok = 0; cudaGetLastError(); break; }
        k.opened[k.n_opened++] = ptr[j];
      }
      k.peer_buf[0][c] = (uint32_t *)ptr[0]; k.peer_buf[1][c] = (uint32_t *)ptr[1]; k.peer_flags[c] = (uint32_t *)ptr[2];
    }
  }
  // second round: did everybody manage to map everybody?
  uint32_t *d_ok = reinterpret_cast<uint32_t *>(d_all);
  cudaMemcpyAsync(d_ok + mb.rank, &opened_ok, 4, cudaMemcpyHostToDevice, ctx->stream);
  r = nc.AllGather(d_ok + mb.rank, d_ok, 4, ncclUint8, mb.comm, ctx->stream);
  std::vector<uint32_t> oks(G, 0);
  if (r == ncclSuccess) cudaMemcpyAsync(oks.data(), d_ok, 4 * G, cudaMemcpyDeviceToHost, ctx->stream);
  const bool synced = cudaStreamSynchronize(ctx->stream) == cudaSuccess;
  cudaFree(d_all);
  if (r != ncclSuccess || !synced) return fail(ctx, GS_ERR_CUDA, "peer link: confirmation exchange failed");
  bool all_ok = true;
  for (uint32_t c = 0; c < G; ++c) all_ok &= oks[c] != 0;
  if (all_ok) { k.ready = true; k.asset = as; k.sort_frames = 0; }
  return GS_OK;
}

void peer_link_release(GsGroup *g) {
  PeerLink &k = g->link;
  if (!g->m.empty() && g->m[0].ctx) { cudaSetDevice(g->m[0].ctx->device); cudaStreamSynchronize(g->m[0].ctx->stream); }
  for (int i = 0; i < k.n_opened; ++i) if (k.opened[i]) cudaIpcCloseMemHandle(k.opened[i]);
  k.n_opened = 0;
  cudaFree(k.flags); cudaFree(k.d_done);
  k.flags = k.d_done = nullptr;
  k.ready = false;
  cudaGetLastError();
}

void balance_rows(const uint32_t *cost, uint32_t rows, uint32_t parts, uint32_t *bounds) {
  // every row also carries a fixed share (its tiles are launched, its pixels stored) so that empty rows are not free
  uint64_t sum = 0;
  for (uint32_t r = 0; r < rows; ++r) sum += cost ? cost[r] : 0u;
  const uint64_t base = sum / ((uint64_t)rows * 8u) + 1u;
  const uint64_t total = sum + base * rows;
  uint64_t acc = 0;
  uint32_t r = 0;
  bounds[0] = 0;
  for (uint32_t p = 1; p < parts; ++p) {
    const uint64_t target = total * p / parts;
    while (r < rows) {
      const uint64_t w = (cost ? cost[r] : 0u) + base;
      if (acc + w / 2 >= target) break;   // a row goes to the part its midpoint falls into
      acc += w;
      ++r;
    }
    bounds[p] = r;
  }
  bounds[parts] = rows;
}

float tev_ms(Member &mb, int a, int b) {
  float ms = 0.0f;
  if (cudaEventElapsedTime(&ms, mb.tev[a], mb.tev[b]) != cudaSuccess) { cudaGetLastError(); return 0.0f; }
  return ms;
}

}  // namespace

extern "C" {

int gs_group_balance_rows(const uint32_t *row_cost, uint32_t rows, uint32_t parts, uint32_t *bounds_out) {
  if (!bounds_out || rows == 0 || parts == 0 || parts > GS_GROUP_MAX_GPUS) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "bad rows/parts");
  balance_rows(row_cost, rows, parts, bounds_out);
  return GS_OK;
}

int gs_group_unique_id(void *id_out) {
  if (!id_out) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null id");
  if (!nccl_api().ok()) return fail(nullptr, GS_ERR_NOT_READY, "libnccl.so.2 not found: a multi-process group needs NCCL");
  ncclUniqueId id;
  GS_NCCL_TRY(nullptr, nccl_api().GetUniqueId(&id));
  static_assert(sizeof(id) == GS_GROUP_ID_BYTES, "id size");
  memcpy(id_out, &id, sizeof(id));
  return GS_OK;
}

int gs_group_join(GsContext *ctx, uint32_t group_size, uint32_t rank, const void *id, GsGroup **out) {
  if (!ctx || !out || !id || group_size == 0 || group_size > GS_GROUP_MAX_GPUS || rank >= group_size)
    return fail(ctx, GS_ERR_INVALID_ARGUMENT, "bad group size / rank / id");
  *out = nullptr;
  if (!nccl_api().ok()) return fail(ctx, GS_ERR_NOT_READY, "libnccl.so.2 not found: a multi-process group needs NCCL");
  GsGroup *g = new (std::nothrow) GsGroup();
  if (!g) return fail(ctx, GS_ERR_OUT_OF_MEMORY, "host allocation failed");
  g->size = group_size;
  g->use_nccl = true;
  g->m.resize(1);
  g->m[0].ctx = ctx;
  g->m[0].rank = rank;
  int rc = member_init(g->m[0]);
  if (rc == GS_OK) {
    ncclUniqueId nid;
    memcpy(&nid, id, sizeof(nid));
    ncclResult_t r = nccl_api().CommInitRank(&g->m[0].comm, (int)group_size, nid, (int)rank);
    if (r != ncclSuccess) rc = fail_nccl(ctx, r, "ncclCommInitRank");
  }
  if (rc != GS_OK) { gs_group_destroy(g); return rc; }
  *out = g;
  return GS_OK;
}

int gs_group_create(const int *devices, uint32_t n, uint32_t flags, GsGroup **out) {
  if (!devices || !out || n == 0 || n > GS_GROUP_MAX_GPUS) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "bad device list");
  *out = nullptr;
  bool distinct = true;
  for (uint32_t i = 0; i < n; ++i)
    for (uint32_t j = 0; j < i; ++j) distinct &= devices[i] != devices[j];
  if (!distinct && !(flags & GS_GROUP_EMULATE)) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "a device is listed twice (only GS_GROUP_EMULATE allows that)");
  GsGroup *g = new (std::nothrow) GsGroup();
  if (!g) return fail(nullptr, GS_ERR_OUT_OF_MEMORY, "host allocation failed");
  g->size = n;
  g->emulate = (flags & GS_GROUP_EMULATE) != 0;
  g->m.resize(n);
  int rc = GS_OK;
  for (uint32_t i = 0; i < n && rc == GS_OK; ++i) {
    GsContext *ctx = nullptr;
    rc = gs_create(devices[i], nullptr, &ctx);
    if (rc != GS_OK) break;
    g->m[i].ctx = ctx;
    g->m[i].own_ctx = true;
    g->m[i].rank = i;
    rc = member_init(g->m[i]);
  }
  if (rc == GS_OK && !g->emulate && n > 1) {
    if (nccl_api().ok()) {
      std::vector<ncclComm_t> comms(n);
      ncclResult_t r = nccl_api().CommInitAll(comms.data(), (int)n, devices);
      if (r != ncclSuccess) rc = fail_nccl(nullptr, r, "ncclCommInitAll");
      else { for (uint32_t i = 0; i < n; ++i) g->m[i].comm = comms[i]; g->use_nccl = true; }
    } else {   // device-to-device copies between the contexts: let them go straight over NVLink
      for (uint32_t i = 0; i < n; ++i) {
        cudaSetDevice(devices[i]);
        for (uint32_t j = 0; j < n; ++j) {
          int can = 0;
          if (i != j && cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) == cudaSuccess && can) cudaDeviceEnablePeerAccess(devices[j], 0);
        }
        cudaGetLastError();
      }
    }
  }
  if (rc != GS_OK) { gs_group_destroy(g); return rc; }
  *out = g;
  return GS_OK;
}

void gs_group_destroy(GsGroup *g) {
  if (!g) return;
  peer_link_release(g);
  for (Member &mb : g->m) member_free(mb);
  delete g;
}

uint32_t gs_group_size(const GsGroup *g) { return g ? g->size : 0; }
uint32_t gs_group_local_count(const GsGroup *g) { return g ? (uint32_t)g->m.size() : 0; }
GsContext *gs_group_context(GsGroup *g, uint32_t i) { return (g && i < g->m.size()) ? g->m[i].ctx : nullptr; }

int gs_group_asset_upload(GsGroup *g, const GsAssetDesc *desc, GsAsset **assets_out) {
  if (!g || !desc || !assets_out) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null argument");
  for (size_t i = 0; i < g->m.size(); ++i) assets_out[i] = nullptr;
  for (size_t i = 0; i < g->m.size(); ++i) {
    int rc = gs_asset_upload(g->m[i].ctx, desc, &assets_out[i]);
    if (rc == GS_OK) { cudaSetDevice(g->m[i].ctx->device); rc = member_asset(g->m[i], assets_out[i]); }
    if (rc != GS_OK) {
      for (size_t j = 0; j <= i; ++j) { gs_asset_destroy(assets_out[j]); assets_out[j] = nullptr; }
      return rc;
    }
  }
  return GS_OK;
}

int gs_group_sync(GsGroup *g) {
  if (!g) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null group");
  int rc = GS_OK;
  for (Member &mb : g->m) {
    cudaSetDevice(mb.ctx->device);
    cudaError_t e = cudaStreamSynchronize(mb.aux);
    if (e == cudaSuccess) e = cudaStreamSynchronize(mb.xfer);
    if (e != cudaSuccess && rc == GS_OK) rc = fail_cuda(mb.ctx, e, "cudaStreamSynchronize(aux/xfer)", __FILE__, __LINE__);
    mb.image_pending = false;
    if (g->link.ready && rc == GS_OK) {   // a peer that never delivered its slab made k_wait_slabs give up: the frame is void
      uint32_t bad = 0;
      e = cudaMemcpy(&bad, g->link.flags + g->size, 4, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) rc = fail_cuda(mb.ctx, e, "cudaMemcpy(peer flags)", __FILE__, __LINE__);
      else if (bad) rc = fail(mb.ctx, GS_ERR_CUDA, "peer-to-peer order exchange timed out: a process of the group did not deliver its slab");
    }
    const int r = gs_sync(mb.ctx);
    if (r != GS_OK && rc == GS_OK) rc = r;
  }
  return rc;
}

int gs_group_frame(GsGroup *g, GsAsset *const *assets, const GsFrameParams *fp, const GsRenderOptions *opt_in, int do_sort_flag,
                   GsImage *const *rts) {
  if (!g || !assets || !fp) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null argument");
  const uint32_t G = g->size;
  const size_t L = g->m.size();
  int rc;
  for (size_t i = 0; i < L; ++i) {
    if (!assets[i]) return fail(g->m[i].ctx, GS_ERR_INVALID_ARGUMENT, "null asset");
    if ((rc = check_params(g->m[i].ctx, assets[i], fp))) return rc;
    if (assets[i]->av.n != assets[0]->av.n) return fail(g->m[i].ctx, GS_ERR_INVALID_ARGUMENT, "members hold different assets");
  }
  const FrameConsts fc = make_frame_consts(fp);
  const uint32_t W = (uint32_t)fp->screen_w, H = (uint32_t)fp->screen_h, N = assets[0]->av.n;
  const uint32_t rows = (H + kTile - 1) / kTile, ntx = (W + kTile - 1) / kTile;
  GsRenderOptions base;
  memset(&base, 0, sizeof(base));
  base.blend_mode = opt_in ? opt_in->blend_mode : (uint32_t)GS_BLEND_FP16_ROP;
  if (base.blend_mode > GS_BLEND_FP32) return fail(g->m[0].ctx, GS_ERR_INVALID_ARGUMENT, "bad blend mode");
  uint32_t fmt = GS_PIX_RGBA16F;
  for (size_t i = 0; i < L; ++i) if (rts && rts[i]) { fmt = rts[i]->format; break; }

  // ---- row ranges of this frame: from the row costs measured two frames ago (the last ones every GPU surely holds) ----
  if (g->hist_w != W || g->hist_h != H) { g->hist_w = W; g->hist_h = H; g->hist_frames = 0; }
  const int slot = (int)(g->hist_frames & 1u);
  for (Member &mb : g->m) { cudaSetDevice(mb.ctx->device); if ((rc = member_rows(mb, rows))) return rc; }
  if (G == 1) { g->bounds[0] = 0; g->bounds[1] = rows; }
  else if (g->hist_frames >= 2) {
    Member &m0 = g->m[0];
    GS_CUDA_TRY(m0.ctx, cudaEventSynchronize(m0.ev_cost[slot]));   // written by frame hist_frames - 2: long done
    balance_rows(m0.h_row_cost[slot], rows, G, g->bounds);
  } else {
    balance_rows(nullptr, rows, G, g->bounds);
  }

  const bool timing = g->m[0].ctx->timing;
  g->timed = timing;
  GsNvtxRange nvtx_frame("GaussianSplat.GroupFrame");
  // ---- phase A: distances + slab table on the context stream; view-calc on the second stream --------------------------
  for (size_t i = 0; i < L; ++i) {
    Member &mb = g->m[i];
    GsContext *ctx = mb.ctx;
    GsAsset *as = assets[i];
    GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if ((rc = member_asset(mb, as))) return rc;
    for (int e = 0; e < EV_COUNT; ++e) ctx->ev_valid[e] = false;
    GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_begin, ctx->stream));
    if (timing) cudaEventRecord(mb.tev[GT_BEGIN], ctx->stream);
    if (do_sort_flag) {
      SlabArgs sl;
      memset(&sl, 0, sizeof(sl));
      sl.count = G; sl.index = mb.rank; sl.order_prev = as->order; sl.mask = as->slab_mask; sl.group_bits = as->slab_group_bits; sl.info = mb.d_info;
      for (uint32_t j = 0; j + 1 < G; ++j) sl.qpos[j] = (uint32_t)(((uint64_t)N * (j + 1)) / G);
      GS_CUDA_TRY(ctx, cudaMemsetAsync(ctx->sort.ghist, 0, 4 * 256 * 4, ctx->stream));
      GS_CUDA_TRY(ctx, cudaMemsetAsync(mb.d_info, 0, 2 * kMaxSlabs * 4, ctx->stream));
      launch_calc_distances(as->av, fc, as->key_table, ctx->sort.ghist, ctx->stream, &sl);
      ctx->launches += 1;
      if (G > 1) {
        GS_CUDA_TRY(ctx, cudaMemcpyAsync(mb.h_info, mb.d_info, 2 * kMaxSlabs * 4, cudaMemcpyDeviceToHost, ctx->stream));
        GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_info, ctx->stream));
      }
    }
    if (timing) cudaEventRecord(mb.tev[GT_DIST], ctx->stream);
    // View-calc reads nothing the sort writes: it runs on the helper stream (lowest priority), right behind the distance
    // kernel (started together, its 24 k blocks crowd the distance kernel out: 63 instead of 32 us at N = 8), and fills
    // whatever the sort chain leaves idle: the host's wait for the slab table, the sort's tails and the exchange
    cudaEvent_t after = mb.ev_begin;
    if (do_sort_flag) { GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_produced, ctx->stream)); after = mb.ev_produced; }
    GsRenderOptions opt = base;
    opt.row_begin = g->bounds[mb.rank]; opt.row_end = g->bounds[mb.rank + 1];
    if (opt.row_end > opt.row_begin || G == 1) {
      if (G == 1) opt.row_begin = opt.row_end = 0;
      GS_CUDA_TRY(ctx, cudaStreamWaitEvent(mb.aux, after, 0));
      if (timing) cudaEventRecord(mb.tev[GT_V0], mb.aux);
      if ((rc = do_view(ctx, as, fp, fc, true, opt, mb.aux))) return rc;
      if (timing) cudaEventRecord(mb.tev[GT_V1], mb.aux);
      GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_view, mb.aux));
    }
  }

  // ---- slab sizes: the one host wait of the frame (the GPUs are busy with view-calc) ----------------------------------
  if (do_sort_flag) {
    if (G == 1) { g->slab_off[0] = 0; g->slab_off[1] = N; g->slab_cnt[0] = N; }
    for (size_t i = 0; i < L && G > 1; ++i) {
      Member &mb = g->m[i];
      GS_CUDA_TRY(mb.ctx, cudaSetDevice(mb.ctx->device));
      GS_CUDA_TRY(mb.ctx, cudaEventSynchronize(mb.ev_info));
      uint32_t off[GS_GROUP_MAX_GPUS + 1];
      off[0] = 0;
      for (uint32_t c = 1; c < G; ++c) {
        const uint32_t ge = mb.h_info[kMaxSlabs + c - 1];   // #{key >= splitter c-1 (ascending)}
        if (ge > N) return fail(mb.ctx, GS_ERR_CUDA, "slab table corrupt");
        off[c] = N - ge;
      }
      off[G] = N;
      for (uint32_t c = 0; c < G; ++c) if (off[c + 1] < off[c]) return fail(mb.ctx, GS_ERR_CUDA, "slab table not monotone");
      if (i == 0) memcpy(g->slab_off, off, sizeof(uint32_t) * (G + 1));
      else if (memcmp(g->slab_off, off, sizeof(uint32_t) * (G + 1)) != 0) return fail(mb.ctx, GS_ERR_CUDA, "members disagree on the slab table");
    }
    for (uint32_t c = 0; c < G; ++c) g->slab_cnt[c] = g->slab_off[c + 1] - g->slab_off[c];

    // ---- phase C: compact my slab out of last frame's order, sort it into its place of the new order ------------------
    GsNvtxRange nvtx_sort("GaussianSplat.Sort");
    // equal slots + one all-gather while the slabs are reasonably balanced (they are after the first frame); a frame whose
    // largest slab is far above N/G exchanges the exact sizes in place instead (no G x cap staging)
    uint32_t cap = 0;
    for (uint32_t c = 0; c < G; ++c) cap = g->slab_cnt[c] > cap ? g->slab_cnt[c] : cap;
    cap = (cap + 3u) & ~3u;
    // one process per GPU: slabs go peer to peer (set up on the first sorted frame)
    if (G > 1 && g->use_nccl && L == 1 && !g->link.tried) { if ((rc = peer_link_setup(g, assets[0]))) return rc; }
    const bool use_p2p = G > 1 && L == 1 && g->link.ready && g->link.asset == assets[0];
    uint32_t *p2p_new = nullptr;
    int p2p_idx = 0;
    if (use_p2p) {   // the two order buffers alternate: last frame's order is read, the other one is assembled
      p2p_idx = assets[0]->order == g->link.buf[0] ? 1 : 0;
      p2p_new = g->link.buf[p2p_idx];
    }
    const bool use_gather = !use_p2p && G > 1 && (uint64_t)cap * G <= (uint64_t)N + (uint64_t)N / 2 + 64u * G;
    if (use_gather) {
      for (size_t i = 0; i < L; ++i) {
        Member &mb = g->m[i];
        const size_t need = (size_t)cap * G;
        if (need > mb.gather_words) {
          GS_CUDA_TRY(mb.ctx, cudaSetDevice(mb.ctx->device));
          cudaStreamSynchronize(mb.ctx->stream);
          cudaFree(mb.d_gather);
          mb.d_gather = nullptr; mb.gather_words = 0;
          const size_t words = (size_t)N + (size_t)N / 2 + 64u * G;   // the largest staging this path ever uses
          GS_CUDA_TRY(mb.ctx, cudaMalloc(&mb.d_gather, words * 4));
          mb.gather_words = words;
        }
      }
    }
    for (size_t i = 0; i < L; ++i) {
      Member &mb = g->m[i];
      GsContext *ctx = mb.ctx;
      GsAsset *as = assets[i];
      GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
      const uint32_t cnt = g->slab_cnt[mb.rank], off = g->slab_off[mb.rank];
      if (G == 1) {
        launch_sort_pairs(as->keys, as->order, as->d_n, N, 4, 8, true, ctx->sort, ctx->stream, nullptr, as->key_table);
        ctx->launches += 4;
      } else if (cnt) {
        launch_compact_order(as->order, N, as->slab_mask, as->slab_group_bits, as->key_table, as->order_tmp, as->keys, mb.d_cmp_status, mb.d_slab_count,
                             ctx->stream);
        launch_sort_pairs(as->keys, as->order_tmp, mb.d_slab_count, cnt, 4, 8, true, ctx->sort, ctx->stream, nullptr, nullptr, true,
                          as->keys + off, use_p2p ? p2p_new + off : use_gather ? mb.d_gather + (size_t)mb.rank * cap : as->order + off);
        ctx->launches += 5;
      }
      if (use_p2p) {
        PeerLink &k = g->link;
        const uint32_t tag = ++k.sort_frames;
        PushArgs pa;
        memset(&pa, 0, sizeof(pa));
        for (uint32_t c = 0; c < G; ++c)
          if (c != mb.rank) { pa.dst[pa.npeers] = k.peer_buf[p2p_idx][c] + off; pa.flag[pa.npeers] = k.peer_flags[c] + mb.rank; ++pa.npeers; }
        k_push_slab<<<148, 512, 0, ctx->stream>>>(p2p_new + off, cnt, pa, tag, k.d_done);
        k_wait_slabs<<<1, 32, 0, ctx->stream>>>(k.flags, G, mb.rank, tag);
        ctx->launches += 2;
        // from here on the assembled buffer IS the draw order; last frame's becomes the next frame's target
        as->order_alt = as->order;
        as->order = p2p_new;
      }
      GS_CUDA_TRY(ctx, cudaGetLastError());
      if (timing) cudaEventRecord(mb.tev[GT_SORT], ctx->stream);
    }
    if (G > 1) {
      std::vector<uint8_t *> bufs(L);
      size_t off[GS_GROUP_MAX_GPUS], cnt[GS_GROUP_MAX_GPUS];
      for (uint32_t c = 0; c < G; ++c) { off[c] = (size_t)g->slab_off[c] * 4; cnt[c] = (size_t)g->slab_cnt[c] * 4; }
      if (use_p2p) {
        // delivered by k_push_slab / awaited by k_wait_slabs above
      } else if (use_gather) {
        for (size_t i = 0; i < L; ++i) bufs[i] = reinterpret_cast<uint8_t *>(g->m[i].d_gather);
        if ((rc = exchange_allgather(g, bufs.data(), (size_t)cap * 4, cnt))) return rc;
        for (size_t i = 0; i < L; ++i) {   // slot c's ids -> their place in the order: G device copies (a copy kernel that found
          Member &mb = g->m[i];            // each element's slab took 41 us for the 24.5 MB of cfg2; the copy engine takes ~10)
          GS_CUDA_TRY(mb.ctx, cudaSetDevice(mb.ctx->device));
          for (uint32_t c = 0; c < G; ++c)
            if (g->slab_cnt[c])
              GS_CUDA_TRY(mb.ctx, cudaMemcpyAsync(assets[i]->order + g->slab_off[c], mb.d_gather + (size_t)c * cap, (size_t)g->slab_cnt[c] * 4,
                                                  cudaMemcpyDeviceToDevice, mb.ctx->stream));
        }
      } else {
        for (size_t i = 0; i < L; ++i) bufs[i] = reinterpret_cast<uint8_t *>(assets[i]->order);
        if ((rc = exchange_begin(g)) || (rc = exchange_add(g, bufs.data(), off, cnt)) || (rc = exchange_end(g))) return rc;
      }
    }
  }
  if (timing) for (Member &mb : g->m) { cudaSetDevice(mb.ctx->device); if (!do_sort_flag) cudaEventRecord(mb.tev[GT_SORT], mb.ctx->stream); cudaEventRecord(mb.tev[GT_ORDER], mb.ctx->stream); }

  // ---- phase D: bin + composite my rows, then exchange rows and row costs ---------------------------------------------
  std::vector<uint8_t *> img(L), costs(L);
  std::vector<uint32_t> pitches(L);
  for (size_t i = 0; i < L; ++i) {
    Member &mb = g->m[i];
    GsContext *ctx = mb.ctx;
    GsAsset *as = assets[i];
    GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    GsImage *rt = rts ? rts[i] : nullptr;
    uint32_t pitch = W * pix_bytes(fmt);
    void *d_rt = nullptr;
    if (rt) {
      uint32_t p = 0;
      if ((rc = image_ok(ctx, rt, W, H, &p))) return rc;
      if (rt->format != fmt) return fail(ctx, GS_ERR_INVALID_ARGUMENT, "members' images differ in pixel format");
      if (rt->memory == GS_MEM_DEVICE) { d_rt = rt->data; pitch = p; }
    }
    if (!d_rt) {
      if (mb.rt_bytes < (size_t)pitch * H) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(mb.rt_scratch);
        mb.rt_scratch = nullptr; mb.rt_bytes = 0;
        GS_CUDA_TRY(ctx, cudaMalloc(&mb.rt_scratch, (size_t)pitch * H));
        mb.rt_bytes = (size_t)pitch * H;
      }
      d_rt = mb.rt_scratch;
    }
    img[i] = reinterpret_cast<uint8_t *>(d_rt);
    pitches[i] = pitch;
    costs[i] = reinterpret_cast<uint8_t *>(mb.d_row_cost);
    GsRenderOptions opt = base;
    opt.row_begin = g->bounds[mb.rank]; opt.row_end = g->bounds[mb.rank + 1];
    if (opt.row_end > opt.row_begin || G == 1) {
      if (G == 1) opt.row_begin = opt.row_end = 0;
      GS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, mb.ev_view, 0));
      // the previous frame's row exchange (transfer stream) may still be filling this image: composite only after it
      if (mb.image_pending) GS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, mb.ev_image, 0));
      if (timing) cudaEventRecord(mb.tev[GT_VIEWWAIT], ctx->stream);
      rec(ctx, EV_VIEW1);
      if ((rc = bind_depth(ctx, fp, ctx->stream))) return rc;
      if ((rc = do_render(ctx, as, fc, opt, d_rt, pitch, fmt))) return rc;
      ctx->launches += 1;   // k_row_costs, launched on the transfer stream below
    } else if (timing) {
      cudaEventRecord(mb.tev[GT_VIEWWAIT], ctx->stream);
    }
    if (timing) cudaEventRecord(mb.tev[GT_RASTER], ctx->stream);
  }
  // The exchange of the composited rows (and of their measured costs) goes to the transfer stream: it needs no SM to speak
  // of, and the next frame's distance / sort chain does not depend on it, so the two overlap; the next frame's compositor
  // waits for it (above), gs_group_sync / a host image complete it.
  for (size_t i = 0; i < L; ++i) {
    Member &mb = g->m[i];
    GS_CUDA_TRY(mb.ctx, cudaSetDevice(mb.ctx->device));
    GS_CUDA_TRY(mb.ctx, cudaEventRecord(mb.ev_raster, mb.ctx->stream));
    GS_CUDA_TRY(mb.ctx, cudaStreamWaitEvent(mb.xfer, mb.ev_raster, 0));
    if (g->bounds[mb.rank + 1] > g->bounds[mb.rank] || G == 1)   // the measured cost of my rows, for the balancer two frames on
      launch_row_costs(mb.ctx->bin.tile_cost, ntx, g->bounds[mb.rank], g->bounds[mb.rank + 1], mb.d_row_cost, mb.xfer);
  }
  if (G > 1) {
    size_t off[GS_GROUP_MAX_GPUS], cnt[GS_GROUP_MAX_GPUS], coff[GS_GROUP_MAX_GPUS], ccnt[GS_GROUP_MAX_GPUS];
    for (size_t i = 1; i < L; ++i) if (pitches[i] != pitches[0]) return fail(g->m[i].ctx, GS_ERR_INVALID_ARGUMENT, "members' images differ in row pitch");
    for (uint32_t c = 0; c < G; ++c) {
      const uint32_t y0 = min(g->bounds[c] * kTile, H), y1 = min(g->bounds[c + 1] * kTile, H);
      off[c] = (size_t)y0 * pitches[0]; cnt[c] = (size_t)(y1 - y0) * pitches[0];
      coff[c] = (size_t)g->bounds[c] * 4; ccnt[c] = (size_t)(g->bounds[c + 1] - g->bounds[c]) * 4;
    }
    if ((rc = exchange_begin(g)) || (rc = exchange_add(g, img.data(), off, cnt, true)) || (rc = exchange_add(g, costs.data(), coff, ccnt, true)) ||
        (rc = exchange_end(g)))
      return rc;
  }
  bool host_out = false;
  for (size_t i = 0; i < L; ++i) {
    Member &mb = g->m[i];
    GsContext *ctx = mb.ctx;
    GS_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (timing) cudaEventRecord(mb.tev[GT_IMAGE], mb.xfer);
    GS_CUDA_TRY(ctx, cudaMemcpyAsync(mb.h_row_cost[slot], mb.d_row_cost, (size_t)rows * 4, cudaMemcpyDeviceToHost, mb.xfer));
    GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_cost[slot], mb.xfer));
    GsImage *rt = rts ? rts[i] : nullptr;
    if (rt && rt->memory != GS_MEM_DEVICE) {
      const uint32_t hp = rt->row_pitch_bytes ? rt->row_pitch_bytes : W * pix_bytes(fmt);
      GS_CUDA_TRY(ctx, cudaMemcpy2DAsync(rt->data, hp, img[i], pitches[i], (size_t)W * pix_bytes(fmt), H, cudaMemcpyDeviceToHost, mb.xfer));
      host_out = true;
    }
    GS_CUDA_TRY(ctx, cudaEventRecord(mb.ev_image, mb.xfer));
    mb.image_pending = true;
    // the row-cost vector is rewritten by the next frame's k_row_costs on the context stream: that must follow this exchange too
    // (it does: k_row_costs runs after the compositor, which waits for ev_image)
  }
  g->frame++;
  g->hist_frames++;
  // host images: filled by the transfer stream.  By default the call blocks until they are (like gs_frame); with
  // GS_FLAG_ASYNC_READBACK it returns now and gs_group_sync completes them -- the images must be pinned and must not be
  // reused before that (alternate two).  The next frame's compositor waits for this frame's copy before it touches the
  // device image, so no second device image is needed.
  const bool async_rb = opt_in && (opt_in->flags & GS_FLAG_ASYNC_READBACK) != 0;
  if (host_out && !async_rb) return gs_group_sync(g);
  return GS_OK;
}

int gs_group_get_stats(GsGroup *g, GsGroupStats *out) {
  if (!g || !out) return fail(nullptr, GS_ERR_INVALID_ARGUMENT, "null argument");
  memset(out, 0, sizeof(*out));
  Member &mb = g->m[0];
  GS_CUDA_TRY(mb.ctx, cudaSetDevice(mb.ctx->device));
  GS_CUDA_TRY(mb.ctx, cudaStreamSynchronize(mb.ctx->stream));
  GS_CUDA_TRY(mb.ctx, cudaStreamSynchronize(mb.aux));
  GS_CUDA_TRY(mb.ctx, cudaStreamSynchronize(mb.xfer));
  out->group_size = g->size;
  out->rank = mb.rank;
  for (uint32_t c = 0; c <= g->size; ++c) out->row_bounds[c] = g->bounds[c];
  for (uint32_t c = 0; c < g->size; ++c) out->slab_counts[c] = g->slab_cnt[c];
  if (g->timed) {
    out->distances_ms = tev_ms(mb, GT_BEGIN, GT_DIST);
    out->slab_sort_ms = tev_ms(mb, GT_DIST, GT_SORT);
    out->order_exchange_ms = tev_ms(mb, GT_SORT, GT_ORDER);
    out->view_ms = tev_ms(mb, GT_V0, GT_V1);
    float bin = 0.0f;
    if (mb.ctx->ev_valid[EV_VIEW1] && mb.ctx->ev_valid[EV_BIN1] && cudaEventElapsedTime(&bin, mb.ctx->ev[EV_VIEW1], mb.ctx->ev[EV_BIN1]) != cudaSuccess) { cudaGetLastError(); bin = 0.0f; }
    out->bin_ms = bin;
    out->raster_ms = tev_ms(mb, GT_VIEWWAIT, GT_RASTER) - bin;
    out->image_exchange_ms = tev_ms(mb, GT_RASTER, GT_IMAGE);
    out->total_ms = tev_ms(mb, GT_BEGIN, GT_IMAGE);
  }
  return GS_OK;
}

}  // extern "C"
