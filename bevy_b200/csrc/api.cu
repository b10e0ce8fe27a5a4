// api.cu -- host runtime + C ABI of libb200vis.so (include/b200vis.h).
//
// Owns the SoA device mirror of the ECS columns, the execution plan built from the hierarchy
// (tiles and passes), the per-frame constants, and the stream every stage is issued on.
// There is NO CPU fallback: without a CUDA device b200vis_create fails with B200VIS_ERR_CUDA.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include <chrono>
#include <cuda_runtime.h>
#include <dlfcn.h>

#include "../../include/b200vis.h"
#include "device_types.cuh"
#include "host_view.hpp"
#include "kernels.cuh"

using namespace b200vis;

static thread_local std::string g_create_error;

// ---- NCCL through dlopen: no link-time dependency, and the process keeps ONE NCCL (the one torch already loaded) ----
namespace {
struct NcclId { char b[128]; };   // ncclUniqueId (passed BY VALUE to ncclCommInitRank)
struct NcclApi {
    using Id = NcclId;
    void *lib = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (lib) return true;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return false;
        GetUniqueId = reinterpret_cast<decltype(GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
        CommInitRank = reinterpret_cast<decltype(CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
        AllGather = reinterpret_cast<decltype(AllGather)>(dlsym(lib, "ncclAllGather"));
        CommDestroy = reinterpret_cast<decltype(CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
        GetErrorString = reinterpret_cast<decltype(GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
        return GetUniqueId && CommInitRank && AllGather && CommDestroy && GetErrorString;
    }
};
NcclApi g_nccl;
constexpr int kNcclUint32 = 3;   // ncclUint32 in nccl.h's ncclDataType_t
}

struct b200vis_ctx {
    b200vis_config cfg{};
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // Frame pipelining: the latency-bound tail of frame f (visible-list expansion, cluster kernels) runs on a side
    // stream while frame f+1's tile pass already runs on the main stream (masks / counters / constants are
    // double or triple buffered by frame number).
    cudaStream_t side_stream = nullptr;
    cudaStream_t clus_stream = nullptr; cudaEvent_t ev_clus = nullptr;   // pipelined frames: the cluster branch of the tail (exchange -> cluster kernel) runs beside the list expansion
    cudaEvent_t ev_tile = nullptr, ev_side[3] = {nullptr, nullptr, nullptr}, ev_expand[2] = {nullptr, nullptr}, ev_pub = nullptr;
    bool pub_pending = false;           // a publish_visible copy is in flight on the side stream
    bool pipeline = true, side_pending = false;
    // a frame whose tail was started (expand + cluster assign on the side stream) but whose CLUSTER_LISTS stage is
    // still to come in a later b200vis_run call (multi-GPU: the host all-gathers the slabs in between)
    bool tail_open = false; uint32_t open_frame = 0; const FrameConsts *open_fc = nullptr;
    // light blocks [3 frame slots]: float4 snap[cap32] | float range[cap32] | uint64 layers[cap32] (cap32 = cl.max_lights).  The
    // snap part is what the tile pass fills per frame; with several GPUs the whole block is what one all-gather exchanges
    uint8_t *d_lrec = nullptr, *d_lrec_all = nullptr; size_t lrec_bytes = 0;
    float4 *light_snap_slot(uint32_t slot) const { return reinterpret_cast<float4 *>(d_lrec + (size_t)slot * lrec_bytes); }
    uint32_t *d_tag_flag = nullptr;     // 1 if every light row carries its ordinal (k_tag_lights)
    uint32_t *d_light_ord = nullptr;    // [max_entities] light ordinal per row, 0xFFFFFFFF = not a light (rewritten on set_lights)
    bool lights_tag_dirty = true, lights_tagged = false;
    std::string err;

    uint32_t n = 0;                 // current row count
    Rows rows{};                    // device SoA (capacity cfg.max_entities)
    uint64_t *d_layers_ext = nullptr; bool have_layers_ext = false; uint64_t view_layers_ext[kMaxViews][3] = {};   // RenderLayers blocks 1..3
    uint32_t *d_parent = nullptr; uint64_t *d_layers = nullptr; uint32_t *d_range = nullptr;
    uint32_t *d_rank = nullptr, *d_row_of_rank = nullptr; uint8_t *d_dirty = nullptr;
    bool have_layers = false, have_range = false, rank_identity = true, topology_set = false;
    bool bounds_set = false;

    // plan
    Tile *d_tiles = nullptr; uint32_t tiles_cap = 0;
    WarpTile *d_wtiles = nullptr; uint8_t *d_sched = nullptr; uint32_t *d_wtopo = nullptr;   // k_tile_warp's view of the plan
    uint32_t *d_tile_counter = nullptr;
    uint32_t *d_tile_ticket = nullptr; uint32_t tile_ticket_base = 0;   // dynamic tile hand-out of the default kernel: never reset, the host tracks the base
    std::vector<uint32_t> pass_begin;   // tile index ranges per pass: [pass_begin[p], pass_begin[p+1])
    std::vector<uint32_t> pass_small;   // the first pass_small[p] tiles of pass p have <= 32 rows (B200VIS_SPLIT_DEEP_TILES)
    std::vector<uint8_t> pass_named;    // every tile of pass p is flat or walks with named level barriers (Tile::lvl_warps): the tile kernel may let a CTA's warps drift a tile apart
    int static_opt = 1;

    // per-frame constants
    // The "frame blob": FrameConsts followed by the packed per-view plane tables and z thresholds.
    // Setters edit the host working copy; run() packs it into the next pinned ring slot and issues
    // ONE async H2D copy, so per-frame constant updates never block on the stream.
    FrameConsts consts{};               // host working copy
    std::vector<float> tab_x[kMaxViews], tab_y[kMaxViews], tab_z[kMaxViews], tab_thr[kMaxViews];
    static constexpr int kRing = 4;
    uint8_t *h_ring[kRing] = {nullptr, nullptr, nullptr, nullptr};   // pinned
    cudaEvent_t ring_ev[kRing] = {nullptr, nullptr, nullptr, nullptr};
    int ring_next = 0;
    size_t blob_cap = 0;
    uint8_t *d_blob2[3] = {nullptr, nullptr, nullptr};   // live-mode device blobs, slot = frame % 3
    uint8_t *d_blob = nullptr;          // the one the current frame uses
    FrameConsts *d_consts = nullptr;    // == d_blob
    bool consts_dirty = true;
    size_t blob_used = 0;               // bytes of the last packed blob
    struct Recorded { FrameConsts host; uint8_t *dev; size_t bytes; };
    std::vector<Recorded> recorded;     // b200vis_record_frame_constants
    int replay_slot = -1;               // >= 0: b200vis_run reads recorded[replay_slot] instead of the live copy
    // optional per-stage timing (b200vis_set_profiling)
    bool profiling = false;
    static constexpr int kProfFrames = 256;
    cudaEvent_t (*prof_ev)[6] = nullptr;   // [kProfFrames][6]: main 0,1 (tile); side 2,3,4 (expand, cluster); created on first use
    int prof_count = 0;

    // visible set
    VisibleBufs vis{};
    DiffBufs diff{}; bool diff_on = false;      // SURVEY 8(f) N1 (b200vis_enable_visible_diff)
    uint32_t *diff_sink_rows_d = nullptr, *diff_sink_counts_d = nullptr; uint32_t diff_sink_cap = 0;
    BindingBufs bind{}; uint32_t *d_bind_map = nullptr; uint32_t bind_map_cap = 0;   // SURVEY 8(f) N2 (b200vis_set_cluster_bindings)
    // SURVEY 8(f) N3: shadow-view culling (b200vis_set_shadow_lights / b200vis_run_shadow_culling)
    ShadowBufs shadow{}; ShadowLight *d_shadow_lights = nullptr; uint8_t *d_caster = nullptr;
    uint32_t shadow_cap_lights = 0, shadow_cap_list = 0; std::vector<ShadowLight> h_shadow;
    // SURVEY 8(f) N4: VisibilityRange columns + range views; Visibility column + the rows the last propagate wrote
    float2 *d_range_se = nullptr; uint8_t *d_range_ua = nullptr; float4 *d_range_views = nullptr; uint32_t n_range_views = 0;
    uint8_t *d_visibility = nullptr, *d_iv_changed = nullptr; bool iv_ran = false;
    DevStats *d_stats = nullptr; DevStats *h_stats = nullptr;   // h pinned
    uint32_t frame = 0, parity = 0;

    // lights + clusters
    std::vector<uint32_t> h_light_row; std::vector<float> h_light_range;   // host copies (b200vis_set_shadow_lights resolves ordinals)
    std::vector<uint64_t> h_light_layers;                                  // empty = default layer (the light blocks are rebuilt from these)
    Lights lights{}; uint32_t *d_light_row = nullptr; float *d_light_range = nullptr; uint64_t *d_light_layers = nullptr;
    ClusterBufs cl{}; uint32_t *d_slab = nullptr; void *ext_send = nullptr, *ext_recv = nullptr;
    size_t slab_bytes = 0;
    // clusterable objects (b200vis_set_clusterable_objects): cluster ordinals [lights.n, lights.n + h_obj_kind.size())
    std::vector<uint8_t> h_obj_kind; std::vector<float> h_obj_range; std::vector<uint64_t> h_obj_layers;
    uint32_t *d_obj_row = nullptr;      // [max_lights] object j's row
    uint8_t *d_ord_kind = nullptr;      // [cl.max_lights] kind of every ordinal (0 = point light), rewritten when an ordinal moves
    uint32_t n_objects() const { return (uint32_t)h_obj_kind.size(); }

    // result sink (mapped pinned host memory written by publish kernels)
    b200vis_result_sink sink{}; bool have_sink = false;
    uint32_t *sink_rows_d = nullptr, *sink_off_d = nullptr, *sink_idx_d = nullptr, *sink_stats_d = nullptr;
    uint8_t *sink_cls_d = nullptr; uint8_t *d_cls = nullptr;   // VisibilityClass masks: sink alias, per-row column

    b200vis_column_sinks colsink{}; bool have_colsink = false;          // b200vis_set_column_sinks (device aliases below)
    float *col_gt_d = nullptr; uint32_t *col_gt_bits_d = nullptr, *col_vv_bits_d = nullptr; uint8_t *col_vv_d = nullptr;
    uint8_t *d_vv_shadow = nullptr;     // what the host ViewVisibility column holds (0xFF = unknown)
    bool gt_aos_valid = false;
    bool step_defers_stats = false;     // inside b200vis_step: the CULL run leaves the sink's stats block to the CLUSTER run
    float *d_gt_aos = nullptr;          // dense write-back: the GlobalTransform column in the host's layout, copied by the DMA engine
    uint32_t last_gt_changed = 0;       // Changed<GlobalTransform> rows of the last frame whose statistics the host has seen
    double step_t[6] = {0, 0, 0, 0, 0, 0}; uint64_t step_n = 0;   // B200VIS_STEP_TRACE: host time per phase of b200vis_step
    void *nccl_comm = nullptr;          // b200vis_comm_init
    uint32_t *d_gather = nullptr;       // [world][slab] when the library owns the exchange
    // peer-memory exchange (b200vis_p2p_export / _import): [2][world][slab] + flags [2][world], mapped into every rank
    uint32_t *d_xbuf = nullptr; size_t xbuf_flag_offset = 0; void *peer_map[8] = {}; bool peer_ipc[8] = {}; bool p2p_ready = false;
    uint32_t *d_push_done = nullptr;
    b200vis_cluster_feedback auto_fb[kMaxViews]{};   // b200vis_step: last frame's Clusters feedback

    // staging for AoS <-> SoA conversion
    uint8_t *d_stage = nullptr; size_t stage_bytes = 0;
    uint8_t *h_stage = nullptr;         // pinned, same size (downloads)
};

static int32_t fail(b200vis_ctx *c, int32_t code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}
#define CU(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? B200VIS_ERR_OUT_OF_MEMORY : B200VIS_ERR_CUDA, \
                        "%s failed: %s", #call, cudaGetErrorString(e_));                                \
    } while (0)

template <typename T>
static cudaError_t dalloc(T **p, size_t count) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) e = cudaMemset(*p, 0, std::max<size_t>(count, 1) * sizeof(T));
    return e;
}

extern "C" int32_t b200vis_abi_version(void) { return B200VIS_ABI_VERSION; }
extern "C" uint64_t b200vis_kernel_launch_count(void) { return kernel_launch_count(); }
extern "C" void b200vis_struct_sizes(uint32_t out[6]) {
    out[0] = sizeof(b200vis_config); out[1] = sizeof(b200vis_view); out[2] = sizeof(b200vis_cluster_view);
    out[3] = sizeof(b200vis_frame_stats); out[4] = sizeof(b200vis_cluster_config); out[5] = sizeof(b200vis_cluster_feedback);
}

extern "C" const char *b200vis_last_error(const b200vis_ctx *ctx) {
    return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" void b200vis_destroy(b200vis_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    Rows &r = ctx->rows;
    void *dev[] = {r.trsA, r.trsB, r.trsC, r.gt0, r.gt1, r.gt2, r.bndA, r.bndB, r.flags, r.state, r.topo,
                   ctx->d_parent, ctx->d_layers, ctx->d_range, ctx->d_rank, ctx->d_row_of_rank, ctx->d_dirty,
                   ctx->d_layers_ext, ctx->d_vv_shadow, ctx->d_gt_aos, ctx->d_tiles, ctx->d_wtiles, ctx->d_sched, ctx->d_wtopo, ctx->d_tile_counter, ctx->d_tile_ticket, ctx->d_blob2[0], ctx->d_blob2[1], ctx->d_blob2[2], ctx->d_lrec, ctx->d_lrec_all, ctx->d_tag_flag, ctx->d_light_ord,
                   ctx->vis.mask, ctx->vis.chunk_count, ctx->vis.lists, ctx->vis.classes, ctx->d_cls, ctx->d_stats, ctx->d_light_row,
                   ctx->d_light_range, ctx->d_light_layers, ctx->d_slab, ctx->cl.offsets, ctx->cl.indices, ctx->d_stage,
                   ctx->diff.prev, ctx->diff.words, ctx->diff.chunk, ctx->diff.lists, ctx->diff.count,
                   ctx->bind.oc, ctx->bind.il, ctx->bind.count, ctx->d_bind_map,
                   ctx->d_range_se, ctx->d_range_ua, ctx->d_range_views, ctx->d_visibility, ctx->d_iv_changed,
                   ctx->d_shadow_lights, ctx->d_caster, ctx->shadow.mask, ctx->shadow.chunk_count, ctx->shadow.lists,
                   ctx->shadow.count, ctx->shadow.active, ctx->d_obj_row, ctx->d_ord_kind};
    for (void *p : dev) if (p) cudaFree(p);
    for (int i = 0; i < b200vis_ctx::kRing; ++i) {
        if (ctx->h_ring[i]) cudaFreeHost(ctx->h_ring[i]);
        if (ctx->ring_ev[i]) cudaEventDestroy(ctx->ring_ev[i]);
    }
    if (ctx->prof_ev) {
        for (int i = 0; i < b200vis_ctx::kProfFrames; ++i) for (cudaEvent_t e : ctx->prof_ev[i]) if (e) cudaEventDestroy(e);
        delete[] ctx->prof_ev;
    }
    if (ctx->h_stats) cudaFreeHost(ctx->h_stats);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    if (ctx->step_n && getenv("B200VIS_STEP_TRACE"))
        fprintf(stderr, "[b200vis_step] %llu steps, host us/step: upload %.1f  frusta %.1f  run(prop|cull) %.1f  cluster prologue %.1f  run(cluster) %.1f  wait %.1f\n",
                (unsigned long long)ctx->step_n, 1e6 * ctx->step_t[0] / ctx->step_n, 1e6 * ctx->step_t[1] / ctx->step_n, 1e6 * ctx->step_t[2] / ctx->step_n,
                1e6 * ctx->step_t[3] / ctx->step_n, 1e6 * ctx->step_t[4] / ctx->step_n, 1e6 * ctx->step_t[5] / ctx->step_n);
    if (ctx->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->nccl_comm);
    if (ctx->d_gather) cudaFree(ctx->d_gather);
    for (uint32_t r = 0; r < 8; ++r) if (ctx->peer_map[r] && r != ctx->cl.rank && ctx->peer_ipc[r]) cudaIpcCloseMemHandle(ctx->peer_map[r]);
    if (ctx->d_xbuf) cudaFree(ctx->d_xbuf);
    if (ctx->d_push_done) cudaFree(ctx->d_push_done);
    for (auto &r : ctx->recorded) if (r.dev) cudaFree(r.dev);
    if (ctx->side_stream) { cudaStreamSynchronize(ctx->side_stream); cudaStreamDestroy(ctx->side_stream); }
    if (ctx->clus_stream) { cudaStreamSynchronize(ctx->clus_stream); cudaStreamDestroy(ctx->clus_stream); }
    if (ctx->ev_clus) cudaEventDestroy(ctx->ev_clus);
    if (ctx->ev_tile) cudaEventDestroy(ctx->ev_tile);
    if (ctx->ev_pub) cudaEventDestroy(ctx->ev_pub);
    for (cudaEvent_t e : ctx->ev_side) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->ev_expand) if (e) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

extern "C" int32_t b200vis_create(const b200vis_config *cfg, b200vis_ctx **out) {
    b200vis_ctx *ctx = nullptr;   // for CU(): errors before allocation go to the thread-local slot
    if (!cfg || !out) return fail(nullptr, B200VIS_ERR_INVALID_ARG, "b200vis_create: null argument");
    *out = nullptr;
    if (cfg->max_views == 0 || cfg->max_views > B200VIS_MAX_VIEWS)
        return fail(nullptr, B200VIS_ERR_INVALID_ARG, "max_views must be in 1..%u", B200VIS_MAX_VIEWS);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, B200VIS_ERR_CUDA, "no CUDA device (%s): libb200vis has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, B200VIS_ERR_INVALID_ARG, "device %d out of range", cfg->device);
    CU(cudaSetDevice(cfg->device));
    ctx = new b200vis_ctx();
    ctx->cfg = *cfg;
    ctx->device = cfg->device;
    if (ctx->cfg.world_size == 0) ctx->cfg.world_size = 1;
    if (ctx->cfg.max_cluster_indices == 0) ctx->cfg.max_cluster_indices = 1u << 20;
    const size_t N = cfg->max_entities, V = cfg->max_views;
    int32_t rc = [&]() -> int32_t {
        CU(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
        ctx->stream = ctx->own_stream;
        Rows &r = ctx->rows;
        const size_t NP = N + 32;   // the TMA-staged tile kernel copies 16-row aligned windows: pad every staged column
        CU(dalloc(&r.trsA, NP)); CU(dalloc(&r.trsB, NP)); CU(dalloc(&r.trsC, NP));
        CU(dalloc(&r.gt0, NP)); CU(dalloc(&r.gt1, NP)); CU(dalloc(&r.gt2, NP));
        CU(dalloc(&r.bndA, NP)); CU(dalloc(&r.bndB, NP));
        CU(dalloc(&r.flags, NP)); CU(dalloc(&r.state, NP)); CU(dalloc(&r.topo, NP));
        CU(dalloc(&ctx->d_parent, N)); CU(dalloc(&ctx->d_layers, N)); CU(dalloc(&ctx->d_range, N));
        CU(dalloc(&ctx->d_rank, N)); CU(dalloc(&ctx->d_row_of_rank, N)); CU(dalloc(&ctx->d_dirty, N));
        r.parent = ctx->d_parent;
        ctx->tiles_cap = (uint32_t)(N / 1 + 1);   // worst case one tile per row is never reached; see planner
        ctx->tiles_cap = (uint32_t)std::min<size_t>(N + 1, (N / 8) + 1024);
        CU(dalloc(&ctx->d_tiles, ctx->tiles_cap));
        CU(dalloc(&ctx->d_wtiles, ctx->tiles_cap));
        CU(dalloc(&ctx->d_sched, (size_t)ctx->tiles_cap * kTileRows));
        CU(dalloc(&ctx->d_wtopo, NP));
        CU(dalloc(&ctx->d_tile_counter, 1));
        CU(dalloc(&ctx->d_tile_ticket, 1)); CU(cudaMemset(ctx->d_tile_ticket, 0, 4));
        r.wtopo = ctx->d_wtopo;
        // worst case tables: every view with three (kMaxClusters+1)-entry plane tables + kMaxClusters thresholds
        ctx->blob_cap = sizeof(FrameConsts) + V * (3 * (size_t)(kMaxClusters + 1) * 16 + (size_t)kMaxClusters * 4);
        CU(dalloc(&ctx->d_blob2[0], ctx->blob_cap)); CU(dalloc(&ctx->d_blob2[1], ctx->blob_cap)); CU(dalloc(&ctx->d_blob2[2], ctx->blob_cap));
        ctx->d_blob = ctx->d_blob2[0];
        ctx->d_consts = reinterpret_cast<FrameConsts *>(ctx->d_blob);
        {   // the tail kernels are small and latency-bound: give their CTAs priority over the bulk tile pass
            int lo = 0, hi = 0;
            CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CU(cudaStreamCreateWithPriority(&ctx->side_stream, cudaStreamNonBlocking, hi));
            CU(cudaStreamCreateWithPriority(&ctx->clus_stream, cudaStreamNonBlocking, hi));
            CU(cudaEventCreateWithFlags(&ctx->ev_clus, cudaEventDisableTiming));
        }
        CU(cudaEventCreateWithFlags(&ctx->ev_tile, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_pub, cudaEventDisableTiming));
        for (cudaEvent_t &e : ctx->ev_side) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (cudaEvent_t &e : ctx->ev_expand) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        { const char *e = getenv("B200VIS_PIPELINE"); if (e && e[0] == '0') ctx->pipeline = false; }
        for (int i = 0; i < b200vis_ctx::kRing; ++i) {
            CU(cudaMallocHost(&ctx->h_ring[i], ctx->blob_cap));
            CU(cudaEventCreateWithFlags(&ctx->ring_ev[i], cudaEventDisableTiming));
        }
        // visible set buffers
        VisibleBufs &vb = ctx->vis;
        vb.words_stride = (uint32_t)((N + 31) / 32 + 2);
        vb.chunks_stride = (vb.words_stride + kChunkWords - 1) / kChunkWords + 1;
        vb.list_stride = (uint32_t)std::max<size_t>(N, 1);
        CU(dalloc(&vb.mask, (size_t)2 * vb.words_stride * V));
        CU(dalloc(&vb.chunk_count, (size_t)3 * kMaxViews * vb.chunks_stride));
        CU(dalloc(&vb.lists, (size_t)vb.list_stride * V));
        CU(dalloc(&vb.classes, (size_t)vb.list_stride * V));
        CU(dalloc(&ctx->d_cls, NP));
        vb.cls = ctx->d_cls;
        CU(dalloc(&ctx->d_stats, 1));
        CU(cudaMallocHost(&ctx->h_stats, sizeof(DevStats)));
        // lights + clusters
        const size_t Lm = std::max<uint32_t>(cfg->max_lights, 1);
        CU(dalloc(&ctx->d_tag_flag, 1));
        CU(dalloc(&ctx->d_light_ord, N));
        CU(cudaMemset(ctx->d_light_ord, 0xFF, std::max<size_t>(N, 1) * 4));
        CU(dalloc(&ctx->d_light_row, Lm)); CU(dalloc(&ctx->d_light_range, Lm)); CU(dalloc(&ctx->d_light_layers, Lm));
        ClusterBufs &cl = ctx->cl;
        cl.words = (uint32_t)((Lm + 31) / 32); cl.max_lights = cl.words * 32; cl.world = ctx->cfg.world_size;
        cl.rank = cfg->rank; cl.max_views = (uint32_t)V; cl.index_cap = ctx->cfg.max_cluster_indices;
        ctx->lrec_bytes = (size_t)cl.max_lights * 28;
        CU(cudaMalloc(&ctx->d_lrec, 3 * ctx->lrec_bytes)); CU(cudaMemset(ctx->d_lrec, 0, 3 * ctx->lrec_bytes));
        if (cl.world > 1) { CU(cudaMalloc(&ctx->d_lrec_all, cl.world * ctx->lrec_bytes)); CU(cudaMemset(ctx->d_lrec_all, 0, cl.world * ctx->lrec_bytes)); }
        cl.slab_words = (uint32_t)(V * cl.words * kMaxClusters + kMaxViews);   // bit matrix + per-view farthest_z trailer
        ctx->slab_bytes = (size_t)cl.slab_words * sizeof(uint32_t);
        CU(dalloc(&ctx->d_slab, ctx->slab_bytes / 4));
        cl.send = ctx->d_slab; cl.recv = ctx->d_slab;
        cl.blob = reinterpret_cast<const float *>(ctx->d_blob);   // re-pointed per frame
        CU(dalloc(&cl.offsets, V * (kMaxClusters + 1)));
        CU(dalloc(&cl.indices, V * (size_t)cl.index_cap));
        ctx->stage_bytes = std::max<size_t>(N, 1) * 64;
        CU(cudaMalloc(&ctx->d_stage, ctx->stage_bytes));
        CU(cudaMallocHost(&ctx->h_stage, ctx->stage_bytes));
        return B200VIS_OK;
    }();
    if (rc != B200VIS_OK) { g_create_error = ctx->err; b200vis_destroy(ctx); return rc; }
    *out = ctx;
    return B200VIS_OK;
}

#define CHECK_CTX()                                                        \
    if (!ctx) return B200VIS_ERR_INVALID_ARG;                              \
    CU(cudaSetDevice(ctx->device))

static int32_t join_side(b200vis_ctx *ctx);
static int32_t join_all(b200vis_ctx *ctx);
#define CHECK_CTX_JOIN()                                                   \
    CHECK_CTX();                                                           \
    { const int32_t jrc_ = join_all(ctx); if (jrc_) return jrc_; }

static int32_t check_range(b200vis_ctx *ctx, uint32_t first, uint32_t count, const char *what) {
    if ((uint64_t)first + count > ctx->cfg.max_entities)
        return fail(ctx, B200VIS_ERR_CAPACITY, "%s: rows [%u, %u) exceed max_entities %u", what, first, first + count,
                    ctx->cfg.max_entities);
    return B200VIS_OK;
}

extern "C" int32_t b200vis_set_stream(b200vis_ctx *ctx, void *cuda_stream) {
    CHECK_CTX_JOIN();
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_synchronize(b200vis_ctx *ctx) {
    CHECK_CTX_JOIN();
    CU(cudaStreamSynchronize(ctx->stream));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_static_transform_optimizations(b200vis_ctx *ctx, int32_t enabled) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    ctx->static_opt = enabled ? 1 : 0;
    return B200VIS_OK;
}

// ------------------------------------------------------------------------------------------
// execution plan
// ------------------------------------------------------------------------------------------
// Validates the hierarchy (range, cycles), cuts the rows into tiles of <= kTileRows rows --
// preferring cuts at tree boundaries so parents sit in the same tile as their children -- and
// orders the tiles into passes so that a tile's out-of-tile parents are finished by an earlier
// launch.  Forests of small trees need one pass; a tree larger than a tile needs a few.
struct Plan {
    std::vector<uint32_t> topo;          // per row, CTA-per-tile kernels (device_types.cuh T_*)
    std::vector<uint32_t> wtopo;         // per row, k_tile_warp
    std::vector<Tile> tiles;             // sorted by pass
    std::vector<WarpTile> wtiles;        // the same tiles, same order, as warp work items
    std::vector<uint8_t> sched;          // kTileRows bytes per tile: schedule slot -> local row, 0xFF = padding
    std::vector<uint32_t> pass_begin;    // tile index ranges per pass: [pass_begin[p], pass_begin[p+1])
    std::vector<uint32_t> pass_small;
    uint32_t n_ext = 0;                  // rows whose parent sits in another tile
};
static int32_t build_plan(b200vis_ctx *ctx, uint32_t n, const uint32_t *parent, uint32_t cap, Plan &plan) {
    std::vector<uint32_t> &topo = plan.topo; std::vector<Tile> &tiles_sorted = plan.tiles;
    std::vector<uint32_t> &pass_begin = plan.pass_begin; std::vector<uint32_t> *pass_small = &plan.pass_small;
    if (cap < 32) cap = 32;
    if (cap > (uint32_t)kTileRows) cap = kTileRows;
    for (uint32_t r = 0; r < n; ++r) {
        const uint32_t p = parent[r];
        if (p == kNoParent || p == kDetached) continue;
        if (p >= n) return fail(ctx, B200VIS_ERR_PARENT_OUT_OF_RANGE, "row %u: parent %u out of range (n=%u)", r, p, n);
    }
    {   // cycle check: every chain must end at a root / detached row
        std::vector<uint8_t> color(n, 0);
        std::vector<uint32_t> path;
        for (uint32_t r = 0; r < n; ++r) {
            if (color[r]) continue;
            path.clear();
            uint32_t c = r;
            while (true) {
                if (color[c] == 2) break;
                if (color[c] == 1) return fail(ctx, B200VIS_ERR_HIERARCHY_CYCLE, "hierarchy cycle through row %u", c);
                color[c] = 1; path.push_back(c);
                const uint32_t p = parent[c];
                if (p >= n) break;
                c = p;
            }
            for (uint32_t x : path) color[x] = 2;
        }
    }
    for (uint32_t r = 0; r < n; ++r)
        if (parent[r] < n && parent[r] >= r)
            return fail(ctx, B200VIS_ERR_UNSUPPORTED,
                        "row %u has parent %u >= itself: rows must be in topological order (use b200vis_plan_row_order)", r,
                        parent[r]);
    // greedy tiling, cutting at the latest tree boundary inside a full tile
    static int split_env = -1;
    if (split_env < 0) { const char *e = getenv("B200VIS_SPLIT_DEEP_TILES"); split_env = (e && atoi(e)) ? 1 : 0; }
    const bool split_deep = split_env == 1;
    std::vector<Tile> tiles;
    std::vector<uint32_t> tile_of(n);
    std::vector<uint8_t> marked(n, 0);
    uint32_t start = 0;
    while (start < n) {
        uint32_t end = std::min<uint32_t>(n, start + cap);
        if (end < n && parent[end] < n) {          // the cut would split a tree: back up to a boundary
            uint32_t c = end;
            while (c > start + 1 && parent[c] < n) --c;   // c = latest row in (start, end] that starts a tree
            if (c > start && !(parent[c] < n)) end = c;
        }
        {   // k_tile_warp keeps the GlobalTransforms of the rows WITH in-tile children in kWarpParentSlots shared-memory
            // slots: cut the tile before the child that would need one more (only chains and unary-heavy trees get there)
            uint32_t parents = 0;
            for (uint32_t c = start; c < end; ++c) {
                const uint32_t p = parent[c];
                if (p < n && p >= start && !marked[p]) {
                    if (parents == (uint32_t)kWarpParentSlots) { end = c; break; }
                    marked[p] = 1; ++parents;
                }
            }
        }
        // EXPERIMENT (B200VIS_SPLIT_DEEP_TILES=1, off by default): the hierarchy walk of a tile is a serial chain of its
        // levels (DESIGN.md section 7: ~680 cycles per level).  When the first <= 32 rows of a deep tile are exactly its top
        // K levels (level-ordered rows, e.g. one tree in BFS order), cut there: the top becomes a tile of its own, one pass
        // earlier (run by 32-thread CTAs), and the bottom keeps only n_levels - K levels with external parents.
        uint32_t cut = 0;
        if (split_deep && end - start > 64) {
            std::vector<uint32_t> dep(end - start, 0), cnt;
            for (uint32_t r = start; r < end; ++r) {
                const uint32_t p = parent[r];
                dep[r - start] = (p < n && p >= start) ? dep[p - start] + 1 : 0;
                if (dep[r - start] >= cnt.size()) cnt.resize(dep[r - start] + 1, 0);
                cnt[dep[r - start]]++;
            }
            const uint32_t levels = (uint32_t)cnt.size();
            if (levels >= 6) {
                uint32_t rows_above = 0;
                for (uint32_t K = 1; K + 2 <= levels; ++K) {       // rows with depth < K
                    rows_above += cnt[K - 1];
                    if (rows_above > 32) break;
                    bool prefix = true;                              // they must be exactly the first rows_above rows
                    for (uint32_t i = 0; i < end - start && prefix; ++i) prefix = (dep[i] < K) == (i < rows_above);
                    if (prefix && K >= 2) cut = rows_above;
                }
            }
        }
        for (uint32_t part = 0; part < (cut ? 2u : 1u); ++part) {
            const uint32_t b = (part == 0) ? start : start + cut, e = (cut && part == 0) ? start + cut : end;
            Tile t; t.base = b; t.n_rows = (uint16_t)(e - b); t.n_levels = 1; t.warp_sync_mask = 0xFFFFFFFFu; t.top_levels = 0; t.lvl_warps = 0;
            for (uint32_t r = b; r < e; ++r) tile_of[r] = (uint32_t)tiles.size();
            tiles.push_back(t);
        }
        start = end;
    }
    // rows with children IN THEIR OWN TILE (a child in a later tile reads its parent from HBM, an earlier pass)
    std::vector<uint8_t> has_children(n, 0), has_local_children(n, 0);
    for (uint32_t r = 0; r < n; ++r)
        if (parent[r] < n) { has_children[parent[r]] = 1; if (tile_of[parent[r]] == tile_of[r]) has_local_children[parent[r]] = 1; }
    // topo words, in-tile depth, tile levels
    topo.assign(n, 0);
    plan.n_ext = 0;
    std::vector<uint32_t> ldepth(n, 0), tile_level(tiles.size(), 0);
    for (uint32_t r = 0; r < n; ++r) {
        const uint32_t p = parent[r], ti = tile_of[r];
        uint32_t w = 0;
        if (p == kNoParent) w |= T_ROOT;
        else if (p == kDetached) w |= T_DETACHED;
        else if (tile_of[p] == ti) {
            ldepth[r] = ldepth[p] + 1;
            w |= (p - tiles[ti].base) | (ldepth[r] << 9);
            tiles[ti].n_levels = std::max<uint16_t>(tiles[ti].n_levels, (uint16_t)(ldepth[r] + 1));
            // a level keeps its warp-sync bit only while every parent->child edge into it stays inside one warp
            if (ldepth[r] < 32 && ((p - tiles[ti].base) >> 5) != ((r - tiles[ti].base) >> 5))
                tiles[ti].warp_sync_mask &= ~(1u << ldepth[r]);
        } else {
            w |= T_EXT_PARENT;
            ++plan.n_ext;
            tile_level[ti] = std::max(tile_level[ti], tile_level[tile_of[p]] + 1);
        }
        if (has_children[r]) w |= T_HAS_CHILDREN;
        topo[r] = w;
    }
    {   // top_levels: the leading depth levels whose rows all sit among the tile's first 32 rows
        std::vector<uint32_t> max_local;
        for (size_t ti = 0; ti < tiles.size(); ++ti) {
            Tile &t = tiles[ti];
            max_local.assign(t.n_levels, 0);
            for (uint32_t r = t.base; r < t.base + t.n_rows; ++r) max_local[ldepth[r]] = std::max(max_local[ldepth[r]], r - t.base);
            uint32_t K = 0;
            while (K < t.n_levels && max_local[K] < 32u) ++K;
            static int cap_env = -1;      // B200VIS_TOP_LEVELS_CAP: how many levels the scout may take (experiment knob)
            if (cap_env < 0) { const char *e = getenv("B200VIS_TOP_LEVELS_CAP"); cap_env = e ? atoi(e) : 255; }
            if (K > (uint32_t)cap_env) K = (uint32_t)cap_env;
            t.top_levels = (t.n_levels > 1) ? K : 0u;       // flat tiles have nothing to walk ahead
        }
    }
    {   // lvl_warps: which warps meet at which level hand-over (named barriers, k_propagate_cull_tma)
        static int level_sync = -1;     // B200VIS_LEVEL_SYNC=cta: keep the CTA-wide level barriers (A/B switch)
        if (level_sync < 0) { const char *e = getenv("B200VIS_LEVEL_SYNC"); level_sync = (e && e[0] == 'c') ? 0 : 1; }
        for (size_t ti = 0; level_sync && ti < tiles.size(); ++ti) {
            Tile &t = tiles[ti];
            if (t.n_levels < 2 || t.n_levels > 8) continue;      // seven barrier ids per tile parity (levels 1..7)
            uint32_t lv[kTileRows / 32] = {};          // per warp: bit l = the warp holds a row of in-tile depth l (a detached
            for (uint32_t r = t.base; r < t.base + t.n_rows; ++r)      // row has depth 0: it publishes "not visited" to its children)
                lv[(r - t.base) >> 5] |= 1u << ldepth[r];
            unsigned long long packed = 0;
            for (uint32_t l = 1; l < t.n_levels; ++l) {
                unsigned long long c = 0;
                for (uint32_t w = 0; w < (uint32_t)kTileRows / 32u; ++w) c += ((lv[w] >> (l - 1)) & 3u) ? 1u : 0u;
                packed |= c << (4u * l);
            }
            t.lvl_warps = packed;
        }
    }
    // ---- warp work items: schedule, parent slots, wtopo ------------------------------------------------------------
    std::vector<WarpTile> wtiles(tiles.size());
    std::vector<uint8_t> sched_all(tiles.size() * (size_t)kTileRows, 0xFF);
    plan.wtopo.assign(n, 0);
    {
        std::vector<uint32_t> slot_of(n, 0);     // parent slot of the rows with in-tile children
        std::vector<uint32_t> level_count, order;
        for (size_t ti = 0; ti < tiles.size(); ++ti) {
            const Tile &t = tiles[ti];
            const uint32_t b = t.base, nr = t.n_rows;
            // rows in (depth, row) order: counting sort by in-tile depth
            level_count.assign((size_t)t.n_levels + 1, 0);
            for (uint32_t r = b; r < b + nr; ++r) level_count[ldepth[r] + 1]++;
            for (uint32_t l = 0; l < t.n_levels; ++l) level_count[l + 1] += level_count[l];
            order.assign(nr, 0);
            { std::vector<uint32_t> cur(level_count.begin(), level_count.end() - 1);
              for (uint32_t r = b; r < b + nr; ++r) order[cur[ldepth[r]]++] = r - b; }
            // slots: a level with >= 32 rows starts on a chunk boundary when the padding still fits into kTileRows slots
            uint8_t *sch = sched_all.data() + ti * (size_t)kTileRows;
            uint32_t pos = 0, next_slot = 0;
            for (uint32_t l = 0; l < t.n_levels; ++l) {
                const uint32_t lb = level_count[l], le = level_count[l + 1], cnt = le - lb;
                if ((pos & 31u) && cnt >= 32u) {
                    const uint32_t padded = (pos + 31u) & ~31u;
                    if (padded + (nr - lb) <= (uint32_t)kTileRows) pos = padded;
                }
                for (uint32_t i = lb; i < le; ++i) {
                    const uint32_t r = b + order[i];
                    sch[pos++] = (uint8_t)order[i];
                    if (has_local_children[r]) slot_of[r] = next_slot++;
                }
            }
            WarpTile &w = wtiles[ti];
            memset(&w, 0, sizeof w);
            w.base = b; w.n_rows = (uint16_t)nr; w.n_chunks = (uint8_t)((pos + 31u) / 32u); w.sched = (uint32_t)ti;
            for (uint32_t c = 0; c < w.n_chunks; ++c) {
                bool contig = true; int64_t delta = 0; bool have = false;
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    const uint8_t lr = sch[c * 32 + lane];
                    if (lr == 0xFF && nr != (uint32_t)kTileRows) continue;   // padding (a full tile has none: 0xFF is row 255)
                    const int64_t d = (int64_t)lr - (int64_t)lane;
                    if (!have) { delta = d; have = true; } else if (d != delta) contig = false;
                    if (ldepth[b + lr] > 0) w.nonroot[c] |= 1u << lane;
                }
                if (contig) w.contig |= (uint8_t)(1u << c);
            }
        }
        for (uint32_t r = 0; r < n; ++r) {
            uint32_t w = topo[r] & 0xF0000000u;      // T_HAS_CHILDREN stays the reference's "has a Children component"
            if (has_local_children[r]) w |= W_HAS_SLOT | (slot_of[r] << 8);
            w |= ldepth[r] & 0xFFu;
            if (ldepth[r]) w |= slot_of[parent[r]] << 15;
            plan.wtopo[r] = w;
        }
    }
    // NOTE: tile_level of tile t only depends on tiles with a smaller index (topological rows), and
    // those are final by the time a row of t is visited, because rows are visited in ascending order.
    const uint32_t n_pass = tiles.empty() ? 0 : *std::max_element(tile_level.begin(), tile_level.end()) + 1;
    pass_begin.assign(n_pass + 1, 0);
    for (uint32_t lv : tile_level) pass_begin[lv + 1]++;
    for (uint32_t p = 0; p < n_pass; ++p) pass_begin[p + 1] += pass_begin[p];
    tiles_sorted.resize(tiles.size());
    plan.wtiles.resize(tiles.size());
    std::vector<uint32_t> cursor(pass_begin.begin(), pass_begin.end() - (n_pass ? 1 : 0));
    if (pass_small) pass_small->assign(n_pass, 0);
    // within a pass: the small tiles (<= 32 rows, only produced by the split above) first, then the rest
    for (int small = 1; small >= 0; --small)
        for (size_t i = 0; i < tiles.size(); ++i) {
            const bool is_small = split_deep && tiles[i].n_rows <= 32;
            if ((int)is_small != small) continue;
            const uint32_t at = cursor[tile_level[i]]++;
            tiles_sorted[at] = tiles[i];
            plan.wtiles[at] = wtiles[i];       // .sched keeps pointing at the tile's block in creation order
            if (is_small && pass_small) (*pass_small)[tile_level[i]]++;
        }
    plan.sched.swap(sched_all);
    return B200VIS_OK;
}

extern "C" int32_t b200vis_set_topology(b200vis_ctx *ctx, uint32_t n, const uint32_t *parent, const uint64_t *entity_bits) {
    CHECK_CTX_JOIN();
    if (n && (!parent || !entity_bits)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_topology: null array");
    if (n > ctx->cfg.max_entities) return fail(ctx, B200VIS_ERR_CAPACITY, "set_topology: %u rows > max_entities %u", n, ctx->cfg.max_entities);
    // Tile size: a tile is one WARP's work item, and the machine has ~4700 resident warps: small scenes get smaller tiles
    // (more warps busy) as long as that does not split trees across tiles (more passes / parents read from HBM).
    Plan plan;
    int32_t rc = build_plan(ctx, n, parent, kTileRows, plan);
    if (rc != B200VIS_OK) return rc;
    {
        static int cap_env = -1;
        if (cap_env < 0) { const char *e = getenv("B200VIS_TILE_ROWS"); cap_env = e ? atoi(e) : 0; }
        uint32_t target = cap_env > 0 ? (uint32_t)cap_env : (uint32_t)std::min<uint64_t>(kTileRows, (((uint64_t)n / 9472u) + 31u) / 32u * 32u);
        if (target < 32) target = 32;
        for (uint32_t cap = target; cap < (uint32_t)kTileRows; cap *= 2) {
            Plan q;
            if (build_plan(ctx, n, parent, cap, q) != B200VIS_OK) break;
            if (q.pass_begin.size() <= plan.pass_begin.size() && q.n_ext <= plan.n_ext) { plan = std::move(q); break; }
        }
    }
    std::vector<uint32_t> &topo = plan.topo; std::vector<Tile> &tiles = plan.tiles;
    std::vector<uint32_t> &pass_begin = plan.pass_begin, &pass_small = plan.pass_small;
    if (tiles.size() > ctx->tiles_cap) {
        void *old[] = {ctx->d_tiles, ctx->d_wtiles, ctx->d_sched};
        for (void *q : old) if (q) cudaFree(q);
        ctx->d_tiles = nullptr; ctx->d_wtiles = nullptr; ctx->d_sched = nullptr; ctx->tiles_cap = (uint32_t)tiles.size() + 1024;
        CU(dalloc(&ctx->d_tiles, ctx->tiles_cap));
        CU(dalloc(&ctx->d_wtiles, ctx->tiles_cap));
        CU(dalloc(&ctx->d_sched, (size_t)ctx->tiles_cap * kTileRows));
    }
    // Entity::to_bits() order -> rank
    bool sorted = true;
    for (uint32_t r = 1; r < n && sorted; ++r) sorted = entity_bits[r - 1] < entity_bits[r];
    std::vector<uint32_t> order, rank;
    if (!sorted) {
        order.resize(n); std::iota(order.begin(), order.end(), 0u);
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return entity_bits[a] < entity_bits[b]; });
        rank.resize(n);
        for (uint32_t i = 0; i < n; ++i) rank[order[i]] = i;
    }
    cudaStream_t st = ctx->stream;
    CU(cudaStreamSynchronize(st));   // the vectors below are pageable and short-lived: copy synchronously
    CU(cudaMemcpy(ctx->rows.topo, topo.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_parent, parent, (size_t)n * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_tiles, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_wtiles, plan.wtiles.data(), plan.wtiles.size() * sizeof(WarpTile), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_sched, plan.sched.data(), plan.sched.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_wtopo, plan.wtopo.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
    if (!sorted) {
        CU(cudaMemcpy(ctx->d_rank, rank.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ctx->d_row_of_rank, order.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
    }
    ctx->pass_begin = pass_begin;
    ctx->pass_small = pass_small;
    ctx->pass_named.assign(pass_begin.empty() ? 0 : pass_begin.size() - 1, 1);
    for (size_t pi = 0; pi + 1 < pass_begin.size(); ++pi)
        for (uint32_t ti = pass_begin[pi]; ti < pass_begin[pi + 1]; ++ti)
            if (tiles[ti].n_levels > 1 && tiles[ti].lvl_warps == 0ull) { ctx->pass_named[pi] = 0; break; }
    ctx->rank_identity = sorted;
    ctx->n = n;
    ctx->rows.n = n;
    ctx->vis.n_words = (n + 31) / 32;
    ctx->vis.n_chunks = (ctx->vis.n_words + kChunkWords - 1) / kChunkWords;
    // fresh accumulation state
    CU(cudaMemset(ctx->vis.mask, 0, (size_t)2 * ctx->vis.words_stride * ctx->cfg.max_views * 4));
    CU(cudaMemset(ctx->vis.chunk_count, 0, (size_t)3 * kMaxViews * ctx->vis.chunks_stride * 4));
    CU(cudaMemset(ctx->d_stats, 0, sizeof(DevStats)));
    CU(cudaMemset(ctx->d_slab, 0, ctx->slab_bytes));
    if (ctx->diff.prev) CU(cudaMemset(ctx->diff.prev, 0, (size_t)ctx->vis.words_stride * ctx->cfg.max_views * 4));   // ranks changed: old list = empty
    ctx->topology_set = true;
    ctx->gt_aos_valid = false;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_host_plan_summary(uint32_t n, const uint32_t *parent, uint32_t out[4]) {
    if ((n && !parent) || !out) return B200VIS_ERR_INVALID_ARG;
    Plan plan;
    const int32_t rc = build_plan(nullptr, n, parent, kTileRows, plan);
    if (rc) return rc;
    std::vector<uint32_t> &topo = plan.topo, &pass_begin = plan.pass_begin; std::vector<Tile> &tiles = plan.tiles;
    uint32_t max_levels = 0, ext = 0;
    for (const Tile &t : tiles) max_levels = std::max<uint32_t>(max_levels, t.n_levels);
    for (uint32_t w : topo) ext += (w & T_EXT_PARENT) ? 1u : 0u;
    out[0] = (uint32_t)tiles.size(); out[1] = pass_begin.empty() ? 0u : (uint32_t)pass_begin.size() - 1; out[2] = max_levels; out[3] = ext;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_host_warp_plan(uint32_t n, const uint32_t *parent, uint32_t tile_rows, uint32_t tiles_capacity, uint32_t *n_tiles,
                                          uint32_t *tile_desc, uint32_t *nonroot, uint8_t *sched, uint32_t *wtopo) {
    if ((n && !parent) || !n_tiles) return B200VIS_ERR_INVALID_ARG;
    Plan plan;
    const int32_t rc = build_plan(nullptr, n, parent, tile_rows ? tile_rows : kTileRows, plan);
    if (rc) return rc;
    *n_tiles = (uint32_t)plan.wtiles.size();
    if (!tile_desc) return B200VIS_OK;
    if (plan.wtiles.size() > tiles_capacity || !nonroot || !sched || (n && !wtopo)) return B200VIS_ERR_CAPACITY;
    std::vector<uint32_t> pass_of(plan.wtiles.size(), 0);
    for (size_t p = 0; p + 1 < plan.pass_begin.size(); ++p)
        for (uint32_t i = plan.pass_begin[p]; i < plan.pass_begin[p + 1]; ++i) pass_of[i] = (uint32_t)p;
    for (size_t i = 0; i < plan.wtiles.size(); ++i) {
        const WarpTile &w = plan.wtiles[i];
        tile_desc[i * 4 + 0] = w.base; tile_desc[i * 4 + 1] = w.n_rows;
        tile_desc[i * 4 + 2] = w.n_chunks | ((uint32_t)w.contig << 8); tile_desc[i * 4 + 3] = pass_of[i];
        memcpy(nonroot + i * kWarpChunks, w.nonroot, sizeof w.nonroot);
        memcpy(sched + i * (size_t)kTileRows, plan.sched.data() + (size_t)w.sched * kTileRows, kTileRows);
    }
    if (n) memcpy(wtopo, plan.wtopo.data(), (size_t)n * 4);
    return B200VIS_OK;
}

extern "C" int32_t b200vis_host_tile_plan(uint32_t n, const uint32_t *parent, uint32_t tile_rows, uint32_t tiles_capacity, uint32_t *n_tiles,
                                          uint32_t *tile_desc, uint32_t *topo) {
    if ((n && !parent) || !n_tiles) return B200VIS_ERR_INVALID_ARG;
    Plan plan;
    const int32_t rc = build_plan(nullptr, n, parent, tile_rows ? tile_rows : kTileRows, plan);
    if (rc) return rc;
    *n_tiles = (uint32_t)plan.tiles.size();
    if (!tile_desc) return B200VIS_OK;
    if (plan.tiles.size() > tiles_capacity || (n && !topo)) return B200VIS_ERR_CAPACITY;
    std::vector<uint32_t> pass_of(plan.tiles.size(), 0);
    for (size_t p = 0; p + 1 < plan.pass_begin.size(); ++p)
        for (uint32_t i = plan.pass_begin[p]; i < plan.pass_begin[p + 1]; ++i) pass_of[i] = (uint32_t)p;
    for (size_t i = 0; i < plan.tiles.size(); ++i) {
        const Tile &t = plan.tiles[i];
        uint32_t *d = tile_desc + i * 8;
        d[0] = t.base; d[1] = t.n_rows; d[2] = t.n_levels; d[3] = t.warp_sync_mask; d[4] = t.top_levels;
        d[5] = (uint32_t)t.lvl_warps; d[6] = (uint32_t)(t.lvl_warps >> 32); d[7] = pass_of[i];
    }
    if (n) memcpy(topo, plan.topo.data(), (size_t)n * 4);
    return B200VIS_OK;
}

extern "C" int32_t b200vis_plan_row_order(uint32_t n, const uint32_t *parent, uint32_t *new_to_old) {
    if (n && (!parent || !new_to_old)) return B200VIS_ERR_INVALID_ARG;
    // children lists (ascending old row), then BFS per root in ascending root order
    std::vector<uint32_t> first(n + 1, 0), kids(n);
    for (uint32_t r = 0; r < n; ++r) {
        const uint32_t p = parent[r];
        if (p < n) first[p + 1]++;
        else if (p != kNoParent && p != kDetached) return B200VIS_ERR_PARENT_OUT_OF_RANGE;
    }
    for (uint32_t r = 0; r < n; ++r) first[r + 1] += first[r];
    { std::vector<uint32_t> cur(first.begin(), first.end() - 1);
      for (uint32_t r = 0; r < n; ++r) if (parent[r] < n) kids[cur[parent[r]]++] = r; }
    uint32_t out = 0;
    for (uint32_t r = 0; r < n; ++r) {
        if (parent[r] < n) continue;               // roots, flat entities and detached subtrees start a block
        const uint32_t head = out;
        new_to_old[out++] = r;
        for (uint32_t i = head; i < out; ++i) {
            const uint32_t c = new_to_old[i];
            for (uint32_t k = first[c]; k < first[c + 1]; ++k) new_to_old[out++] = kids[k];
        }
    }
    return out == n ? B200VIS_OK : B200VIS_ERR_HIERARCHY_CYCLE;   // rows on a cycle are never reached
}

// ------------------------------------------------------------------------------------------
// uploads
// ------------------------------------------------------------------------------------------
static int32_t stage_in(b200vis_ctx *ctx, const void *src, size_t bytes, size_t offset) {
    if (offset + bytes > ctx->stage_bytes) return fail(ctx, B200VIS_ERR_CAPACITY, "staging buffer too small");
    CU(cudaMemcpyAsync(ctx->d_stage + offset, src, bytes, cudaMemcpyDefault, ctx->stream));   // host or device source (UVA)
    return B200VIS_OK;
}

extern "C" int32_t b200vis_upload_transforms(b200vis_ctx *ctx, uint32_t first, uint32_t count, const float *trs) {
    CHECK_CTX();
    if (count && !trs) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_transforms: null");
    int32_t rc = check_range(ctx, first, count, "upload_transforms"); if (rc) return rc;
    rc = stage_in(ctx, trs, (size_t)count * 40, 0); if (rc) return rc;
    launch_unpack_trs(ctx->stream, ctx->rows, first, count, reinterpret_cast<const float *>(ctx->d_stage), 0);
    CU(cudaGetLastError());
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_transforms_scattered(b200vis_ctx *ctx, uint32_t count, const uint32_t *rows, const float *trs) {
    CHECK_CTX();
    if (count && (!rows || !trs)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_transforms_scattered: null");
    if (count > ctx->cfg.max_entities) return fail(ctx, B200VIS_ERR_CAPACITY, "upload_transforms_scattered: count > max_entities");
    {   // sources already in device memory (a renderer / physics step on the same GPU): no staging copy
        cudaPointerAttributes pa{}, pb{};
        if (cudaPointerGetAttributes(&pa, rows) == cudaSuccess && cudaPointerGetAttributes(&pb, trs) == cudaSuccess) {
            if (pa.type == cudaMemoryTypeDevice && pb.type == cudaMemoryTypeDevice) {
                launch_scatter_trs(ctx->stream, ctx->rows, count, rows, trs);
                CU(cudaGetLastError());
                return B200VIS_OK;
            }
            // pinned (page-locked, mapped) host memory: the scatter kernel reads it over PCIe itself -- one launch instead
            // of two staging copies plus a launch.  The caller must not rewrite the buffers until the stream has passed.
            if (pa.type == cudaMemoryTypeHost && pb.type == cudaMemoryTypeHost && pa.devicePointer && pb.devicePointer) {
                launch_scatter_trs(ctx->stream, ctx->rows, count, static_cast<const uint32_t *>(pa.devicePointer),
                                   static_cast<const float *>(pb.devicePointer));
                CU(cudaGetLastError());
                return B200VIS_OK;
            }
        }
        cudaGetLastError();   // clear the error state cudaPointerGetAttributes leaves for unregistered host memory
    }
    const size_t off_rows = ((size_t)count * 40 + 15) & ~(size_t)15;
    int32_t rc = stage_in(ctx, trs, (size_t)count * 40, 0); if (rc) return rc;
    rc = stage_in(ctx, rows, (size_t)count * 4, off_rows); if (rc) return rc;
    launch_scatter_trs(ctx->stream, ctx->rows, count, reinterpret_cast<const uint32_t *>(ctx->d_stage + off_rows),
                       reinterpret_cast<const float *>(ctx->d_stage));
    CU(cudaGetLastError());
    return B200VIS_OK;
}
extern "C" int32_t b200vis_mark_transforms_changed(b200vis_ctx *ctx, uint32_t first, uint32_t count) {
    CHECK_CTX();
    int32_t rc = check_range(ctx, first, count, "mark_transforms_changed"); if (rc) return rc;
    launch_unpack_trs(ctx->stream, ctx->rows, first, count, nullptr, 1);
    CU(cudaGetLastError());
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_global_transforms(b200vis_ctx *ctx, uint32_t first, uint32_t count, const float *gt) {
    CHECK_CTX();
    if (count && !gt) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_global_transforms: null");
    int32_t rc = check_range(ctx, first, count, "upload_global_transforms"); if (rc) return rc;
    rc = stage_in(ctx, gt, (size_t)count * 48, 0); if (rc) return rc;
    launch_unpack_gt(ctx->stream, ctx->rows, first, count, reinterpret_cast<const float *>(ctx->d_stage));
    CU(cudaGetLastError());
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_bounds(b200vis_ctx *ctx, uint32_t first, uint32_t count, const float *bounds,
                                         const uint8_t *flags, const uint8_t *class_mask, const uint64_t *layer_mask,
                                         const uint32_t *range_mask) {
    CHECK_CTX();
    if (count && (!bounds || !flags || !class_mask)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_bounds: null");
    int32_t rc = check_range(ctx, first, count, "upload_bounds"); if (rc) return rc;
    const size_t ob = 0, of = (size_t)count * 24, oc = of + (((size_t)count + 15) & ~(size_t)15);
    rc = stage_in(ctx, bounds, (size_t)count * 24, ob); if (rc) return rc;
    rc = stage_in(ctx, flags, count, of); if (rc) return rc;
    rc = stage_in(ctx, class_mask, count, oc); if (rc) return rc;
    launch_unpack_bounds(ctx->stream, ctx->rows, first, count, reinterpret_cast<const float *>(ctx->d_stage + ob),
                         ctx->d_stage + of, ctx->d_stage + oc, ctx->d_cls);
    CU(cudaGetLastError());
    if (layer_mask) {
        CU(cudaMemcpyAsync(ctx->d_layers + first, layer_mask, (size_t)count * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (!ctx->have_layers) {
            // rows never uploaded keep the default layer (RenderLayers::default() = layer 0)
            std::vector<uint64_t> ones(ctx->cfg.max_entities, 1ull);
            CU(cudaStreamSynchronize(ctx->stream));
            if (first) CU(cudaMemcpy(ctx->d_layers, ones.data(), (size_t)first * 8, cudaMemcpyHostToDevice));
            const size_t tail = ctx->cfg.max_entities - (first + count);
            if (tail) CU(cudaMemcpy(ctx->d_layers + first + count, ones.data(), tail * 8, cudaMemcpyHostToDevice));
            ctx->have_layers = true;
        }
    }
    if (range_mask) {
        CU(cudaMemcpyAsync(ctx->d_range + first, range_mask, (size_t)count * 4, cudaMemcpyHostToDevice, ctx->stream));
        ctx->have_range = true;
    }
    ctx->bounds_set = true;
    ctx->lights_tag_dirty = true;   // flags were rewritten: re-verify that every light row is a sphere-from-GT row
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_render_layers_ext(b200vis_ctx *ctx, uint32_t first, uint32_t count, const uint64_t *blocks) {
    CHECK_CTX();
    if (count && !blocks) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_render_layers_ext: null");
    int32_t rc = check_range(ctx, first, count, "upload_render_layers_ext"); if (rc) return rc;
    if (!ctx->d_layers_ext) CU(dalloc(&ctx->d_layers_ext, (size_t)ctx->cfg.max_entities * 3));   // rows never uploaded: blocks empty
    CU(cudaMemcpyAsync(ctx->d_layers_ext + (size_t)first * 3, blocks, (size_t)count * 24, cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->have_layers) {   // the general cull path reads block 0 per row too: default layer for everybody until uploaded
        std::vector<uint64_t> ones(ctx->cfg.max_entities, 1ull);
        CU(cudaStreamSynchronize(ctx->stream));
        CU(cudaMemcpy(ctx->d_layers, ones.data(), ones.size() * 8, cudaMemcpyHostToDevice));
        ctx->have_layers = true;
    }
    ctx->have_layers_ext = true;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_view_render_layers_ext(b200vis_ctx *ctx, uint32_t view, const uint64_t blocks[3]) {
    if (!ctx || view >= (uint32_t)kMaxViews) return B200VIS_ERR_INVALID_ARG;
    for (int k = 0; k < 3; ++k) ctx->view_layers_ext[view][k] = blocks ? blocks[k] : 0ull;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_view_visibility(b200vis_ctx *ctx, uint32_t first, uint32_t count, const uint8_t *vv) {
    CHECK_CTX();
    if (count && !vv) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_view_visibility: null");
    int32_t rc = check_range(ctx, first, count, "upload_view_visibility"); if (rc) return rc;
    rc = stage_in(ctx, vv, count, 0); if (rc) return rc;
    launch_unpack_vv(ctx->stream, ctx->rows, first, count, ctx->d_stage);
    CU(cudaGetLastError());
    return B200VIS_OK;
}

// ------------------------------------------------------------------------------------------
// per-frame constants
// ------------------------------------------------------------------------------------------
extern "C" int32_t b200vis_set_views(b200vis_ctx *ctx, uint32_t n_views, const b200vis_view *views) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    if (n_views > ctx->cfg.max_views) return fail(ctx, B200VIS_ERR_CAPACITY, "set_views: %u > max_views %u", n_views, ctx->cfg.max_views);
    if (n_views && !views) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_views: null");
    FrameConsts &fc = ctx->consts;
    fc.n_views = n_views;
    for (uint32_t v = 0; v < n_views; ++v) {
        DevView &d = fc.views[v];
        memcpy(d.hs, views[v].half_spaces, sizeof d.hs);
        d.layer_mask = views[v].layer_mask; d.flags = views[v].flags; d.range_index = views[v].range_view_index;
    }
    ctx->consts_dirty = true;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_set_view_count(b200vis_ctx *ctx, uint32_t n_views) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    if (n_views > ctx->cfg.max_views) return fail(ctx, B200VIS_ERR_CAPACITY, "set_view_count: %u > max_views %u", n_views, ctx->cfg.max_views);
    ctx->consts.n_views = n_views;
    ctx->consts_dirty = true;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_update_camera(b200vis_ctx *ctx, uint32_t view, const b200vis_camera *cam,
                                         const b200vis_cluster_config *cfg, const b200vis_cluster_feedback *fb,
                                         b200vis_cluster_view *out) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    if (view >= ctx->cfg.max_views || !cam) return fail(ctx, B200VIS_ERR_INVALID_ARG, "update_camera: bad view %u", view);
    float cfv[16], hs[6][4];
    host::perspective_infinite_reverse_rh(cam->fov_y, cam->aspect, cam->near_z, cfv);
    host::compute_frustum(cfv, cam->global_transform, cam->far_z, hs);
    DevView &d = ctx->consts.views[view];
    memcpy(d.hs, hs, sizeof d.hs);
    d.layer_mask = cam->layer_mask; d.flags = cam->flags; d.range_index = cam->range_view_index;
    if (ctx->consts.n_views <= view) ctx->consts.n_views = view + 1;
    ctx->consts_dirty = true;
    if (cfg) {
        static thread_local std::vector<float> scratch(3 * 4097 * 4);
        b200vis_cluster_view cv;
        int32_t rc = host::cluster_view_setup(cfg, cam->global_transform, cfv, hs, cam->layer_mask, fb, scratch.data(), &cv);
        if (rc) return fail(ctx, rc, "update_camera: cluster grid of view %u exceeds %d clusters", view, kMaxClusters);
        rc = b200vis_set_cluster_view(ctx, view, &cv);
        if (rc) return rc;
        if (out) *out = cv;
    } else {
        ctx->consts.cviews[view].enabled = 0;
        if (out) memset(out, 0, sizeof *out);
    }
    return B200VIS_OK;
}

// The light blocks of the three frame slots: stale snapshots out, the ranges and layer masks of every ordinal in (point lights,
// then the clusterable objects), and the kind byte of every ordinal when objects are set.  Rare (set time only): the tail of
// the frame in flight is joined first.
static int32_t write_light_blocks(b200vis_ctx *ctx) {
    const int32_t jrc = join_all(ctx); if (jrc) return jrc;
    const uint32_t cap = ctx->cl.max_lights, nl = ctx->lights.n, no = ctx->n_objects();
    std::vector<uint8_t> blk(ctx->lrec_bytes, 0);
    float *rg = reinterpret_cast<float *>(blk.data() + (size_t)cap * 16);
    uint64_t *ly = reinterpret_cast<uint64_t *>(blk.data() + (size_t)cap * 20);
    for (uint32_t i = 0; i < nl; ++i) { rg[i] = ctx->h_light_range[i]; ly[i] = ctx->h_light_layers.empty() ? 1ull : ctx->h_light_layers[i]; }
    for (uint32_t j = 0; j < no; ++j) { rg[nl + j] = ctx->h_obj_range[j]; ly[nl + j] = ctx->h_obj_layers[j]; }
    CU(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 3; ++k) CU(cudaMemcpy(ctx->d_lrec + k * ctx->lrec_bytes, blk.data(), ctx->lrec_bytes, cudaMemcpyHostToDevice));
    if (no) {
        std::vector<uint8_t> kinds(nl, (uint8_t)kKindPoint);
        kinds.insert(kinds.end(), ctx->h_obj_kind.begin(), ctx->h_obj_kind.end());
        CU(cudaMemcpy(ctx->d_ord_kind, kinds.data(), kinds.size(), cudaMemcpyHostToDevice));
    }
    return B200VIS_OK;
}

extern "C" int32_t b200vis_set_lights(b200vis_ctx *ctx, uint32_t n_lights, const uint32_t *light_row, const float *range,
                                      const uint64_t *layer_mask) {
    CHECK_CTX();
    if (n_lights > ctx->cfg.max_lights) return fail(ctx, B200VIS_ERR_CAPACITY, "set_lights: %u > max_lights %u", n_lights, ctx->cfg.max_lights);
    if (n_lights + ctx->n_objects() > ctx->cfg.max_lights)
        return fail(ctx, B200VIS_ERR_CAPACITY, "set_lights: %u lights + %u clusterable objects > max_lights %u", n_lights, ctx->n_objects(), ctx->cfg.max_lights);
    if (n_lights && (!light_row || !range)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_lights: null");
    for (uint32_t i = 0; i < n_lights; ++i)
        if (light_row[i] >= ctx->cfg.max_entities) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_lights: light %u row %u out of range", i, light_row[i]);
    CU(cudaMemcpyAsync(ctx->d_light_row, light_row, (size_t)n_lights * 4, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_light_range, range, (size_t)n_lights * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (layer_mask) CU(cudaMemcpyAsync(ctx->d_light_layers, layer_mask, (size_t)n_lights * 8, cudaMemcpyHostToDevice, ctx->stream));
    ctx->h_light_row.assign(light_row, light_row + n_lights); ctx->h_light_range.assign(range, range + n_lights);
    if (layer_mask) ctx->h_light_layers.assign(layer_mask, layer_mask + n_lights); else ctx->h_light_layers.clear();
    ctx->lights.n = n_lights; ctx->lights.row = ctx->d_light_row; ctx->lights.range = ctx->d_light_range;
    ctx->lights.layers = layer_mask ? ctx->d_light_layers : nullptr;
    ctx->lights_tag_dirty = true;
    return write_light_blocks(ctx);   // the objects' ordinals follow the new point-light count
}

extern "C" int32_t b200vis_set_clusterable_objects(b200vis_ctx *ctx, uint32_t n, const uint32_t *kind, const uint32_t *row,
                                                   const float *range, const uint64_t *layer_mask) {
    CHECK_CTX();
    if (n && ctx->cfg.world_size > 1)
        return fail(ctx, B200VIS_ERR_UNSUPPORTED, "set_clusterable_objects: world_size %u > 1 (rank-major ordinals would break the grouping by kind)", ctx->cfg.world_size);
    if (ctx->lights.n + n > ctx->cfg.max_lights)
        return fail(ctx, B200VIS_ERR_CAPACITY, "set_clusterable_objects: %u lights + %u objects > max_lights %u", ctx->lights.n, n, ctx->cfg.max_lights);
    if (n && (!kind || !row)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: null");
    if (n && ctx->bind.mode == B200VIS_BINDINGS_UNIFORM)
        return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: uniform cluster bindings hold point and spot lights only");
    uint32_t last_group = 0;
    for (uint32_t j = 0; j < n; ++j) {
        const uint32_t k = kind[j];
        if (k == 1u) return fail(ctx, B200VIS_ERR_UNSUPPORTED, "set_clusterable_objects: object %u is a spot light", j);
        if (k < B200VIS_CLUSTERABLE_RECT_LIGHT || k > B200VIS_CLUSTERABLE_DECAL)
            return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: object %u has kind %u", j, k);
        // push order (assign.rs:231-295): rect lights, then probes and volumes (one query, interleaved), then decals
        const uint32_t group = k == B200VIS_CLUSTERABLE_RECT_LIGHT ? 0u : k == B200VIS_CLUSTERABLE_DECAL ? 2u : 1u;
        if (group < last_group) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: object %u (kind %u) is out of push order", j, k);
        last_group = group;
        if (row[j] >= ctx->cfg.max_entities) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: object %u row %u out of range", j, row[j]);
        if (k == B200VIS_CLUSTERABLE_RECT_LIGHT && !range) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_clusterable_objects: rect lights need a range");
    }
    if (n && !ctx->d_obj_row) {
        CU(dalloc(&ctx->d_obj_row, std::max<uint32_t>(ctx->cfg.max_lights, 1)));
        CU(dalloc(&ctx->d_ord_kind, ctx->cl.max_lights));
    }
    const int32_t jrc = join_all(ctx); if (jrc) return jrc;   // the frame in flight may still read the rows
    CU(cudaStreamSynchronize(ctx->stream));
    if (n) CU(cudaMemcpy(ctx->d_obj_row, row, (size_t)n * 4, cudaMemcpyHostToDevice));
    ctx->h_obj_kind.resize(n); ctx->h_obj_range.assign(n, 0.0f); ctx->h_obj_layers.assign(n, 1ull);
    for (uint32_t j = 0; j < n; ++j) {
        ctx->h_obj_kind[j] = (uint8_t)kind[j];
        if (kind[j] == B200VIS_CLUSTERABLE_RECT_LIGHT) { ctx->h_obj_range[j] = range[j]; if (layer_mask) ctx->h_obj_layers[j] = layer_mask[j]; }
    }
    return write_light_blocks(ctx);
}

extern "C" int32_t b200vis_cluster_view_dims(const b200vis_ctx *ctx, uint32_t view, uint32_t dims[3]) {
    if (!ctx || !dims || view >= ctx->cfg.max_views) return B200VIS_ERR_INVALID_ARG;
    const DevClusterView &d = ctx->consts.cviews[view];
    for (int i = 0; i < 3; ++i) dims[i] = d.enabled ? d.dims[i] : 0u;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_cluster_view(b200vis_ctx *ctx, uint32_t view, const b200vis_cluster_view *p) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    if (view >= ctx->cfg.max_views || !p) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_cluster_view: bad view %u", view);
    DevClusterView &d = ctx->consts.cviews[view];
    memset(&d, 0, sizeof d);
    ctx->tab_x[view].clear(); ctx->tab_y[view].clear(); ctx->tab_z[view].clear(); ctx->tab_thr[view].clear();
    d.enabled = p->enabled;
    if (p->enabled) {
        const uint64_t nc = (uint64_t)p->dims[0] * p->dims[1] * p->dims[2];
        if (nc == 0 || nc > kMaxClusters) return fail(ctx, B200VIS_ERR_CAPACITY, "set_cluster_view: %llu clusters (max %d)", (unsigned long long)nc, kMaxClusters);
        if (!p->x_planes || !p->y_planes || !p->z_planes) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_cluster_view: null plane table");
        for (int i = 0; i < 3; ++i) d.dims[i] = p->dims[i];
        d.is_ortho = p->is_orthographic; d.n_clusters = (uint32_t)nc;
        memcpy(d.vfw, p->view_from_world, sizeof d.vfw); memcpy(d.cfv, p->clip_from_view, sizeof d.cfv);
        memcpy(d.scale, p->view_from_world_scale, sizeof d.scale); d.scale_max = p->view_from_world_scale_max;
        memcpy(d.frustum, p->frustum, sizeof d.frustum); d.layer_mask = p->layer_mask;
        ctx->tab_x[view].assign(p->x_planes, p->x_planes + (size_t)(p->dims[0] + 1) * 4);
        ctx->tab_y[view].assign(p->y_planes, p->y_planes + (size_t)(p->dims[1] + 1) * 4);
        ctx->tab_z[view].assign(p->z_planes, p->z_planes + (size_t)(p->dims[2] + 1) * 4);
        // view_z_to_z_slice through exact thresholds found with the host's libm (host_view.cpp)
        ctx->tab_thr[view].assign(((size_t)p->dims[2] + 3) & ~(size_t)3, NAN);
        host::z_slice_thresholds(p->cluster_factors, p->dims[2], p->is_orthographic != 0, ctx->tab_thr[view].data());
    }
    ctx->consts_dirty = true;
    return B200VIS_OK;
}

// Packs the working copy into the next pinned ring slot and issues one async copy.
static int32_t flush_consts(b200vis_ctx *ctx) {
    if (!ctx->consts_dirty) return B200VIS_OK;
    const int slot = ctx->ring_next;
    ctx->ring_next = (slot + 1) % b200vis_ctx::kRing;
    CU(cudaEventSynchronize(ctx->ring_ev[slot]));   // the copy issued kRing frames ago has long finished
    uint8_t *h = ctx->h_ring[slot];
    size_t off = (sizeof(FrameConsts) + 15) & ~(size_t)15;   // bytes; tables are float4 aligned
    for (uint32_t v = 0; v < ctx->consts.n_views && v < ctx->cfg.max_views; ++v) {
        DevClusterView &d = ctx->consts.cviews[v];
        if (!d.enabled) continue;
        std::vector<float> *tabs[4] = {&ctx->tab_x[v], &ctx->tab_y[v], &ctx->tab_z[v], &ctx->tab_thr[v]};
        uint32_t *offs[4] = {&d.x_off, &d.y_off, &d.z_off, &d.thr_off};
        for (int k = 0; k < 4; ++k) {
            *offs[k] = (uint32_t)(off / 4);
            memcpy(h + off, tabs[k]->data(), tabs[k]->size() * 4);
            off += (tabs[k]->size() * 4 + 15) & ~(size_t)15;
        }
    }
    memcpy(h, &ctx->consts, sizeof(FrameConsts));
    CU(cudaMemcpyAsync(ctx->d_blob, h, off, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaEventRecord(ctx->ring_ev[slot], ctx->stream));
    ctx->blob_used = off;
    ctx->consts_dirty = false;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_record_frame_constants(b200vis_ctx *ctx, uint32_t *slot) {
    CHECK_CTX();
    if (!slot) return fail(ctx, B200VIS_ERR_INVALID_ARG, "record_frame_constants: null");
    ctx->consts_dirty = true;
    const int32_t rc = flush_consts(ctx); if (rc) return rc;
    b200vis_ctx::Recorded r;
    r.host = ctx->consts; r.bytes = ctx->blob_used; r.dev = nullptr;
    CU(cudaMalloc(reinterpret_cast<void **>(&r.dev), r.bytes));
    CU(cudaMemcpyAsync(r.dev, ctx->d_blob, r.bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->recorded.push_back(r);
    *slot = (uint32_t)ctx->recorded.size() - 1;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_use_recorded_frame_constants(b200vis_ctx *ctx, int32_t slot) {
    if (!ctx) return B200VIS_ERR_INVALID_ARG;
    if (slot >= (int32_t)ctx->recorded.size()) return fail(ctx, B200VIS_ERR_INVALID_ARG, "use_recorded_frame_constants: bad slot %d", slot);
    ctx->replay_slot = slot < 0 ? -1 : slot;
    return B200VIS_OK;
}
static const FrameConsts &active_consts(const b200vis_ctx *ctx) {
    return ctx->replay_slot >= 0 ? ctx->recorded[ctx->replay_slot].host : ctx->consts;
}
static CullViews make_cull_views(const FrameConsts &fc) {
    CullViews c;
    memset(&c, 0, sizeof c);
    c.n_views = fc.n_views;
    for (uint32_t v = 0; v < fc.n_views && v < (uint32_t)kMaxViews; ++v) {
        c.on[v] = (fc.views[v].flags & 3u) | ((fc.views[v].layer_mask & 1ull) ? 4u : 0u); c.range_index[v] = fc.views[v].range_index; c.layers[v] = fc.views[v].layer_mask;
        for (int k = 0; k < 5; ++k) c.planes[v][k] = fc.views[v].hs[k];
    }
    return c;
}

extern "C" int32_t b200vis_set_profiling(b200vis_ctx *ctx, int32_t enabled) {
    CHECK_CTX();
    if (enabled && !ctx->prof_ev) {
        ctx->prof_ev = new cudaEvent_t[b200vis_ctx::kProfFrames][6]();
        for (int i = 0; i < b200vis_ctx::kProfFrames; ++i) for (cudaEvent_t &e : ctx->prof_ev[i]) CU(cudaEventCreate(&e));
    }
    ctx->profiling = enabled != 0;
    ctx->prof_count = 0;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_collect_stage_times_ms(b200vis_ctx *ctx, float *tile_ms, float *expand_ms, float *cluster_ms, uint32_t *frames) {
    CHECK_CTX();
    if (!ctx->prof_ev) return fail(ctx, B200VIS_ERR_NOT_READY, "profiling was never enabled");
    { const int32_t rc = join_side(ctx); if (rc) return rc; }
    CU(cudaStreamSynchronize(ctx->stream));
    double s[3] = {0, 0, 0};
    for (int i = 0; i < ctx->prof_count; ++i) {
        float t = 0;
        CU(cudaEventElapsedTime(&t, ctx->prof_ev[i][0], ctx->prof_ev[i][1])); s[0] += t;   // tile pass (main stream)
        CU(cudaEventElapsedTime(&t, ctx->prof_ev[i][5], ctx->prof_ev[i][3])); s[1] += t;   // visible-list expansion
        CU(cudaEventElapsedTime(&t, ctx->prof_ev[i][3], ctx->prof_ev[i][4])); s[2] += t;   // cluster kernels ...
        CU(cudaEventElapsedTime(&t, ctx->prof_ev[i][2], ctx->prof_ev[i][5])); s[2] += t;   // ... incl. assign + exchange when issued first
    }
    if (tile_ms) *tile_ms = (float)s[0];
    if (expand_ms) *expand_ms = (float)s[1];
    if (cluster_ms) *cluster_ms = (float)s[2];
    if (frames) *frames = (uint32_t)ctx->prof_count;
    ctx->prof_count = 0;
    return B200VIS_OK;
}

// ------------------------------------------------------------------------------------------
// multi-GPU exchange buffers
// ------------------------------------------------------------------------------------------
extern "C" int32_t b200vis_comm_unique_id(uint8_t id[B200VIS_COMM_ID_BYTES]) {
    if (!id) return B200VIS_ERR_INVALID_ARG;
    if (!g_nccl.load()) return fail(nullptr, B200VIS_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded: %s", dlerror());
    const int rc = g_nccl.GetUniqueId(id);
    if (rc) return fail(nullptr, B200VIS_ERR_CUDA, "ncclGetUniqueId: %s", g_nccl.GetErrorString(rc));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_comm_init(b200vis_ctx *ctx, const uint8_t id[B200VIS_COMM_ID_BYTES]) {
    CHECK_CTX_JOIN();
    if (!id) return fail(ctx, B200VIS_ERR_INVALID_ARG, "comm_init: null id");
    if (ctx->cl.world <= 1) return fail(ctx, B200VIS_ERR_INVALID_ARG, "comm_init: the context was created with world_size <= 1");
    if (!g_nccl.load()) return fail(ctx, B200VIS_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded: %s", dlerror());
    NcclApi::Id uid; memcpy(uid.b, id, sizeof uid.b);
    const int rc = g_nccl.CommInitRank(&ctx->nccl_comm, (int)ctx->cl.world, uid, (int)ctx->cl.rank);
    if (rc) { ctx->nccl_comm = nullptr; return fail(ctx, B200VIS_ERR_CUDA, "ncclCommInitRank: %s", g_nccl.GetErrorString(rc)); }
    if (!ctx->d_gather) CU(dalloc(&ctx->d_gather, (size_t)ctx->cl.world * ctx->slab_bytes / 4));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->cl.send = ctx->d_slab; ctx->cl.recv = ctx->d_gather;
    return B200VIS_OK;
}
// Peer-memory exchange: export allocates this rank's gathered buffer and returns its CUDA IPC handle; the host gathers the
// handles of all ranks by any means; import maps the other ranks' buffers.  From then on b200vis_run(B200VIS_STAGE_ALL)
// pushes the slab into every rank's buffer with plain NVLink stores (k_slab_push) instead of calling ncclAllGather.
extern "C" int32_t b200vis_p2p_export(b200vis_ctx *ctx, uint8_t handle[B200VIS_P2P_HANDLE_BYTES]) {
    CHECK_CTX_JOIN();
    static_assert(sizeof(cudaIpcMemHandle_t) == B200VIS_P2P_HANDLE_BYTES, "IPC handle size");
    if (!handle) return fail(ctx, B200VIS_ERR_INVALID_ARG, "p2p_export: null");
    if (ctx->cl.world <= 1 || ctx->cl.world > 8) return fail(ctx, B200VIS_ERR_INVALID_ARG, "p2p_export: world_size must be 2..8");
    if (!ctx->d_xbuf) {
        const size_t data_words = (size_t)2 * ctx->cl.world * ctx->slab_bytes / 4;
        ctx->xbuf_flag_offset = data_words;
        void *p = nullptr;   // plain cudaMalloc: the allocation must be exportable through cudaIpcGetMemHandle
        CU(cudaMalloc(&p, (data_words + 64) * 4));
        CU(cudaMemset(p, 0, (data_words + 64) * 4));
        ctx->d_xbuf = static_cast<uint32_t *>(p);
        CU(dalloc(&ctx->d_push_done, 1));
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ctx->d_xbuf));
    memcpy(handle, &h, sizeof h);
    return B200VIS_OK;
}
extern "C" int32_t b200vis_p2p_import(b200vis_ctx *ctx, const uint8_t *handles) {
    CHECK_CTX_JOIN();
    if (!handles) return fail(ctx, B200VIS_ERR_INVALID_ARG, "p2p_import: null");
    if (!ctx->d_xbuf) return fail(ctx, B200VIS_ERR_NOT_READY, "p2p_import: call b200vis_p2p_export first");
    for (uint32_t r = 0; r < ctx->cl.world; ++r) {
        if (r == ctx->cl.rank) { ctx->peer_map[r] = ctx->d_xbuf; continue; }
        if (ctx->peer_map[r]) continue;
        cudaIpcMemHandle_t h; memcpy(&h, handles + (size_t)r * B200VIS_P2P_HANDLE_BYTES, sizeof h);
        void *p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ctx, B200VIS_ERR_UNSUPPORTED, "p2p_import: cudaIpcOpenMemHandle(rank %u): %s", r, cudaGetErrorString(e)); }
        ctx->peer_map[r] = p; ctx->peer_ipc[r] = true;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    for (uint32_t r = 0; r < ctx->cl.world; ++r) {
        ctx->cl.peer[r] = static_cast<uint32_t *>(ctx->peer_map[r]);
        ctx->cl.peer_flags[r] = ctx->cl.peer[r] + ctx->xbuf_flag_offset;
    }
    ctx->cl.send = ctx->d_slab;
    ctx->p2p_ready = true;
    return B200VIS_OK;
}
// The same exchange for contexts that live in ONE process (a Bevy App is one process driving all its GPUs): no IPC handles,
// the contexts' gathered buffers are reached through plain peer access.  ctxs[r] must have been created with world_size = n and
// rank = r, each on its own device.  Afterwards the host thread simply calls b200vis_run(ctxs[r], B200VIS_STAGE_ALL) for every r
// (all launches are asynchronous; the list kernels wait for the peers' stamps on the device).
extern "C" int32_t b200vis_p2p_link(b200vis_ctx *const *ctxs, uint32_t n) {
    if (!ctxs || n < 2 || n > 8) return B200VIS_ERR_INVALID_ARG;
    for (uint32_t r = 0; r < n; ++r) {
        b200vis_ctx *ctx = ctxs[r];
        if (!ctx || ctx->cl.world != n || ctx->cl.rank != r)
            return fail(ctx, B200VIS_ERR_INVALID_ARG, "p2p_link: context %u must be created with world_size %u and rank %u", r, n, r);
        uint8_t unused[B200VIS_P2P_HANDLE_BYTES];
        const int32_t rc = b200vis_p2p_export(ctx, unused);      // allocates the gathered buffer + flags
        if (rc) return rc;
    }
    for (uint32_t r = 0; r < n; ++r) {
        b200vis_ctx *ctx = ctxs[r];
        CU(cudaSetDevice(ctx->device));
        for (uint32_t q = 0; q < n; ++q) {
            if (q != r && ctxs[q]->device != ctx->device) {
                int can = 0;
                CU(cudaDeviceCanAccessPeer(&can, ctx->device, ctxs[q]->device));
                if (!can) return fail(ctx, B200VIS_ERR_UNSUPPORTED, "p2p_link: device %d cannot access device %d", ctx->device, ctxs[q]->device);
                const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return fail(ctx, B200VIS_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); }
                cudaGetLastError();
            }
            ctx->peer_map[q] = ctxs[q]->d_xbuf; ctx->peer_ipc[q] = false;
            ctx->cl.peer[q] = ctxs[q]->d_xbuf;
            ctx->cl.peer_flags[q] = ctxs[q]->d_xbuf + ctxs[q]->xbuf_flag_offset;
        }
        CU(cudaStreamSynchronize(ctx->stream));
        ctx->cl.send = ctx->d_slab;
        ctx->p2p_ready = true;
    }
    return B200VIS_OK;
}
extern "C" int32_t b200vis_cluster_exchange_bytes(const b200vis_ctx *ctx, size_t *slab_bytes) {
    if (!ctx || !slab_bytes) return B200VIS_ERR_INVALID_ARG;
    *slab_bytes = ctx->slab_bytes;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_cluster_exchange_buffers(b200vis_ctx *ctx, void *send, void *recv) {
    CHECK_CTX_JOIN();
    if ((send == nullptr) != (recv == nullptr)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "exchange buffers: both or neither");
    CU(cudaStreamSynchronize(ctx->stream));
    if (send) {
        ctx->cl.send = static_cast<uint32_t *>(send); ctx->cl.recv = static_cast<const uint32_t *>(recv);
        CU(cudaMemsetAsync(send, 0, ctx->slab_bytes, ctx->stream));
    } else { ctx->cl.send = ctx->d_slab; ctx->cl.recv = ctx->d_slab; }
    ctx->ext_send = send; ctx->ext_recv = recv;
    return B200VIS_OK;
}

// ------------------------------------------------------------------------------------------
// run
// ------------------------------------------------------------------------------------------
// Makes the main stream wait for whatever the side stream still has in flight (cheap, asynchronous).
static int32_t join_side(b200vis_ctx *ctx) {
    if (ctx->tail_open) {   // work of an unfinished tail is on the side stream too
        CU(cudaEventRecord(ctx->ev_tile, ctx->side_stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_tile, 0));
    }
    if (ctx->side_pending) {
        for (cudaEvent_t e : ctx->ev_side) CU(cudaStreamWaitEvent(ctx->stream, e, 0));
        ctx->side_pending = false;
    }
    return B200VIS_OK;
}
// additionally waits for an in-flight publish of the visible rows (readers of the sink / of the lists call this)
static int32_t join_all(b200vis_ctx *ctx) {
    if (ctx->pub_pending) { CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_pub, 0)); ctx->pub_pending = false; }
    return join_side(ctx);
}
extern "C" int32_t b200vis_tail_stream(b200vis_ctx *ctx, void **cuda_stream) {
    if (!ctx || !cuda_stream) return B200VIS_ERR_INVALID_ARG;
    *cuda_stream = ctx->pipeline ? static_cast<void *>(ctx->side_stream) : static_cast<void *>(ctx->stream);
    return B200VIS_OK;
}
extern "C" int32_t b200vis_join(b200vis_ctx *ctx) {
    CHECK_CTX();
    return join_all(ctx);
}

extern "C" int32_t b200vis_run(b200vis_ctx *ctx, uint32_t stages) {
    CHECK_CTX();
    if (!ctx->topology_set) return fail(ctx, B200VIS_ERR_NOT_READY, "run: b200vis_set_topology has not been called");
    if ((stages & B200VIS_STAGE_CULL) && !ctx->bounds_set) return fail(ctx, B200VIS_ERR_NOT_READY, "run: bounds/flags were never uploaded");
    cudaStream_t st = ctx->stream;
    const bool do_prop = stages & B200VIS_STAGE_PROPAGATE, do_cull = stages & B200VIS_STAGE_CULL;
    const bool has_assign = stages & B200VIS_STAGE_CLUSTER_ASSIGN, has_lists = stages & B200VIS_STAGE_CLUSTER_LISTS;
    // ---- continuation of an open tail: CLUSTER_LISTS after the host's all-gather, still on the side stream --------
    if (ctx->pipeline && ctx->tail_open && stages == B200VIS_STAGE_CLUSTER_LISTS) {
        ClusterBufs cl = ctx->cl;
        cl.blob = reinterpret_cast<const float *>(ctx->open_fc);
        cudaStream_t tail = ctx->side_stream;
        launch_cluster_lists(tail, ctx->open_fc, cl, ctx->d_stats, ctx->cfg.max_views);
        if (ctx->have_sink)
            launch_publish_clusters(tail, ctx->open_fc, cl, ctx->sink_off_d, ctx->sink_idx_d, ctx->sink.cluster_capacity, ctx->d_stats,
                                    ctx->sink_stats_d, ctx->open_frame % 3u, ctx->open_frame + 1u, ctx->cfg.max_views);
        CU(cudaEventRecord(ctx->ev_side[ctx->open_frame % 3u], tail));
        ctx->side_pending = true; ctx->tail_open = false;
        CU(cudaGetLastError());
        return B200VIS_OK;
    }
    // Pipelined mode: a whole frame (or a frame up to the cluster exchange).  The tail of frame f (expand + cluster) goes to
    // the side stream and overlaps the tile passes of frames f+1 AND f+2: frame f+2's tile pass only waits for frame f's
    // list EXPANSION (it reuses frame f's visible masks and counters, two / three copies), frame f+3's for frame f's whole
    // tail (frame constants and light snapshots: three copies).  So a tail may take up to two frame periods -- which is what
    // the multi-GPU case needs, where the tail contains the cluster exchange and waits on other GPUs.
    const bool pipelined = ctx->pipeline && do_prop && do_cull && has_assign && !ctx->tail_open;
    const uint32_t frame = ctx->frame;
    const uint32_t cslot = frame % 3u, mslot = frame & 1u;
    if (pipelined) {
        if (ctx->side_pending && frame >= 2) CU(cudaStreamWaitEvent(st, ctx->ev_expand[mslot], 0));   // expansion of frame f-2
        if (ctx->side_pending && frame >= 3) CU(cudaStreamWaitEvent(st, ctx->ev_side[cslot], 0));     // tail of frame f-3
    } else {
        if (ctx->tail_open) {   // an abandoned open tail: close it so that the event chain stays consistent
            CU(cudaEventRecord(ctx->ev_side[ctx->open_frame % 3u], ctx->side_stream));
            ctx->side_pending = true; ctx->tail_open = false;
        }
        const int32_t rc = join_side(ctx); if (rc) return rc;
    }
    ClusterBufs cl = ctx->cl;
    const FrameConsts *fc;
    if (ctx->replay_slot >= 0) {   // constants already resident in HBM (recorded earlier): no host work, no copy
        fc = reinterpret_cast<const FrameConsts *>(ctx->recorded[ctx->replay_slot].dev);
    } else {
        ctx->d_blob = ctx->d_blob2[cslot];          // the side stream may still read the other two copies
        ctx->d_consts = reinterpret_cast<FrameConsts *>(ctx->d_blob);
        ctx->consts_dirty = ctx->consts_dirty || pipelined;   // each copy must be current
        const int32_t rc = flush_consts(ctx); if (rc) return rc;
        fc = ctx->d_consts;
    }
    cl.blob = reinterpret_cast<const float *>(fc);
    CullViews cvw = make_cull_views(active_consts(ctx));
    Rows R = ctx->rows;
    R.layers = ctx->have_layers ? ctx->d_layers : nullptr;
    R.layers_ext = ctx->have_layers_ext ? ctx->d_layers_ext : nullptr;
    if (ctx->have_layers_ext) memcpy(cvw.layers_ext, ctx->view_layers_ext, sizeof cvw.layers_ext);
    R.range = ctx->have_range ? ctx->d_range : nullptr;
    R.range_se = ctx->d_range_se; R.range_use_aabb = ctx->d_range_ua;
    R.range_views = ctx->d_range_views; R.n_range_views = ctx->n_range_views;
    R.rank = ctx->rank_identity ? nullptr : ctx->d_rank;
    R.row_of_rank = ctx->rank_identity ? nullptr : ctx->d_row_of_rank;
    VisibleBufs vb = ctx->vis;
    vb.mask = ctx->vis.mask + (size_t)mslot * ctx->vis.words_stride * ctx->cfg.max_views;
    const uint32_t n_pass = ctx->pass_begin.empty() ? 0 : (uint32_t)ctx->pass_begin.size() - 1;
    R.dirty = nullptr;
    R.light_snap = nullptr; R.light_ord = nullptr; R.n_lights = 0;
    if (do_prop && ctx->static_opt && n_pass > 1) {
        CU(cudaMemsetAsync(ctx->d_dirty, 0, ctx->n, st));
        R.dirty = ctx->d_dirty;
        launch_mark_dirty_global(st, R);
    }
    // Light snapshot by the tile kernel itself: needs every light row tagged with its ordinal (one-off, on change).
    bool tile_snap = false;
    if (pipelined && ctx->lights.n) {
        if (ctx->lights_tag_dirty) {
            const uint32_t one = 1;
            CU(cudaMemcpyAsync(ctx->d_tag_flag, &one, 4, cudaMemcpyHostToDevice, st));
            // rows that were lights under the previous list lose their ordinal: the whole column is rewritten
            CU(cudaMemsetAsync(ctx->d_light_ord, 0xFF, std::max<size_t>(ctx->cfg.max_entities, 1) * 4, st));
            launch_tag_lights(st, R, ctx->lights, ctx->d_light_ord, ctx->d_tag_flag);
            uint32_t ok = 0;
            CU(cudaMemcpyAsync(&ok, ctx->d_tag_flag, 4, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            ctx->lights_tagged = ok != 0; ctx->lights_tag_dirty = false;
        }
        bool any_small = false;
        for (uint32_t x : ctx->pass_small) any_small |= x != 0;
        tile_snap = ctx->lights_tagged && tile_kernel_publishes_light_snapshot() && !any_small;   // the 32-thread kernel does not publish snapshots
        if (tile_snap) {
            R.light_snap = ctx->light_snap_slot(cslot);
            R.light_ord = ctx->d_light_ord; R.n_lights = ctx->lights.n;
        }
    }
    cudaEvent_t *pe = (ctx->profiling && ctx->prof_count < b200vis_ctx::kProfFrames) ? ctx->prof_ev[ctx->prof_count++] : nullptr;
    if (pe) CU(cudaEventRecord(pe[0], st));
    if (do_prop || do_cull) {
        const uint32_t tile_stages = (do_prop ? 1u : 0u) | (do_cull ? 2u : 0u);
        if (do_prop) {
            for (uint32_t p = 0; p < n_pass; ++p) {
                const uint32_t ns = p < ctx->pass_small.size() ? ctx->pass_small[p] : 0u, b = ctx->pass_begin[p];
                if (ns) launch_propagate_cull_small(st, R, ctx->d_tiles + b, ns, cvw, vb, ctx->d_stats, tile_stages, (uint32_t)ctx->static_opt, cslot);
                if (tile_kernel_is_warp())
                    launch_tile_warp(st, R, ctx->d_wtiles + b + ns, ctx->d_sched, ctx->pass_begin[p + 1] - b - ns,
                                     cvw, vb, ctx->d_stats, tile_stages, (uint32_t)ctx->static_opt, cslot, ctx->d_tile_counter);
                else
                    launch_propagate_cull(st, R, ctx->d_tiles + b + ns, ctx->pass_begin[p + 1] - b - ns,
                                          cvw, vb, ctx->d_stats, tile_stages, (uint32_t)ctx->static_opt, cslot, ctx->d_tile_ticket, &ctx->tile_ticket_base,
                                          p < ctx->pass_named.size() && ctx->pass_named[p] != 0);
            }
        } else if (n_pass) {
            launch_cull(st, R, cvw, vb, ctx->d_stats, cslot);
        }
    }
    Lights lights = ctx->lights;
    lights.snap = nullptr;
    // Clusterable objects: snapshotted into the frame slot beside the point lights, and then every ordinal's sphere (the
    // objects' ranges included) is read through that slot.  Without objects nothing here is launched.
    ClusterObjects objs{};
    objs.n = has_assign ? ctx->n_objects() : 0u; objs.base = ctx->lights.n; objs.row = ctx->d_obj_row;
    objs.kind = objs.n ? ctx->d_ord_kind + ctx->lights.n : nullptr;
    float *slot_range = reinterpret_cast<float *>(ctx->d_lrec + (size_t)cslot * ctx->lrec_bytes + (size_t)ctx->cl.max_lights * 16);
    cudaStream_t tail = st;
    if (pipelined) {
        lights.snap = ctx->light_snap_slot(cslot);
        if (!tile_snap) launch_snapshot_lights(st, R, lights, const_cast<float4 *>(lights.snap));
        launch_snapshot_objects(st, R, objs, const_cast<float4 *>(lights.snap), slot_range);
        if (pe) CU(cudaEventRecord(pe[1], st));
        CU(cudaEventRecord(ctx->ev_tile, st));
        tail = ctx->side_stream;
        CU(cudaStreamWaitEvent(tail, ctx->ev_tile, 0));
    } else {
        if (objs.n) {      // serial: the same snapshot, behind whatever this call ran on the stream
            lights.snap = ctx->light_snap_slot(cslot);
            launch_snapshot_lights(st, R, lights, const_cast<float4 *>(lights.snap));
            launch_snapshot_objects(st, R, objs, const_cast<float4 *>(lights.snap), slot_range);
        }
        if (pe) CU(cudaEventRecord(pe[1], st));
    }
    if (objs.n) {
        lights.n += objs.n;
        lights.range = slot_range;
        lights.layers = reinterpret_cast<const uint64_t *>(ctx->d_lrec + (size_t)cslot * ctx->lrec_bytes + (size_t)ctx->cl.max_lights * 20);
    }
    if (pe) CU(cudaEventRecord(pe[2], tail));
    // Multi-GPU: the cluster exchange is the one step of the tail that waits on other GPUs, so it goes FIRST -- assign and
    // the slab push / all-gather are issued before the visible-list expansion (they do not depend on it), and the peers'
    // data travels while this rank expands its lists.
    const bool exchange_first = has_assign && has_lists && cl.world > 1;
    // Several GPUs, built-in collective: what travels is the LIGHT RECORD block (28 bytes per light: position + ViewVisibility
    // from this frame's tile pass, range, layers) instead of the cluster x light bit slabs, and every rank then runs the
    // one-launch cluster stage over all ranks' lights -- the same kernel, the same ordinals (rank * capacity + local), the same
    // Clusters feedback on every rank, and a few KB on the wire instead of V x words x 16 KB.  Used whenever the gathered bit
    // matrix fits the fused kernel's distributed shared memory (<= 6400 lights in all); B200VIS_EXCHANGE_WHAT=slabs (or a host-
    // driven / peer-store exchange) keeps the slab path.
    static int records_env = -1;
    if (records_env < 0) { const char *e = getenv("B200VIS_EXCHANGE_WHAT"); records_env = (e && e[0] == 's') ? 0 : 1; }
    const bool records = exchange_first && records_env && (ctx->nccl_comm || ctx->p2p_ready) && ctx->ext_send == nullptr &&
                         cluster_fused_fits(cl.world * cl.max_lights);
    bool fused_clusters = false;     // both cluster stages in this call and all lights at hand: one launch does assign + lists
    // Pipelined frames: the cluster branch of the tail (exchange -> cluster kernel(s) -> bindings) depends on the tile pass only,
    // not on the list expansion, and its first step may wait for other GPUs: it gets a stream of its own (`ctail`) beside the
    // expansion / visible-list publish on `tail`; the two meet again before the stats + cluster lists are published.  The
    // branch also waits for the previous frame's tail (its cluster lists and stats are single-buffered).
    static int branch_env = -1;
    if (branch_env < 0) { const char *e = getenv("B200VIS_CLUSTER_BRANCH"); branch_env = (e && e[0] == '0') ? 0 : 1; }
    const bool branch = pipelined && has_assign && has_lists && branch_env && ctx->clus_stream != nullptr;
    cudaStream_t ctail = tail;
    if (branch) {
        ctail = ctx->clus_stream;
        CU(cudaStreamWaitEvent(ctail, ctx->ev_tile, 0));
        if (ctx->side_pending && frame >= 1) CU(cudaStreamWaitEvent(ctail, ctx->ev_side[(frame + 2u) % 3u], 0));
    }
    auto issue_assign_and_exchange = [&]() -> int32_t {
        if (records) {
            if (!(pipelined && ctx->lights.n)) {      // no snapshot was taken with the tile pass: take it now (same stream order)
                Lights lsnap = ctx->lights;
                launch_snapshot_lights(ctail, R, lsnap, ctx->light_snap_slot(cslot));
            }
            if (ctx->p2p_ready) {        // peer stores over NVLink + stamps; the cluster kernel waits for every rank's stamp
                cl.p2p = 1; cl.xparity = mslot; cl.stamp = frame + 1u;
                launch_record_push(ctail, reinterpret_cast<const uint32_t *>(ctx->d_lrec + (size_t)cslot * ctx->lrec_bytes), (uint32_t)(ctx->lrec_bytes / 4), cl);
                return B200VIS_OK;
            }
            const int nrc = g_nccl.AllGather(ctx->d_lrec + (size_t)cslot * ctx->lrec_bytes, ctx->d_lrec_all, ctx->lrec_bytes / 4, kNcclUint32,
                                             ctx->nccl_comm, ctail);
            if (nrc) return fail(ctx, B200VIS_ERR_CUDA, "ncclAllGather: %s", g_nccl.GetErrorString(nrc));
            return B200VIS_OK;
        }
        if (has_assign && has_lists && cl.world == 1 && ctx->ext_send == nullptr && lights.n)
            fused_clusters = launch_cluster_fused(ctail, R, lights, fc, cl, ctx->d_stats, ctx->cfg.max_views);
        if ((stages & B200VIS_STAGE_CLUSTER_ASSIGN) && !fused_clusters)
            launch_cluster_assign(ctail, R, lights, fc, cl, ctx->d_stats, ctx->cfg.max_views);
        if (has_assign && has_lists && cl.world > 1) {
            if (ctx->p2p_ready) {
                // peer stores over NVLink + stamps; k_cluster_lists waits for every rank's stamp of this frame
                cl.p2p = 1; cl.xparity = mslot; cl.stamp = frame + 1u;
                cl.recv = ctx->d_xbuf + (size_t)mslot * cl.world * (ctx->slab_bytes / 4);
                launch_slab_push(ctail, fc, cl, ctx->d_push_done, ctx->cfg.max_views);
            } else {
                // the ONE data-path collective: rank-major all-gather of the fixed-size cluster x light slabs over NVLink
                if (!ctx->nccl_comm) return fail(ctx, B200VIS_ERR_NOT_READY, "run(ALL) with world_size > 1 needs b200vis_p2p_import or b200vis_comm_init (or run ASSIGN and LISTS separately around your own all-gather)");
                const int nrc = g_nccl.AllGather(cl.send, const_cast<uint32_t *>(cl.recv), ctx->slab_bytes / 4, kNcclUint32, ctx->nccl_comm, ctail);
                if (nrc) return fail(ctx, B200VIS_ERR_CUDA, "ncclAllGather: %s", g_nccl.GetErrorString(nrc));
            }
        }
        return B200VIS_OK;
    };
    if (exchange_first) { const int32_t rc = issue_assign_and_exchange(); if (rc) return rc; }
    if (pe) CU(cudaEventRecord(pe[5], tail));
    if (do_cull && ctx->pub_pending) { CU(cudaStreamWaitEvent(tail, ctx->ev_pub, 0)); ctx->pub_pending = false; }   // lists are rewritten
    if (do_cull) {
        launch_expand_visible(tail, vb, ctx->diff_on ? ctx->diff : DiffBufs{}, R.row_of_rank, fc, ctx->d_stats, cslot, ctx->n, ctx->cfg.max_views);
        if (pipelined) CU(cudaEventRecord(ctx->ev_expand[mslot], tail));   // this frame's masks / counters are free again
        if (ctx->diff_on && ctx->diff_sink_rows_d)
            launch_publish_visible_diff(tail, vb, ctx->diff, ctx->diff_sink_rows_d, ctx->diff_sink_cap, ctx->diff_sink_counts_d,
                                        active_consts(ctx).n_views, ctx->cfg.max_views);
    }
    if (do_cull && ctx->have_sink && ctx->sink_rows_d) {
        // posting ~1 MB of visible rows over PCIe takes tens of microseconds: in the serial (non-pipelined) case do it on the
        // side stream so it overlaps the cluster kernels; every later consumer joins the side stream
        cudaStream_t pub = tail;
        if (!pipelined) {
            CU(cudaEventRecord(ctx->ev_tile, tail));
            CU(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_tile, 0));
            pub = ctx->side_stream;
        }
        launch_publish_visible(pub, vb, ctx->d_stats, ctx->sink_rows_d, ctx->sink.visible_capacity, ctx->n, active_consts(ctx).n_views, ctx->sink_cls_d);
        if (!pipelined) { CU(cudaEventRecord(ctx->ev_pub, pub)); ctx->pub_pending = true; }
    }
    if (pe) CU(cudaEventRecord(pe[3], tail));
    if (!exchange_first) { const int32_t rc = issue_assign_and_exchange(); if (rc) return rc; }
    if (records) {
        Lights lg{};
        lg.n = cl.world * cl.max_lights; lg.per_rank = cl.max_lights; lg.block_bytes = (uint32_t)ctx->lrec_bytes; lg.blocks = ctx->d_lrec_all;
        if (ctx->p2p_ready) {       // the gathered buffer the peers wrote into: one slab-sized region per (parity, rank), the block at its front
            lg.block_bytes = (uint32_t)ctx->slab_bytes;
            lg.blocks = reinterpret_cast<const uint8_t *>(ctx->d_xbuf + (size_t)mslot * cl.world * (ctx->slab_bytes / 4));
        }
        fused_clusters = launch_cluster_fused(ctail, R, lg, fc, cl, ctx->d_stats, ctx->cfg.max_views);
        if (!fused_clusters) return fail(ctx, B200VIS_ERR_CUDA, "run: the cluster kernel could not be launched over the gathered light records");
    }
    if ((stages & B200VIS_STAGE_CLUSTER_LISTS) && !fused_clusters)
        launch_cluster_lists(ctail, fc, cl, ctx->d_stats, ctx->cfg.max_views);
    if ((stages & B200VIS_STAGE_CLUSTER_LISTS) && ctx->bind.mode) {
        BindingBufs bb = ctx->bind;
        bb.kind = ctx->n_objects() ? ctx->d_ord_kind : nullptr;
        launch_pack_cluster_bindings(ctail, fc, cl, bb, ctx->cfg.max_views);
    }
    if (branch) { CU(cudaEventRecord(ctx->ev_clus, ctail)); CU(cudaStreamWaitEvent(tail, ctx->ev_clus, 0)); }   // the branches meet
    // (b200vis_step with clusters runs CLUSTER right behind PROPAGATE|CULL: that run publishes the stats block once for both)
    if (ctx->have_sink && (do_cull || (stages & B200VIS_STAGE_CLUSTER_LISTS)) && !(ctx->step_defers_stats && !(stages & B200VIS_STAGE_CLUSTER_LISTS)))
        launch_publish_clusters(tail, fc, cl, (stages & B200VIS_STAGE_CLUSTER_LISTS) ? ctx->sink_off_d : nullptr, ctx->sink_idx_d,
                                ctx->sink.cluster_capacity, ctx->d_stats, ctx->sink_stats_d, do_cull ? cslot : (frame + 2u) % 3u, frame + (do_cull ? 1u : 0u), ctx->cfg.max_views);
    if (pe) CU(cudaEventRecord(pe[4], tail));
    if (pipelined) {
        if (has_lists) { CU(cudaEventRecord(ctx->ev_side[cslot], tail)); ctx->side_pending = true; }
        else { ctx->tail_open = true; ctx->open_frame = frame; ctx->open_fc = fc; }
    }
    CU(cudaGetLastError());
    if (do_cull) { ctx->frame++; ctx->parity = ctx->frame % 3u; }
    return B200VIS_OK;
}

// ------------------------------------------------------------------------------------------
// downloads (synchronous: the host buffers are valid on return)
// ------------------------------------------------------------------------------------------
extern "C" int32_t b200vis_download_frame_stats(b200vis_ctx *ctx, b200vis_frame_stats *out) {
    CHECK_CTX_JOIN();
    if (!out) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_frame_stats: null");
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const DevStats &s = *ctx->h_stats;
    memset(out, 0, sizeof *out);
    for (int v = 0; v < kMaxViews; ++v) {
        out->visible_count[v] = s.visible_count[v];
        out->cluster_index_count[v] = s.cl_index_count[v];
        memcpy(&out->cluster_farthest_z[v], &s.cl_farthest_bits[v], 4);
        out->cluster_index_overflow[v] = s.cl_overflow[v];
    }
    const uint32_t lp = (ctx->frame + 2u) % 3u;   // slot the last CULL frame (frame - 1) accumulated into
    out->gt_changed_count = s.changed[lp][0]; out->vv_changed_count = s.changed[lp][1]; out->frame = ctx->frame;
    ctx->last_gt_changed = out->gt_changed_count;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_download_global_transforms(b200vis_ctx *ctx, uint32_t first, uint32_t count, float *gt,
                                                      uint32_t stride, uint8_t *changed) {
    CHECK_CTX_JOIN();
    int32_t rc = check_range(ctx, first, count, "download_global_transforms"); if (rc) return rc;
    if (gt && stride != 12 && stride != 16) return fail(ctx, B200VIS_ERR_INVALID_ARG, "stride_floats must be 12 or 16");
    cudaStream_t st = ctx->stream;
    if (gt) {
        launch_pack_gt(st, ctx->rows, first, count, reinterpret_cast<float *>(ctx->d_stage), stride);
        CU(cudaMemcpyAsync(gt, ctx->d_stage, (size_t)count * stride * 4, cudaMemcpyDeviceToHost, st));
    }
    if (changed) {
        CU(cudaStreamSynchronize(st));
        launch_pack_state(st, ctx->rows, first, count, ctx->d_stage, S_GT_CHANGED);
        CU(cudaMemcpyAsync(changed, ctx->d_stage + count, count, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_view_visibility(b200vis_ctx *ctx, uint32_t first, uint32_t count, uint8_t *vv, uint8_t *changed) {
    CHECK_CTX_JOIN();
    int32_t rc = check_range(ctx, first, count, "download_view_visibility"); if (rc) return rc;
    cudaStream_t st = ctx->stream;
    launch_pack_state(st, ctx->rows, first, count, ctx->d_stage, S_VV_CHANGED);
    if (vv) CU(cudaMemcpyAsync(vv, ctx->d_stage, count, cudaMemcpyDeviceToHost, st));
    if (changed) CU(cudaMemcpyAsync(changed, ctx->d_stage + count, count, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_visible(b200vis_ctx *ctx, uint32_t view, uint32_t *rows, uint32_t capacity, uint32_t *count) {
    CHECK_CTX_JOIN();
    if (view >= ctx->cfg.max_views || !count) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_visible: bad argument");
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const uint32_t c = ctx->h_stats->visible_count[view];   // an inactive view keeps its last list (mod.rs:780-782)
    *count = c;
    if (rows) {
        if (c > capacity) return fail(ctx, B200VIS_ERR_CAPACITY, "download_visible: %u rows > capacity %u", c, capacity);
        CU(cudaMemcpyAsync(rows, ctx->vis.lists + (size_t)view * ctx->vis.list_stride, (size_t)c * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_visible_classes(b200vis_ctx *ctx, uint32_t view, uint8_t *classes, uint32_t capacity, uint32_t *count) {
    CHECK_CTX_JOIN();
    if (view >= ctx->cfg.max_views || !count) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_visible_classes: bad argument");
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const uint32_t c = ctx->h_stats->visible_count[view];
    *count = c;
    if (classes) {
        if (c > capacity) return fail(ctx, B200VIS_ERR_CAPACITY, "download_visible_classes: %u entries > capacity %u", c, capacity);
        CU(cudaMemcpyAsync(classes, ctx->vis.classes + (size_t)view * ctx->vis.list_stride, c, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_clusters(b200vis_ctx *ctx, uint32_t view, uint32_t *offsets, uint32_t *indices,
                                             uint32_t indices_capacity, uint32_t *total) {
    CHECK_CTX_JOIN();
    if (view >= ctx->cfg.max_views || !offsets || !total) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_clusters: bad argument");
    const DevClusterView &cv = active_consts(ctx).cviews[view];
    const uint32_t nc = cv.enabled ? cv.n_clusters : 0;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(offsets, ctx->cl.offsets + (size_t)view * (kMaxClusters + 1), (size_t)(nc + 1) * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *total = offsets[nc];
    if (*total > ctx->cl.index_cap) return fail(ctx, B200VIS_ERR_CAPACITY, "cluster index list overflow: %u > max_cluster_indices %u", *total, ctx->cl.index_cap);
    if (indices) {
        if (*total > indices_capacity) return fail(ctx, B200VIS_ERR_CAPACITY, "download_clusters: %u indices > capacity %u", *total, indices_capacity);
        CU(cudaMemcpyAsync(indices, ctx->cl.indices + (size_t)view * ctx->cl.index_cap, (size_t)*total * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return B200VIS_OK;
}

// ---- SURVEY 8(f) N3: check_point_light_mesh_visibility (point lights) ------------------------------------------------
extern "C" int32_t b200vis_enable_visible_diff(b200vis_ctx *ctx, int32_t enabled);
extern "C" int32_t b200vis_upload_shadow_casters(b200vis_ctx *ctx, uint32_t first, uint32_t count, const uint8_t *caster) {
    CHECK_CTX();
    if (count && !caster) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_shadow_casters: null");
    int32_t rc = check_range(ctx, first, count, "upload_shadow_casters"); if (rc) return rc;
    if (!ctx->d_caster) CU(dalloc(&ctx->d_caster, ctx->cfg.max_entities));
    // the stage reads each view's VisibleEntities as a bit set: the sets the visible-diff bookkeeping keeps.  Switched on
    // here, with the first column upload, so that the CULL stage of the coming frame already records them.
    if (!ctx->diff_on) { const int32_t rc2 = b200vis_enable_visible_diff(ctx, 1); if (rc2) return rc2; }
    CU(cudaMemcpyAsync(ctx->d_caster + first, caster, count, cudaMemcpyHostToDevice, ctx->stream));
    return B200VIS_OK;
}
static int32_t install_shadow_items(b200vis_ctx *ctx, uint32_t n_items, uint32_t list_capacity) {
    if (!list_capacity) list_capacity = std::max<uint32_t>(ctx->cfg.max_entities, 1);
    if (!ctx->diff_on) return fail(ctx, B200VIS_ERR_NOT_READY, "set_shadow_items: the visible-set bookkeeping was switched off after upload_shadow_casters");
    CU(cudaStreamSynchronize(ctx->stream));
    if (n_items > ctx->shadow_cap_lights || list_capacity > ctx->shadow_cap_list) {
        void *old[] = {ctx->d_shadow_lights, ctx->shadow.mask, ctx->shadow.chunk_count, ctx->shadow.lists, ctx->shadow.count, ctx->shadow.active};
        for (void *p : old) if (p) cudaFree(p);
        ctx->d_shadow_lights = nullptr; ctx->shadow = ShadowBufs{};
        const size_t nl = std::max<uint32_t>(n_items, ctx->shadow_cap_lights), lc = std::max<uint32_t>(list_capacity, ctx->shadow_cap_list);
        CU(dalloc(&ctx->d_shadow_lights, nl));
        CU(dalloc(&ctx->shadow.mask, nl * 6 * ctx->vis.words_stride));
        CU(dalloc(&ctx->shadow.chunk_count, nl * 6 * ctx->vis.chunks_stride));
        CU(dalloc(&ctx->shadow.lists, nl * 6 * lc));
        CU(dalloc(&ctx->shadow.count, nl * 6));
        CU(dalloc(&ctx->shadow.active, nl));
        ctx->shadow_cap_lights = (uint32_t)nl; ctx->shadow_cap_list = (uint32_t)lc;
    }
    if (n_items) CU(cudaMemcpy(ctx->d_shadow_lights, ctx->h_shadow.data(), n_items * sizeof(ShadowLight), cudaMemcpyHostToDevice));
    ctx->shadow.n_lights = n_items; ctx->shadow.lights = ctx->d_shadow_lights; ctx->shadow.caster = ctx->d_caster;
    ctx->shadow.list_cap = ctx->shadow_cap_list;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_shadow_lights(b200vis_ctx *ctx, uint32_t n_lights, const uint32_t *light_ordinals, const float *frusta,
                                             const uint64_t *layer_mask, int32_t lod_origin_range_index, uint32_t list_capacity) {
    CHECK_CTX_JOIN();
    if (n_lights && (!light_ordinals || !frusta)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_shadow_lights: null");
    if (!ctx->d_caster) return fail(ctx, B200VIS_ERR_NOT_READY, "set_shadow_lights: upload the shadow-caster column first");
    for (uint32_t i = 0; i < n_lights; ++i)
        if (light_ordinals[i] >= ctx->lights.n) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_shadow_lights: light ordinal %u >= %u lights", light_ordinals[i], ctx->lights.n);
    ctx->h_shadow.resize(n_lights);
    for (uint32_t i = 0; i < n_lights; ++i) {
        ShadowLight &s = ctx->h_shadow[i];
        memset(&s, 0, sizeof s);
        memcpy(s.planes, frusta + (size_t)i * 144, sizeof s.planes);
        s.layers = layer_mask ? layer_mask[i] : 1ull;
        s.row = ctx->h_light_row[light_ordinals[i]]; s.range = ctx->h_light_range[light_ordinals[i]]; s.kind = 0;
        s.range_index = (lod_origin_range_index >= 0 && lod_origin_range_index < 32) ? lod_origin_range_index : -1;
    }
    return install_shadow_items(ctx, n_lights, list_capacity);
}
extern "C" int32_t b200vis_set_shadow_items(b200vis_ctx *ctx, uint32_t n_items, const b200vis_shadow_item *items, uint32_t list_capacity) {
    CHECK_CTX_JOIN();
    if (n_items && !items) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_shadow_items: null");
    if (!ctx->d_caster) return fail(ctx, B200VIS_ERR_NOT_READY, "set_shadow_items: upload the shadow-caster column first");
    ctx->h_shadow.resize(n_items);
    for (uint32_t i = 0; i < n_items; ++i) {
        const b200vis_shadow_item &it = items[i];
        if (it.kind > B200VIS_SHADOW_DIRECTIONAL_CASCADE) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_shadow_items: item %u has kind %u", i, it.kind);
        if (it.kind != B200VIS_SHADOW_DIRECTIONAL_CASCADE && it.light_row >= ctx->n)
            return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_shadow_items: item %u: light row %u out of range", i, it.light_row);
        ShadowLight &s = ctx->h_shadow[i];
        memset(&s, 0, sizeof s);
        memcpy(s.planes, it.frusta, sizeof s.planes);
        s.layers = it.layer_mask; s.row = it.kind == B200VIS_SHADOW_DIRECTIONAL_CASCADE ? 0u : it.light_row; s.range = it.range;
        s.kind = it.kind; s.range_index = (it.range_view_index >= 0 && it.range_view_index < 32) ? it.range_view_index : -1;
    }
    return install_shadow_items(ctx, n_items, list_capacity);
}
extern "C" int32_t b200vis_run_shadow_culling(b200vis_ctx *ctx) {
    CHECK_CTX_JOIN();   // reads what the frame's CULL stage (incl. its tail on the side stream) left behind
    if (!ctx->d_caster || !ctx->diff.prev) return fail(ctx, B200VIS_ERR_NOT_READY, "run_shadow_culling: call b200vis_set_shadow_lights first");
    if (ctx->frame == 0) return fail(ctx, B200VIS_ERR_NOT_READY, "run_shadow_culling: run the CULL stage first");
    if (!ctx->shadow.n_lights) return B200VIS_OK;
    cudaStream_t st = ctx->stream;
    Rows R = ctx->rows;
    R.layers = ctx->have_layers ? ctx->d_layers : nullptr;
    R.range = ctx->have_range ? ctx->d_range : nullptr;
    R.rank = ctx->rank_identity ? nullptr : ctx->d_rank;
    R.row_of_rank = ctx->rank_identity ? nullptr : ctx->d_row_of_rank;
    ShadowBufs sb = ctx->shadow;
    sb.has_ranges = ctx->have_range ? 1u : 0u;
    CU(cudaMemsetAsync(sb.chunk_count, 0, (size_t)sb.n_lights * 6 * ctx->vis.chunks_stride * 4, st));
    launch_shadow_cull(st, R, sb, ctx->diff.prev, active_consts(ctx).n_views, ctx->vis.n_words, ctx->vis.n_chunks,
                       ctx->vis.words_stride, ctx->vis.chunks_stride, ctx->d_stats, (ctx->frame + 2u) % 3u);
    CU(cudaGetLastError());
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_shadow_visible(b200vis_ctx *ctx, uint32_t shadow_light, uint32_t face, uint32_t *rows, uint32_t capacity,
                                                   uint32_t *count) {
    CHECK_CTX_JOIN();
    if (shadow_light >= ctx->shadow.n_lights || face >= 6 || !count) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_shadow_visible: bad argument");
    cudaStream_t st = ctx->stream;
    const uint32_t list = shadow_light * 6 + face;
    uint32_t c = 0;
    CU(cudaMemcpyAsync(&c, ctx->shadow.count + list, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *count = c;
    if (rows) {
        if (c > capacity || c > ctx->shadow.list_cap)
            return fail(ctx, B200VIS_ERR_CAPACITY, "download_shadow_visible: %u rows > capacity %u (list capacity %u)", c, capacity, ctx->shadow.list_cap);
        if (c) CU(cudaMemcpyAsync(rows, ctx->shadow.lists + (size_t)list * ctx->shadow.list_cap, (size_t)c * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return B200VIS_OK;
}

// ---- SURVEY 8(f) N4: check_visibility_ranges and visibility_propagate_system --------------------------------------
extern "C" int32_t b200vis_upload_visibility_ranges(b200vis_ctx *ctx, uint32_t first, uint32_t count, const float *start_end,
                                                    const uint8_t *use_aabb) {
    CHECK_CTX();
    if (count && (!start_end || !use_aabb)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_visibility_ranges: null");
    int32_t rc = check_range(ctx, first, count, "upload_visibility_ranges"); if (rc) return rc;
    if (!ctx->d_range_se) {
        CU(dalloc(&ctx->d_range_se, ctx->cfg.max_entities));
        CU(dalloc(&ctx->d_range_ua, ctx->cfg.max_entities));
        CU(dalloc(&ctx->d_range_views, 32));
    }
    const size_t ou = (size_t)count * 8;
    rc = stage_in(ctx, start_end, (size_t)count * 8, 0); if (rc) return rc;
    rc = stage_in(ctx, use_aabb, count, ou); if (rc) return rc;
    launch_unpack_range_params(ctx->stream, ctx->d_range_se, ctx->d_range_ua, first, count,
                               reinterpret_cast<const float *>(ctx->d_stage), ctx->d_stage + ou);
    CU(cudaGetLastError());
    ctx->have_range = true;   // the cull kernels now take the non-SIMPLE path and fill d_range themselves
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_visibility_range_views(b200vis_ctx *ctx, uint32_t n_views, const float *positions) {
    CHECK_CTX();
    if (n_views && !positions) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_visibility_range_views: null");
    if (!ctx->d_range_views) return fail(ctx, B200VIS_ERR_NOT_READY, "set_visibility_range_views: upload the VisibilityRange columns first");
    if (n_views > 32) n_views = 32;   // view_query.iter().take(32) (range.rs:247)
    float4 h[32];
    for (uint32_t v = 0; v < n_views; ++v) h[v] = make_float4(positions[v * 3], positions[v * 3 + 1], positions[v * 3 + 2], 0.0f);
    // pageable source: the copy is staged before the call returns, and is ordered before the next frame on the stream
    if (n_views) CU(cudaMemcpyAsync(ctx->d_range_views, h, n_views * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    ctx->n_range_views = n_views;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_visibility_ranges(b200vis_ctx *ctx, uint32_t first, uint32_t count, uint32_t *mask) {
    CHECK_CTX_JOIN();
    if (count && !mask) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_visibility_ranges: null");
    int32_t rc = check_range(ctx, first, count, "download_visibility_ranges"); if (rc) return rc;
    if (!ctx->have_range) return fail(ctx, B200VIS_ERR_NOT_READY, "download_visibility_ranges: no VisibilityRange data was uploaded");
    Rows R = ctx->rows; R.range = ctx->d_range;
    launch_pack_ranges(ctx->stream, R, first, count, reinterpret_cast<uint32_t *>(ctx->d_stage));
    CU(cudaMemcpyAsync(mask, ctx->d_stage, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_upload_visibility(b200vis_ctx *ctx, uint32_t first, uint32_t count, const uint8_t *visibility) {
    CHECK_CTX();
    if (count && !visibility) return fail(ctx, B200VIS_ERR_INVALID_ARG, "upload_visibility: null");
    int32_t rc = check_range(ctx, first, count, "upload_visibility"); if (rc) return rc;
    if (!ctx->d_visibility) {   // rows never uploaded: Visibility::Inherited (the component default)
        CU(dalloc(&ctx->d_visibility, ctx->cfg.max_entities));
        CU(dalloc(&ctx->d_iv_changed, ctx->cfg.max_entities));
    }
    CU(cudaMemcpyAsync(ctx->d_visibility + first, visibility, count, cudaMemcpyHostToDevice, ctx->stream));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_propagate_visibility(b200vis_ctx *ctx) {
    CHECK_CTX_JOIN();   // the tail of an earlier frame may still read the flags column
    if (!ctx->topology_set) return fail(ctx, B200VIS_ERR_NOT_READY, "propagate_visibility: set_topology first");
    if (!ctx->d_visibility) return fail(ctx, B200VIS_ERR_NOT_READY, "propagate_visibility: upload the Visibility column first");
    const uint32_t n_pass = ctx->pass_begin.empty() ? 0 : (uint32_t)ctx->pass_begin.size() - 1;
    for (uint32_t p = 0; p < n_pass; ++p)
        launch_visibility_propagate(ctx->stream, ctx->rows, ctx->d_tiles + ctx->pass_begin[p], ctx->pass_begin[p + 1] - ctx->pass_begin[p],
                                    ctx->d_visibility, ctx->d_iv_changed);
    CU(cudaGetLastError());
    ctx->iv_ran = true;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_inherited_visibility(b200vis_ctx *ctx, uint32_t first, uint32_t count, uint8_t *inherited, uint8_t *changed) {
    CHECK_CTX_JOIN();
    int32_t rc = check_range(ctx, first, count, "download_inherited_visibility"); if (rc) return rc;
    cudaStream_t st = ctx->stream;
    launch_pack_inherited(st, ctx->rows, first, count, ctx->iv_ran ? ctx->d_iv_changed : nullptr, ctx->d_stage);
    if (inherited) CU(cudaMemcpyAsync(inherited, ctx->d_stage, count, cudaMemcpyDeviceToHost, st));
    if (changed) CU(cudaMemcpyAsync(changed, ctx->d_stage + count, count, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}

// ---- SURVEY 8(f) N2: Clusters -> ViewClusterBindings buffers ---------------------------------------------------
extern "C" int32_t b200vis_set_cluster_bindings(b200vis_ctx *ctx, uint32_t mode, const uint32_t *gpu_index_of_light, uint32_t n_map) {
    CHECK_CTX_JOIN();
    if (mode > B200VIS_BINDINGS_UNIFORM) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_cluster_bindings: mode %u", mode);
    if (gpu_index_of_light && !n_map) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_cluster_bindings: empty index map");
    if (mode == B200VIS_BINDINGS_UNIFORM && ctx->n_objects())
        return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_cluster_bindings: uniform bindings with %u clusterable objects set", ctx->n_objects());
    const size_t V = ctx->cfg.max_views;
    if (mode && !ctx->bind.oc) {
        ctx->bind.il_stride = std::max<uint32_t>(ctx->cl.index_cap, 4096u);
        CU(dalloc(&ctx->bind.oc, V * kMaxClusters * 8));
        CU(dalloc(&ctx->bind.il, V * (size_t)ctx->bind.il_stride));
        CU(dalloc(&ctx->bind.count, V * 2));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    if (gpu_index_of_light) {
        if (n_map > ctx->bind_map_cap) {
            if (ctx->d_bind_map) cudaFree(ctx->d_bind_map);
            ctx->d_bind_map = nullptr; ctx->bind_map_cap = n_map;
            CU(dalloc(&ctx->d_bind_map, n_map));
        }
        CU(cudaMemcpy(ctx->d_bind_map, gpu_index_of_light, (size_t)n_map * 4, cudaMemcpyHostToDevice));
        ctx->bind.map = ctx->d_bind_map; ctx->bind.n_map = n_map;
    } else { ctx->bind.map = nullptr; ctx->bind.n_map = 0; }
    ctx->bind.mode = mode;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_cluster_bindings(b200vis_ctx *ctx, uint32_t view, uint32_t *offsets_and_counts, uint32_t oc_capacity,
                                                     uint32_t *index_lists, uint32_t il_capacity, uint32_t *n_offsets, uint32_t *n_indices) {
    CHECK_CTX_JOIN();
    if (view >= ctx->cfg.max_views || !n_offsets || !n_indices) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_cluster_bindings: bad argument");
    if (!ctx->bind.mode) return fail(ctx, B200VIS_ERR_NOT_READY, "download_cluster_bindings: call b200vis_set_cluster_bindings first");
    cudaStream_t st = ctx->stream;
    uint32_t cnt[2] = {0, 0};
    CU(cudaMemcpyAsync(cnt, ctx->bind.count + view * 2, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_offsets = cnt[0]; *n_indices = cnt[1];
    const bool storage = ctx->bind.mode == B200VIS_BINDINGS_STORAGE;
    const uint32_t oc_words = storage ? cnt[0] * 8u : 4096u, il_words = storage ? cnt[1] : 4096u;
    if ((offsets_and_counts && oc_words > oc_capacity) || (index_lists && il_words > il_capacity))
        return fail(ctx, B200VIS_ERR_CAPACITY, "download_cluster_bindings: needs %u + %u words, capacities %u + %u", oc_words, il_words, oc_capacity, il_capacity);
    if (offsets_and_counts && oc_words)
        CU(cudaMemcpyAsync(offsets_and_counts, ctx->bind.oc + (size_t)view * kMaxClusters * 8, (size_t)oc_words * 4, cudaMemcpyDeviceToHost, st));
    if (index_lists && il_words)
        CU(cudaMemcpyAsync(index_lists, ctx->bind.il + (size_t)view * ctx->bind.il_stride, (size_t)il_words * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}

// ---- SURVEY 8(f) N1: added / removed rows of each view's VisibleEntities against last frame -----------------
static int32_t reset_visible_diff(b200vis_ctx *ctx) {
    if (ctx->diff.prev)
        CU(cudaMemsetAsync(ctx->diff.prev, 0, (size_t)ctx->vis.words_stride * ctx->cfg.max_views * 4, ctx->stream));
    return B200VIS_OK;
}
extern "C" int32_t b200vis_enable_visible_diff(b200vis_ctx *ctx, int32_t enabled) {
    CHECK_CTX_JOIN();
    if (enabled && !ctx->diff.prev) {
        const size_t V = ctx->cfg.max_views, W = ctx->vis.words_stride;
        CU(dalloc(&ctx->diff.prev, W * V));
        CU(dalloc(&ctx->diff.words, 2 * W * V));
        CU(dalloc(&ctx->diff.chunk, (size_t)ctx->vis.chunks_stride * V));
        CU(dalloc(&ctx->diff.lists, 2 * (size_t)ctx->vis.list_stride * V));
        CU(dalloc(&ctx->diff.count, 2 * V));
    }
    if (enabled && !ctx->diff_on) { const int32_t rc = reset_visible_diff(ctx); if (rc) return rc; }   // old list = empty
    ctx->diff_on = enabled != 0;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_download_visible_diff(b200vis_ctx *ctx, uint32_t view, uint32_t *added_rows, uint32_t added_capacity,
                                                 uint32_t *n_added, uint32_t *removed_rows, uint32_t removed_capacity,
                                                 uint32_t *n_removed) {
    CHECK_CTX_JOIN();
    if (view >= ctx->cfg.max_views || !n_added || !n_removed) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_visible_diff: bad argument");
    if (!ctx->diff_on) return fail(ctx, B200VIS_ERR_NOT_READY, "download_visible_diff: call b200vis_enable_visible_diff first");
    cudaStream_t st = ctx->stream;
    uint32_t cnt[2] = {0, 0};
    CU(cudaMemcpyAsync(cnt, ctx->diff.count + view * 2, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_added = cnt[0]; *n_removed = cnt[1];
    if ((added_rows && cnt[0] > added_capacity) || (removed_rows && cnt[1] > removed_capacity))
        return fail(ctx, B200VIS_ERR_CAPACITY, "download_visible_diff: %u added / %u removed rows exceed the capacities %u / %u",
                    cnt[0], cnt[1], added_capacity, removed_capacity);
    const size_t V = ctx->cfg.max_views, LS = ctx->vis.list_stride;
    if (added_rows && cnt[0]) CU(cudaMemcpyAsync(added_rows, ctx->diff.lists + (size_t)view * LS, (size_t)cnt[0] * 4, cudaMemcpyDeviceToHost, st));
    if (removed_rows && cnt[1]) CU(cudaMemcpyAsync(removed_rows, ctx->diff.lists + (V + view) * LS, (size_t)cnt[1] * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}

static int32_t map_host(b200vis_ctx *ctx, void *p, size_t bytes, uint32_t **dev);
extern "C" int32_t b200vis_set_visible_diff_sink(b200vis_ctx *ctx, uint32_t *rows, uint32_t capacity, uint32_t *counts) {
    CHECK_CTX_JOIN();
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->diff_sink_rows_d = ctx->diff_sink_counts_d = nullptr; ctx->diff_sink_cap = 0;
    if (!rows && !counts) return B200VIS_OK;
    if (!rows || !counts || !capacity) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_visible_diff_sink: rows, counts and a capacity go together");
    const size_t V = ctx->cfg.max_views;
    int32_t rc;
    uint32_t *dr = nullptr, *dc = nullptr;
    if ((rc = map_host(ctx, rows, 2 * V * (size_t)capacity * 4, &dr))) return rc;
    if ((rc = map_host(ctx, counts, 2 * V * 4, &dc))) return rc;
    ctx->diff_sink_rows_d = dr; ctx->diff_sink_counts_d = dc; ctx->diff_sink_cap = capacity;
    return B200VIS_OK;
}

static int32_t map_host(b200vis_ctx *ctx, void *p, size_t bytes, uint32_t **dev) {
    *dev = nullptr;
    if (!p) return B200VIS_OK;
    // already pinned (cudaHostAlloc / a previous cudaHostRegister, e.g. torch pinned tensors): UVA gives the device alias
    void *d = nullptr;
    if (cudaHostGetDevicePointer(&d, p, 0) != cudaSuccess) {
        cudaGetLastError();
        cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable);
        if (e != cudaSuccess && e != cudaErrorHostMemoryAlreadyRegistered)
            return fail(ctx, B200VIS_ERR_CUDA, "set_result_sink: memory is not pinned and cudaHostRegister failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
        CU(cudaHostGetDevicePointer(&d, p, 0));
    }
    *dev = static_cast<uint32_t *>(d);
    return B200VIS_OK;
}
extern "C" int32_t b200vis_set_result_sink(b200vis_ctx *ctx, const b200vis_result_sink *sink) {
    CHECK_CTX_JOIN();
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->have_sink = false;
    if (!sink) return B200VIS_OK;
    if (!sink->stats) return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_result_sink: stats is required");
    const size_t V = ctx->cfg.max_views;
    int32_t rc;
    if ((rc = map_host(ctx, sink->stats, sizeof(b200vis_frame_stats), &ctx->sink_stats_d))) return rc;
    if ((rc = map_host(ctx, sink->visible_rows, V * sink->visible_capacity * 4, &ctx->sink_rows_d))) return rc;
    { uint32_t *d = nullptr; if ((rc = map_host(ctx, sink->visible_classes, V * (size_t)sink->visible_capacity, &d))) return rc; ctx->sink_cls_d = reinterpret_cast<uint8_t *>(d); }
    if ((rc = map_host(ctx, sink->cluster_offsets, V * (kMaxClusters + 1) * 4, &ctx->sink_off_d))) return rc;
    if ((rc = map_host(ctx, sink->cluster_indices, V * (size_t)sink->cluster_capacity * 4, &ctx->sink_idx_d))) return rc;
    if ((sink->cluster_offsets == nullptr) != (sink->cluster_indices == nullptr))
        return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_result_sink: cluster_offsets and cluster_indices go together");
    ctx->sink = *sink;
    ctx->have_sink = true;
    return B200VIS_OK;
}

extern "C" int32_t b200vis_set_column_sinks(b200vis_ctx *ctx, const b200vis_column_sinks *sinks) {
    CHECK_CTX_JOIN();
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->have_colsink = false;
    ctx->col_gt_d = nullptr; ctx->col_gt_bits_d = nullptr; ctx->col_vv_bits_d = nullptr; ctx->col_vv_d = nullptr;
    if (!sinks) return B200VIS_OK;
    if (sinks->global_transforms && sinks->gt_stride_floats != 12 && sinks->gt_stride_floats != 16)
        return fail(ctx, B200VIS_ERR_INVALID_ARG, "set_column_sinks: gt_stride_floats must be 12 or 16");
    const size_t N = ctx->cfg.max_entities, W = (N + 31) / 32;
    int32_t rc;
    uint32_t *d = nullptr;
    if ((rc = map_host(ctx, sinks->global_transforms, N * sinks->gt_stride_floats * 4, &d))) return rc;
    ctx->col_gt_d = reinterpret_cast<float *>(d);
    if ((rc = map_host(ctx, sinks->gt_changed_bits, W * 4, &ctx->col_gt_bits_d))) return rc;
    if ((rc = map_host(ctx, sinks->view_visibility, N, &d))) return rc;
    ctx->col_vv_d = reinterpret_cast<uint8_t *>(d);
    if ((rc = map_host(ctx, sinks->vv_changed_bits, W * 4, &ctx->col_vv_bits_d))) return rc;
    if (!ctx->d_vv_shadow) CU(dalloc(&ctx->d_vv_shadow, N + 32));
    CU(cudaMemset(ctx->d_vv_shadow, 0xFF, N + 32));      // the host column's contents are unknown: the first write-back sends all
    ctx->colsink = *sinks;
    ctx->have_colsink = true;
    ctx->gt_aos_valid = false;
    return B200VIS_OK;
}
extern "C" int32_t b200vis_writeback_columns_ex(b200vis_ctx *ctx, uint32_t which);
extern "C" int32_t b200vis_writeback_columns(b200vis_ctx *ctx) { return b200vis_writeback_columns_ex(ctx, B200VIS_WB_GLOBAL_TRANSFORM | B200VIS_WB_VIEW_VISIBILITY); }
extern "C" int32_t b200vis_writeback_columns_ex(b200vis_ctx *ctx, uint32_t which) {
    CHECK_CTX();
    if (!ctx->have_colsink) return fail(ctx, B200VIS_ERR_NOT_READY, "writeback_columns: call b200vis_set_column_sinks first");
    // on the main stream, right behind the tile pass (and the shadow-culling stage, if the caller ran it): the tail of the
    // frame (list expansion, clusters) runs beside it on the side stream, the next frame's tile pass behind it
    const bool wgt = which & B200VIS_WB_GLOBAL_TRANSFORM, wvv = which & B200VIS_WB_VIEW_VISIBILITY;
    float *gt_sink = wgt ? ctx->col_gt_d : nullptr;
    static int dense_env = -1;
    if (dense_env < 0) { const char *e = getenv("B200VIS_WRITEBACK_DENSE"); dense_env = e ? atoi(e) : 1; }
    if (gt_sink && dense_env && (uint64_t)ctx->last_gt_changed * 2u >= ctx->n && ctx->n) {
        // most rows changed last frame (and will again): repack the whole column on the device (HBM speed) and let the copy
        // engine move it -- unchanged rows are rewritten with the bytes the host already holds.  Sparse frames take the
        // scatter kernel below instead (it touches only the changed rows).
        // (the staging copy starts as the device column in the host's layout, so that rows the scatter kernel skips -- unchanged
        // ones -- still carry the bytes the host holds)
        const uint32_t stride = ctx->colsink.gt_stride_floats;
        if (!ctx->d_gt_aos) { CU(dalloc(&ctx->d_gt_aos, (size_t)ctx->cfg.max_entities * 16)); ctx->gt_aos_valid = false; }
        if (!ctx->gt_aos_valid) { launch_pack_gt(ctx->stream, ctx->rows, 0, ctx->n, ctx->d_gt_aos, stride); ctx->gt_aos_valid = true; }
        // the same kernel as the sparse path (512-byte contiguous stores through shared memory), aimed at HBM instead of PCIe
        launch_writeback_columns(ctx->stream, ctx->rows, ctx->d_gt_aos, stride, wgt ? ctx->col_gt_bits_d : nullptr,
                                 wvv ? ctx->col_vv_d : nullptr, wvv ? ctx->col_vv_bits_d : nullptr, ctx->d_vv_shadow);
        CU(cudaMemcpyAsync(ctx->colsink.global_transforms, ctx->d_gt_aos, (size_t)ctx->n * stride * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaGetLastError());
        return B200VIS_OK;
    }
    if (gt_sink) ctx->gt_aos_valid = false;   // rows written straight to the host bypass the staging copy: it is stale from here on
    launch_writeback_columns(ctx->stream, ctx->rows, gt_sink, ctx->colsink.gt_stride_floats, wgt ? ctx->col_gt_bits_d : nullptr,
                             wvv ? ctx->col_vv_d : nullptr, wvv ? ctx->col_vv_bits_d : nullptr, ctx->d_vv_shadow);
    CU(cudaGetLastError());
    return B200VIS_OK;
}

extern "C" int32_t b200vis_download_frame(b200vis_ctx *ctx, b200vis_frame_stats *stats, uint32_t *visible_rows,
                                          uint32_t visible_capacity, uint32_t *cluster_offsets,
                                          uint32_t *cluster_indices, uint32_t cluster_capacity) {
    CHECK_CTX_JOIN();
    if (!stats) return fail(ctx, B200VIS_ERR_INVALID_ARG, "download_frame: null stats");
    cudaStream_t st = ctx->stream;
    const FrameConsts &fc = active_consts(ctx);
    const uint32_t V = std::min<uint32_t>(fc.n_views, ctx->cfg.max_views);
    // sync 1: the stats block and the cluster offsets (both small, fixed size) tell how much else to copy
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, st));
    if (cluster_offsets)
        for (uint32_t v = 0; v < V; ++v) {
            const uint32_t nc = fc.cviews[v].enabled ? fc.cviews[v].n_clusters : 0;
            CU(cudaMemcpyAsync(cluster_offsets + (size_t)v * (kMaxClusters + 1), ctx->cl.offsets + (size_t)v * (kMaxClusters + 1),
                               (size_t)(nc + 1) * 4, cudaMemcpyDeviceToHost, st));
        }
    CU(cudaStreamSynchronize(st));
    int32_t rc = b200vis_download_frame_stats(ctx, stats);   // formats h_stats (re-copies 200 bytes)
    if (rc) return rc;
    // sync 2: exact-size list copies
    for (uint32_t v = 0; v < V; ++v) {
        if (visible_rows) {
            const uint32_t c = stats->visible_count[v];
            if (c > visible_capacity) return fail(ctx, B200VIS_ERR_CAPACITY, "download_frame: view %u has %u visible rows > capacity %u", v, c, visible_capacity);
            CU(cudaMemcpyAsync(visible_rows + (size_t)v * visible_capacity, ctx->vis.lists + (size_t)v * ctx->vis.list_stride, (size_t)c * 4, cudaMemcpyDeviceToHost, st));
        }
        if (cluster_indices && cluster_offsets && fc.cviews[v].enabled) {
            const uint32_t total = cluster_offsets[(size_t)v * (kMaxClusters + 1) + fc.cviews[v].n_clusters];
            if (total > cluster_capacity || total > ctx->cl.index_cap)
                return fail(ctx, B200VIS_ERR_CAPACITY, "download_frame: view %u has %u cluster indices > capacity", v, total);
            CU(cudaMemcpyAsync(cluster_indices + (size_t)v * cluster_capacity, ctx->cl.indices + (size_t)v * ctx->cl.index_cap, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
        }
    }
    CU(cudaStreamSynchronize(st));
    return B200VIS_OK;
}

extern "C" int32_t b200vis_step(b200vis_ctx *ctx, uint32_t n_changed, const uint32_t *rows, const float *trs,
                                uint32_t n_cameras, const b200vis_camera *cameras, const b200vis_cluster_config *cfg, uint32_t flags) {
    CHECK_CTX();
    if (n_cameras > ctx->cfg.max_views || (n_cameras && !cameras)) return fail(ctx, B200VIS_ERR_INVALID_ARG, "step: bad camera array");
    int32_t rc;
    using clk = std::chrono::steady_clock;
    auto t0 = clk::now();
    auto lap = [&](int i) { auto t1 = clk::now(); ctx->step_t[i] += std::chrono::duration<double>(t1 - t0).count(); t0 = t1; };
    if (n_changed && (rc = b200vis_upload_transforms_scattered(ctx, n_changed, rows, trs))) return rc;
    lap(0);
    if ((rc = b200vis_set_view_count(ctx, n_cameras))) return rc;
    const bool clusters = cfg != nullptr && ctx->lights.n + ctx->n_objects() > 0;
    // frusta first, so the tile pass starts at once; the per-view cluster prologue (plane tables, z thresholds: tens of
    // microseconds of host maths) is computed while that kernel runs, then the cluster stage is enqueued behind it
    for (uint32_t v = 0; v < n_cameras; ++v)
        if ((rc = b200vis_update_camera(ctx, v, &cameras[v], nullptr, nullptr, nullptr))) return rc;
    lap(1);
    ctx->step_defers_stats = clusters;
    rc = b200vis_run(ctx, B200VIS_STAGE_PROPAGATE | B200VIS_STAGE_CULL);
    ctx->step_defers_stats = false;
    if (rc) return rc;
    if ((flags & B200VIS_STEP_WRITEBACK) && (rc = b200vis_writeback_columns(ctx))) return rc;
    lap(2);
    if (clusters) {
        for (uint32_t v = 0; v < n_cameras; ++v)
            if ((rc = b200vis_update_camera(ctx, v, &cameras[v], cfg, &ctx->auto_fb[v], nullptr))) return rc;
        lap(3);
        if ((rc = b200vis_run(ctx, B200VIS_STAGE_CLUSTER))) return rc;
        lap(4);
    }
    ctx->step_n++;
    if (!(flags & B200VIS_STEP_WAIT)) return B200VIS_OK;
    if ((rc = join_all(ctx))) return rc;
    const b200vis_frame_stats *st = nullptr;
    b200vis_frame_stats local;
    if (ctx->have_sink) { CU(cudaStreamSynchronize(ctx->stream)); st = ctx->sink.stats; }
    else { if ((rc = b200vis_download_frame_stats(ctx, &local))) return rc; st = &local; }
    lap(5);
    ctx->last_gt_changed = st->gt_changed_count;
    if (clusters)
        for (uint32_t v = 0; v < n_cameras; ++v) {   // Clusters::last_frame_* (assign.rs:810-811)
            b200vis_cluster_feedback &fb = ctx->auto_fb[v];
            if (!ctx->consts.cviews[v].enabled) continue;
            fb.has_farthest_z = 1; fb.farthest_z = st->cluster_farthest_z[v];
            fb.has_index_count = 1; fb.index_count = st->cluster_index_count[v];
        }
    return B200VIS_OK;
}
