// device_types.cuh -- structures shared by the kernels and the host runtime of libb200vis.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200vis {

constexpr int kTileRows = 256;          // rows per tile == threads per CTA of the tile kernel
constexpr int kMaxViews = 8;
constexpr int kMaxClusters = 4096;
constexpr int kChunkWords = 1024;       // visible-mask words per compaction chunk (32768 rows)
constexpr uint32_t kNoParent = 0xFFFFFFFFu;
constexpr uint32_t kDetached = 0xFFFFFFFEu;

// row flag byte (include/b200vis.h)
constexpr uint32_t F_INHERITED = 0x01, F_AABB = 0x02, F_SPHERE = 0x04, F_NO_FRUSTUM = 0x08, F_RANGE = 0x10,
                   F_NO_CPU_CULL = 0x20, F_SPHERE_GT = 0x40, F_TCHANGED = 0x80;
// per-row device state byte: bits 0-1 ViewVisibility, 4 gt_changed, 5 vv_changed, 6 visited, 7 has_class
constexpr uint32_t S_VV = 0x03, S_GT_CHANGED = 0x10, S_VV_CHANGED = 0x20, S_VISITED = 0x40, S_HAS_CLASS = 0x80;
// topo word: parent_local[0:9) local_depth[9:18) | flags
constexpr uint32_t T_ROOT = 1u << 28, T_HAS_CHILDREN = 1u << 29, T_EXT_PARENT = 1u << 30, T_DETACHED = 1u << 31;

struct Tile {               // one CTA's work: a contiguous, (mostly) hierarchy-closed row range
    uint32_t base;
    uint16_t n_rows;
    uint16_t n_levels;      // in-tile depth levels (1 for flat rows)
    uint32_t warp_sync_mask; // bit l (1 <= l < 32): every row of level l has its parent in the same warp,
                             //   so __syncwarp orders the shared-memory hand-over instead of a CTA barrier
    uint32_t top_levels;     // K: every row of in-tile depth < K is one of the tile's first 32 rows (a BFS-ordered tree: its top
                             //   5 levels), so ONE warp can walk those levels on its own (k_propagate_cull_scout), a tile ahead
    unsigned long long lvl_warps;   // tiles of 2..8 levels: nibble l (1 <= l < n_levels) = how many of the tile's warps hold a row of
                             //   level l-1 (producers) or level l (consumers).  Level l is then handed over through hardware named
                             //   barrier l with exactly those warps: consumers bar.sync, pure producers bar.arrive and move on, all
                             //   other warps never touch it (k_propagate_cull_tma).  0: the kernel walks with CTA-wide barriers
};

// The same tile as one WARP's work (k_tile_warp): the warp walks the tile in chunks of 32 schedule slots.  The schedule
// (one byte per slot: local row, 0xFF = padding) lists the tile's rows in (in-tile depth, row) order, so that a row's
// parent always sits in an earlier chunk or at a lower level of the same chunk; rows with in-tile children own one of
// the warp's kWarpParentSlots shared-memory GlobalTransform slots.
constexpr int kWarpParentSlots = 128;
constexpr int kWarpChunks = kTileRows / 32;
struct WarpTile {
    uint32_t base;
    uint16_t n_rows;
    uint8_t n_chunks;         // schedule slots / 32
    uint8_t contig;           // bit c: in chunk c, row - lane is the same for all occupied lanes (ballot bits map to mask bits)
    uint32_t sched;           // index of the tile's 256-byte block in the schedule array
    uint32_t pad;
    uint32_t nonroot[kWarpChunks];   // per chunk: slots holding a row whose parent is in this tile
};
// wtopo word of k_tile_warp: depth[0:8) own parent-slot[8:15) parent's parent-slot[15:22) W_HAS_SLOT | T_* flags (bits 28-31)
constexpr uint32_t W_HAS_SLOT = 1u << 22;   // the row has children in its own tile: it parks its GlobalTransform in a slot

// SoA mirror of the ECS columns in HBM.  Every array is indexed by row.
struct Rows {
    uint32_t n;
    // Transform: 40 B/row  (A = t.xyz, s.x | B = q.xyzw | C = s.y, s.z)
    float4 *trsA; float4 *trsB; float2 *trsC;
    // GlobalTransform: 48 B/row, the three rows of the 3x4 matrix: gtK = (X[k], Y[k], Z[k], T[k])
    float4 *gt0; float4 *gt1; float4 *gt2;
    // Aabb / Sphere: 24 B/row (A = c.xyz, h.x | B = h.y, h.z)
    float4 *bndA; float2 *bndB;
    uint8_t *flags;          // B200VIS_F_* | F_TCHANGED
    uint8_t *state;          // S_*
    uint32_t *topo;          // T_* | local parent | local depth
    const uint32_t *wtopo;   // T_* | depth | parent slots, for k_tile_warp
    const uint32_t *parent;  // global parent row (read only for T_EXT_PARENT rows)
    const uint64_t *layers;  // RenderLayers first block, or nullptr
    const uint64_t *layers_ext;  // [n][3] RenderLayers blocks 1..3 (layers 64..255), or nullptr (render_layers.rs:20-23)
    uint32_t *range;         // VisibleEntityRanges bitmask, or nullptr
    // SURVEY 8(f) N4: VisibilityRange columns; when resident the cull phase computes `range` itself
    const float2 *range_se;      // (start_margin.start, end_margin.end), or nullptr
    const uint8_t *range_use_aabb;
    const float4 *range_views;   // translations of the (<= 32) views check_visibility_ranges indexes
    uint32_t n_range_views;
    const uint32_t *rank;    // position in Entity::to_bits() order, or nullptr when rank == row
    const uint32_t *row_of_rank;
    uint8_t *dirty;          // global TransformTreeChanged bytes (multi-pass plans only), or nullptr
    float4 *light_snap;      // when non-null, rows flagged F_SPHERE_GT look up their light ordinal in light_ord (written by
                             //   k_tag_lights; 0xFFFFFFFF = not a light) and publish (translation, visible) here at the end
                             //   of the tile pass
    const uint32_t *light_ord;   // per row: ordinal in the b200vis_set_lights arrays, or 0xFFFFFFFF
    uint32_t n_lights;
};

struct DevView {
    float4 hs[6];
    unsigned long long layer_mask;
    uint32_t flags;
    int32_t range_index;
};

// What the cull phase reads per view, passed BY VALUE as a __grid_constant__ kernel parameter so that
// every plane component is a constant-bank operand (772 bytes of the 4 KB parameter space).
struct CullViews {
    uint32_t n_views;
    uint32_t on[kMaxViews];            // bit0 camera.is_active, bit1 NoCpuCulling camera, bit2 default layer in the view's mask
    int32_t range_index[kMaxViews];
    unsigned long long layers[kMaxViews];
    unsigned long long layers_ext[kMaxViews][3];   // the views' RenderLayers blocks 1..3
    float4 planes[kMaxViews][5];       // L,R,T,B,Near (the far plane is never used by culling)
};

struct DevClusterView {
    uint32_t enabled, dims[3], is_ortho, n_clusters;
    uint32_t x_off, y_off;   // offsets (in floats) of the plane tables inside the frame blob
    float vfw[16];           // view_from_world, column major
    float cfv[16];           // clip_from_view
    float scale[3];          // view_from_world_scale
    float scale_max;
    float4 frustum[6];
    unsigned long long layer_mask;
    uint32_t z_off, thr_off; // z plane table, z-slice thresholds on u = -view_z
};

struct FrameConsts {
    uint32_t n_views, pad[3];
    DevView views[kMaxViews];
    DevClusterView cviews[kMaxViews];
};

// counters written by the kernels (one D2H copy per frame)
struct DevStats {
    uint32_t visible_count[kMaxViews];     // written by the expand kernel for ACTIVE views only
    uint32_t cl_index_count[kMaxViews];    // outputs of the last cluster frame (copied from the accumulators
    uint32_t cl_farthest_bits[kMaxViews];  //   by the lists kernel, which also re-zeroes them)
    uint32_t cl_overflow[kMaxViews];
    uint32_t cl_acc_index[kMaxViews];      // accumulators of the assign kernel
    uint32_t cl_acc_far[kMaxViews];        // float bits; values > 0 only, so integer max == float max
    uint32_t changed[3][2];                // [frame % 3][0 = gt, 1 = vv]; the expand kernel of frame f zeroes the
                                           // slot frame f+2 accumulates into (frame f+1 may already be running)
};

struct VisibleBufs {
    uint32_t n_words;        // ceil(n/32)
    uint32_t n_chunks;       // ceil(n_words / kChunkWords)
    uint32_t words_stride;   // words per view
    uint32_t chunks_stride;  // chunk counters per view
    uint32_t *mask;          // [V][words_stride], bit = rank (two copies, the host passes frame % 2's)
    uint32_t *chunk_count;   // [3][V][chunks_stride], slot = frame % 3
    uint32_t *lists;         // [V][list_stride] rows, ascending Entity::to_bits()
    uint32_t list_stride;
    uint8_t *classes;        // [V][list_stride] VisibilityClass mask of each listed row (the shim splits the list per class)
    const uint8_t *cls;      // per row: VisibilityClass mask (bit k = class k of the shim's registry)
};

// SURVEY 8(f) N1: RenderVisibleEntitiesClass::update_cpu_culled_entities on the device -- the added / removed
// lists between last frame's and this frame's sorted visible list of a view (all pointers null = disabled)
struct DiffBufs {
    uint32_t *prev;          // [V][words_stride] visible set of the last frame the view was active, bit = rank
    uint32_t *words;         // [2][V][words_stride] added / removed bits of this frame
    uint32_t *chunk;         // [V][chunks_stride] per chunk: added count | removed count << 16
    uint32_t *lists;         // [2][V][list_stride] rows: added, removed (ascending Entity::to_bits())
    uint32_t *count;         // [V][2]
};

struct Lights {
    uint32_t n;
    const float4 *snap;      // optional (pos.xyz, visible) snapshot taken right after the tile pass, or nullptr
    const uint32_t *row;
    const float *range;
    const uint64_t *layers;  // or nullptr
    // Several GPUs, light-RECORD exchange: `blocks` holds every rank's light block (gathered), light li = rank * per_rank + j
    // is entry j of block `rank`.  A block = float4 snap[per_rank] | float range[per_rank] | uint64 layers[per_rank]
    // (28 bytes per light: what assign_objects_to_clusters needs of a light).  per_rank == 0: the flat arrays above.
    uint32_t per_rank, block_bytes;
    const uint8_t *blocks;
};
#ifdef __CUDACC__
__device__ __forceinline__ float4 light_snap_of(const Lights &L, uint32_t li) {
    if (!L.per_rank) return L.snap[li];
    const uint32_t r = li / L.per_rank, j = li - r * L.per_rank;
    return reinterpret_cast<const float4 *>(L.blocks + (size_t)r * L.block_bytes)[j];
}
__device__ __forceinline__ float light_range_of(const Lights &L, uint32_t li) {
    if (!L.per_rank) return L.range[li];
    const uint32_t r = li / L.per_rank, j = li - r * L.per_rank;
    return reinterpret_cast<const float *>(L.blocks + (size_t)r * L.block_bytes + (size_t)L.per_rank * 16u)[j];
}
__device__ __forceinline__ unsigned long long light_layers_of(const Lights &L, uint32_t li) {
    if (!L.per_rank) return L.layers ? L.layers[li] : 1ull;
    const uint32_t r = li / L.per_rank, j = li - r * L.per_rank;
    return reinterpret_cast<const unsigned long long *>(L.blocks + (size_t)r * L.block_bytes + (size_t)L.per_rank * 20u)[j];
}
#endif

// b200vis_set_clusterable_objects: object j (row[j], kind[j]) is cluster ordinal base + j, base = the point-light count.
// k_snapshot_objects writes its (translation, visible) and -- for probes and decals -- its radius into the frame slot's
// light block, so that the cluster kernels read every ordinal's sphere the same way.
constexpr uint32_t kKindPoint = 0, kKindRect = 2, kKindReflectionProbe = 3, kKindIrradianceVolume = 4, kKindDecal = 5;
struct ClusterObjects {
    uint32_t n, base;
    const uint32_t *row;
    const uint8_t *kind;     // [n]
};

struct ClusterBufs {
    uint32_t words;          // mask words per rank = ceil(max_lights/32)
    uint32_t max_lights;     // per rank
    uint32_t world, rank;
    uint32_t max_views;
    uint32_t index_cap;      // per view
    uint32_t *send;          // this rank's slab: [V][words][kMaxClusters] + trailer [kMaxViews] (the rank's farthest_z candidate per
                             //   view, float bits: it travels with the slab, so that Clusters::last_frame_* are identical on all ranks)
    const uint32_t *recv;    // gathered: [world] slabs
    uint32_t slab_words;     // words per slab incl. the trailer == the rank stride of recv
    const float *blob;       // frame blob base: FrameConsts, then the packed per-view tables
    uint32_t *offsets;       // [V][kMaxClusters+1]
    uint32_t *indices;       // [V][index_cap]
    // peer-memory exchange (b200vis_p2p_import): every rank's gathered buffer [2 parities][world][slab] as mapped into this
    // process, the flag words behind it [2][world], and this frame's parity / stamp.  p2p == 0: recv was filled by a collective.
    uint32_t p2p, xparity, stamp, pad;
    uint32_t *peer[8];
    uint32_t *peer_flags[8];
};

// SURVEY 8(f) N3: check_point_light_mesh_visibility (bevy_light/src/lib.rs:517-668) for the shadow-casting point lights
struct ShadowLight {         // one shadow item: a point light (six cubemap faces), a spot light or one directional-light cascade (frustum 0)
    float4 planes[6][6];     // frustum (face), half space (normal, d)
    unsigned long long layers;
    uint32_t row;            // point / spot: the light's row (range sphere centre = its GlobalTransform translation)
    float range;
    uint32_t kind;           // 0 point, 1 spot, 2 directional cascade (no range sphere, near plane not tested, always active)
    int32_t range_index;     // bit of the VisibleEntityRanges masks that gates ranged rows: shadow LOD origin / the cascade's view; -1 none
    uint32_t pad[2];
};
struct ShadowBufs {
    uint32_t n_lights;       // shadow lights this frame
    const ShadowLight *lights;
    const uint8_t *caster;   // per row: in visible_entity_query (Mesh3d, no NotShadowCaster, no DirectionalLight)
    uint32_t has_ranges;     // a VisibleEntityRanges resource exists
    uint32_t *mask;          // [n_lights * 6][words_stride], bit = rank; zeroed by the expand kernel as it reads
    uint32_t *chunk_count;   // [n_lights * 6][chunks_stride]
    uint32_t *lists;         // [n_lights * 6][list_cap]
    uint32_t *count;         // [n_lights * 6]
    uint32_t list_cap;
    uint32_t *active;        // [n_lights]: the light is in some view's VisibleEntities (written by k_shadow_select)
};

// SURVEY 8(f) N2: the ViewClusterBindings wire format (bevy_pbr/src/cluster/mod.rs:584-800) packed on the device
struct BindingBufs {
    uint32_t mode;           // 0 off, 1 storage buffers, 2 uniform buffers
    const uint32_t *map;     // GlobalClusterableObjectMeta::entity_to_index per light ordinal, or nullptr (identity)
    uint32_t n_map;
    uint32_t *oc;            // [V][kMaxClusters * 8]  storage: 2 x uvec4 per cluster; uniform: the first 4096 words
    uint32_t *il;            // [V][il_stride]         storage: one u32 per index; uniform: the first 4096 words
    uint32_t il_stride;
    uint32_t *count;         // [V][2] n_offsets, n_indices
    const uint8_t *kind;     // per cluster ordinal: kKind* (storage mode splits the counts by kind), or nullptr (all point lights)
};

}  // namespace b200vis
