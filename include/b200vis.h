/*
 * b200vis.h -- C ABI of libb200vis.so: the B200-native replacement for the
 * per-frame visibility pipeline of bevyengine/bevy 0.20.0-dev
 * (propagate -> cull -> cluster).
 *
 * The reference has NO FFI seam for these stages: they are plain Rust systems.
 * Each entry point below therefore cites the reference system / type whose
 * work it takes over; the Rust-side binding a maintainer adds (a
 * `B200VisibilityPlugin` calling these through `extern "C"`) is shown in
 * INTEGRATION.md and rust/b200vis_plugin.rs.
 *
 * Conventions: every call returns an int32 status (0 = B200VIS_OK); no
 * unwinding, no global state; the caller owns all host memory, the library
 * owns all device memory; a context is thread-compatible (one caller at a
 * time), like a Bevy system holding `ResMut`.  Plain pointers and sizes only.
 * Rows are the caller's mirror of ECS archetype rows (one row per entity that
 * has Transform + GlobalTransform); ranges are [first_row, first_row+count).
 */
#ifndef B200VIS_H
#define B200VIS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200VIS_ABI_VERSION 2
#if defined(__GNUC__)
#define B200VIS_API __attribute__((visibility("default")))
#else
#define B200VIS_API
#endif

/* ---- status codes -------------------------------------------------------- */
enum {
    B200VIS_OK = 0,
    B200VIS_ERR_INVALID_ARG = 1,
    B200VIS_ERR_CUDA = 2,            /* CUDA runtime error or no CUDA device: see b200vis_last_error */
    B200VIS_ERR_OUT_OF_MEMORY = 3,
    B200VIS_ERR_HIERARCHY_CYCLE = 4, /* the shim must panic!(): crates/bevy_transform/src/systems.rs:715, test :1101 */
    B200VIS_ERR_PARENT_OUT_OF_RANGE = 5,
    B200VIS_ERR_CAPACITY = 6,        /* more rows / lights / views / indices than the context was created for */
    B200VIS_ERR_NOT_READY = 7,       /* a stage was run before its inputs were uploaded */
    B200VIS_ERR_UNSUPPORTED = 8
};

/* parent_row sentinels (b200vis_set_topology) */
#define B200VIS_NO_PARENT 0xFFFFFFFFu /* no ChildOf: a hierarchy root or a flat entity */
#define B200VIS_DETACHED  0xFFFFFFFEu /* has ChildOf, but the parent lacks Transform/GlobalTransform: never
                                         reached by propagation (NodeQuery, systems.rs:752-764) */

/* per-row flag byte (b200vis_upload_bounds) */
#define B200VIS_F_INHERITED_VISIBLE  0x01u /* InheritedVisibility::get() (visibility/mod.rs:164) */
#define B200VIS_F_HAS_AABB           0x02u /* Option<&Aabb> is Some (primitives.rs:63-68) */
#define B200VIS_F_HAS_SPHERE         0x04u /* Option<&Sphere> is Some (primitives.rs:197-211) */
#define B200VIS_F_NO_FRUSTUM_CULLING 0x08u /* Has<NoFrustumCulling> */
#define B200VIS_F_HAS_VIS_RANGE      0x10u /* Has<VisibilityRange> (visibility/range.rs) */
#define B200VIS_F_NO_CPU_CULLING     0x20u /* With<NoCpuCulling>: row is outside the visibility queries */
#define B200VIS_F_SPHERE_FROM_GT     0x40u /* Sphere.center is the row's own GlobalTransform translation, i.e. the
                                              steady state of update_point_light_bounding_spheres
                                              (crates/bevy_light/src/point_light.rs:195-209) */
/* bit 0x80 is owned by the library: "Transform changed since the last propagate" */

/* per-view flag byte */
#define B200VIS_VIEW_ACTIVE          0x01u /* camera.is_active (visibility/mod.rs:780) */
#define B200VIS_VIEW_NO_CPU_CULLING  0x02u /* Has<NoCpuCulling> on the camera (visibility/mod.rs:823) */

/* stages for b200vis_run */
#define B200VIS_STAGE_PROPAGATE      0x1u  /* TransformSystems::Propagate */
#define B200VIS_STAGE_CULL           0x2u  /* reset_view_visibility + check_visibility_cpu_culling +
                                              mark_newly_hidden_entities_invisible */
#define B200VIS_STAGE_CLUSTER_ASSIGN 0x4u  /* assign_objects_to_clusters: lights -> cluster x light bitmask slab */
#define B200VIS_STAGE_CLUSTER_LISTS  0x8u  /* bitmask (after the optional all-gather) -> ordered index lists */
#define B200VIS_STAGE_CLUSTER        (B200VIS_STAGE_CLUSTER_ASSIGN | B200VIS_STAGE_CLUSTER_LISTS)
#define B200VIS_STAGE_ALL            0xFu

#define B200VIS_MAX_VIEWS     8u
#define B200VIS_MAX_CLUSTERS  4096u  /* assign.rs:410-413 */

typedef struct b200vis_ctx b200vis_ctx;

typedef struct b200vis_config {
    int32_t  device;              /* CUDA device ordinal */
    uint32_t max_entities;        /* row capacity */
    uint32_t max_lights;          /* cluster ordinals this context (this rank's shard) may hold: point lights plus the
                                     objects of b200vis_set_clusterable_objects */
    uint32_t max_views;           /* <= B200VIS_MAX_VIEWS */
    uint32_t max_cluster_indices; /* per-view capacity of the cluster index list (0 => 1<<20) */
    uint32_t world_size;          /* ranks sharing the cluster exchange (0/1 => single GPU) */
    uint32_t rank;
    uint32_t reserved;
} b200vis_config;

/* One camera: what check_visibility_cpu_culling reads per view
 * (view_query, crates/bevy_camera/src/visibility/mod.rs:750-757). */
typedef struct b200vis_view {
    float    half_spaces[6][4];   /* Frustum: normal.xyz, d; order L,R,T,B,Near,Far (view_frustum.rs:25-34) */
    uint64_t layer_mask;          /* RenderLayers first block; default layer 0 => 1 */
    uint8_t  flags;               /* B200VIS_VIEW_* */
    int8_t   range_view_index;    /* bit index in VisibleEntityRanges, -1 if the view is not in it */
    uint8_t  pad[6];
} b200vis_view;

/* Per-view constants of assign_objects_to_clusters, computed on the host exactly
 * where the reference computes them (assign.rs:324-485); b200vis_host_cluster_view_setup
 * fills one of these from a camera + ClusterConfig + last frame's feedback. */
typedef struct b200vis_cluster_view {
    uint32_t enabled;             /* 0 => clusters.clear() path (ClusterConfig::None / empty viewport) */
    uint32_t dims[3];             /* Clusters::dimensions */
    uint32_t tile_size[2];        /* Clusters::tile_size (reported back, unused on the device) */
    uint32_t is_orthographic;
    float    near_z, far_z;       /* Clusters::near / far */
    float    cluster_factors[2];  /* calculate_cluster_factors (assign.rs:817-832) */
    float    view_from_world[16]; /* Mat4, column major */
    float    clip_from_view[16];
    float    view_from_world_scale[3];
    float    view_from_world_scale_max;
    float    frustum[6][4];       /* the view's Frustum, all six planes are used (assign.rs:496) */
    uint64_t layer_mask;
    const float *x_planes;        /* [(dims.x+1)][4] HalfSpace normal_d, view space (assign.rs:455-475) */
    const float *y_planes;        /* [(dims.y+1)][4] */
    const float *z_planes;        /* [(dims.z+1)][4] */
} b200vis_cluster_view;

/* Small per-frame result block (one D2H copy): what the shim writes back into
 * VisibleEntities / Clusters bookkeeping. */
typedef struct b200vis_frame_stats {
    uint32_t visible_count[B200VIS_MAX_VIEWS];       /* entries in each view's visible list */
    uint32_t cluster_index_count[B200VIS_MAX_VIEWS]; /* -> Clusters::last_frame_total_cluster_index_count */
    float    cluster_farthest_z[B200VIS_MAX_VIEWS];  /* -> Clusters::last_frame_farthest_z */
    uint32_t cluster_index_overflow[B200VIS_MAX_VIEWS]; /* 1 if the list did not fit max_cluster_indices */
    uint32_t gt_changed_count;                       /* rows whose Changed<GlobalTransform> fired */
    uint32_t vv_changed_count;                       /* rows whose Changed<ViewVisibility> fired */
    uint32_t frame;                                  /* frames run so far */
    uint32_t pad;
} b200vis_frame_stats;

/* ClusterConfig + GlobalClusterSettings + viewport, and last frame's Clusters feedback: inputs of the
 * host-side per-view prologue (b200vis_update_camera / b200vis_host_cluster_view_setup). */
typedef struct b200vis_cluster_config {      /* ClusterConfig + GlobalClusterSettings + viewport */
    uint32_t kind;               /* 0 None, 1 Single, 2 XYZ, 3 FixedZ (cluster/mod.rs:107-139) */
    uint32_t dims[3];            /* XYZ */
    uint32_t total, z_slices;    /* FixedZ */
    float    first_slice_depth;  /* ClusterZConfig */
    uint32_t far_z_mode;         /* 0 MaxClusterableObjectRange, 1 Constant */
    float    far_z_constant;
    uint32_t dynamic_resizing;
    uint32_t screen_w, screen_h; /* Camera::physical_viewport_size */
    uint32_t view_cluster_bindings_max_indices;
} b200vis_cluster_config;
typedef struct b200vis_cluster_feedback {    /* Clusters::last_frame_* (cluster/mod.rs:155-161) */
    uint32_t has_farthest_z;     float farthest_z;
    uint32_t has_index_count;    uint32_t index_count;
} b200vis_cluster_feedback;

/* ---- lifetime ------------------------------------------------------------- */
B200VIS_API int32_t b200vis_abi_version(void);
/* Kernel launches this library has issued since it was loaded (all contexts); bench.py reports the difference over its
 * timed regions as `gpu_launches`. */
B200VIS_API uint64_t b200vis_kernel_launch_count(void);
/* sizeof of the ABI structs, in declaration order (config, view, cluster_view, frame_stats, cluster_config,
 * cluster_feedback): lets a foreign-language binding verify its layout at start-up. */
B200VIS_API void b200vis_struct_sizes(uint32_t out[6]);
B200VIS_API int32_t b200vis_create(const b200vis_config *cfg, b200vis_ctx **out);
B200VIS_API void b200vis_destroy(b200vis_ctx *ctx);
B200VIS_API const char *b200vis_last_error(const b200vis_ctx *ctx); /* valid until the next call on ctx; ctx may be NULL */
/* All uploads, kernels and downloads of this context are issued on `cuda_stream`
 * (a cudaStream_t; NULL => the context's own stream). */
B200VIS_API int32_t b200vis_set_stream(b200vis_ctx *ctx, void *cuda_stream);
B200VIS_API int32_t b200vis_synchronize(b200vis_ctx *ctx);
/* b200vis_run(B200VIS_STAGE_ALL) pipelines frames: the latency-bound tail of frame f (visible-list expansion,
 * cluster kernels) runs on an internal side stream and overlaps frame f+1's tile pass.  b200vis_join makes the
 * context's stream wait (asynchronously) for that tail, e.g. before recording a timing event; every download and
 * b200vis_synchronize join implicitly.  Set B200VIS_PIPELINE=0 to serialise everything on one stream. */
B200VIS_API int32_t b200vis_join(b200vis_ctx *ctx);
/* Multi-GPU: b200vis_run(PROPAGATE|CULL|CLUSTER_ASSIGN) leaves the frame's tail open on this stream; the host issues
 * its all-gather of the cluster slabs ON THIS STREAM (so it is ordered after CLUSTER_ASSIGN) and then calls
 * b200vis_run(CLUSTER_LISTS), which continues there.  Equals the context's stream when pipelining is off. */
B200VIS_API int32_t b200vis_tail_stream(b200vis_ctx *ctx, void **cuda_stream);

/* ---- mirroring the ECS columns --------------------------------------------- */
/* Hierarchy + identity; call on spawn/despawn/Changed<ChildOf> only.
 * Replaces the Children/ChildOf walks of propagate_descendants_unchecked
 * (systems.rs:679-748) with a cached execution plan.  entity_bits = Entity::to_bits()
 * (crates/bevy_ecs/src/entity/mod.rs:468-476), which fixes the order of every
 * visible list (visibility/mod.rs:870-874).  Rows must be in topological order
 * (parent_row[r] < r); b200vis_plan_row_order produces such an order. */
B200VIS_API int32_t b200vis_set_topology(b200vis_ctx *ctx, uint32_t n_rows, const uint32_t *parent_row,
                             const uint64_t *entity_bits);
/* Helper for the shim: a permutation (new_row -> old_row) that is topological and
 * keeps every tree contiguous in BFS order (the layout the tile kernel likes). */
B200VIS_API int32_t b200vis_plan_row_order(uint32_t n_rows, const uint32_t *parent_row, uint32_t *new_to_old);
/* What b200vis_set_topology would plan for this hierarchy (no GPU needed): out = { tiles, passes (kernel launches per
 * propagate), deepest in-tile level count, rows whose parent lives in another tile }.  Same error codes. */
B200VIS_API int32_t b200vis_host_plan_summary(uint32_t n_rows, const uint32_t *parent_row, uint32_t out[4]);
/* The plan as the default tile kernel (one CTA of 8 warps per tile) sees it (no GPU needed; for tests and tools):
 * tile_desc[i] = { first row, rows, in-tile levels, warp_sync_mask (bit l: every edge into level l stays inside a warp),
 * top_levels, lvl_warps low word, lvl_warps high word (nibble l = warps that meet at the hand-over of level l; 0 = the
 * tile is walked with CTA-wide barriers), pass }, topo[row] = parent's local row | in-tile depth << 9 | flags (bits 28-31).
 * With tile_desc == NULL only *n_tiles is written. */
B200VIS_API int32_t b200vis_host_tile_plan(uint32_t n_rows, const uint32_t *parent_row, uint32_t tile_rows, uint32_t tiles_capacity,
                                           uint32_t *n_tiles, uint32_t *tile_desc, uint32_t *topo);
/* The plan as the warp-per-tile kernel (B200VIS_TILE_KERNEL=warp) sees it (no GPU needed; for tests and tools): one work item per WARP.
 * tile_desc[i] = { first row, rows, chunks | contiguous-chunk bits << 8, pass }, nonroot[i][8] = per chunk the schedule
 * slots holding a row whose parent is in the tile, sched[i][256] = schedule slot -> local row (0xFF = padding, except in
 * a 256-row tile), wtopo[row] = depth | own slot << 8 | parent's slot << 15 | has-slot << 22 | flags (bits 28-31).
 * tile_rows = 0 means the default tile size (256).  With tile_desc == NULL only *n_tiles is written. */
B200VIS_API int32_t b200vis_host_warp_plan(uint32_t n_rows, const uint32_t *parent_row, uint32_t tile_rows, uint32_t tiles_capacity,
                                           uint32_t *n_tiles, uint32_t *tile_desc, uint32_t *nonroot, uint8_t *sched, uint32_t *wtopo);

/* Transform column, dirty ranges: trs[count][10] = translation.xyz, rotation.xyzw, scale.xyz
 * (components/transform.rs:86-105).  Marks the rows Changed<Transform>. */
B200VIS_API int32_t b200vis_upload_transforms(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const float *trs);
/* Same, for the scattered row set a `Changed<Transform>` query yields: rows[count], trs[count][10]. */
B200VIS_API int32_t b200vis_upload_transforms_scattered(b200vis_ctx *ctx, uint32_t count, const uint32_t *rows,
                                                        const float *trs);
/* Rows that are Changed<ChildOf> | Added<GlobalTransform> | freshly orphaned without new Transform data
 * (mark_dirty_trees' input set, systems.rs:112-113). */
B200VIS_API int32_t b200vis_mark_transforms_changed(b200vis_ctx *ctx, uint32_t first_row, uint32_t count);
/* GlobalTransform column as it stands on the host (initial mirror / external writes):
 * gt[count][12] = Affine3A x_axis.xyz, y_axis.xyz, z_axis.xyz, translation.xyz */
B200VIS_API int32_t b200vis_upload_global_transforms(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const float *gt);
/* Aabb / Sphere / flags / VisibilityClass / RenderLayers / VisibleEntityRanges columns:
 * bounds[count][6] = center.xyz, half_extents.xyz (Aabb) or center.xyz, radius,0,0 (Sphere);
 * class_mask: one bit per VisibilityClass the entity is in (0 => set_visible() but no list entry,
 * visibility/mod.rs:846-857); layer_mask / range_mask may be NULL (=> default layer / no
 * VisibleEntityRanges resource). */
B200VIS_API int32_t b200vis_upload_bounds(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const float *bounds,
                              const uint8_t *flags, const uint8_t *class_mask, const uint64_t *layer_mask,
                              const uint32_t *range_mask);
/* ViewVisibility column (bit0 current, bit1 previous; visibility/mod.rs:226-242) */
/* RenderLayers beyond the first 64 layers: the component is a SmallVec of 64-bit blocks (render_layers.rs:20-23) and
 * intersects() ORs the block-wise ANDs (:121-135).  Block 0 is the layer_mask of b200vis_upload_bounds / b200vis_view;
 * blocks[count][3] / blocks[3] are blocks 1..3 (layers 64..255) of the rows / of a view.  Lights keep to block 0
 * (b200vis_set_lights, shadow items). */
B200VIS_API int32_t b200vis_upload_render_layers_ext(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const uint64_t *blocks);
B200VIS_API int32_t b200vis_set_view_render_layers_ext(b200vis_ctx *ctx, uint32_t view, const uint64_t blocks[3]);
B200VIS_API int32_t b200vis_upload_view_visibility(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const uint8_t *vv);

/* StaticTransformOptimizations resource (systems.rs:87-103); default Enabled (1). */
B200VIS_API int32_t b200vis_set_static_transform_optimizations(b200vis_ctx *ctx, int32_t enabled);

/* ---- per-frame constants ----------------------------------------------------- */
B200VIS_API int32_t b200vis_set_views(b200vis_ctx *ctx, uint32_t n_views, const b200vis_view *views);
/* PointLight set (point_lights_query, assign.rs:146-153): light_row = the light entity's row (its
 * GlobalTransform translation and ViewVisibility are read on the device), in query order. */
B200VIS_API int32_t b200vis_set_lights(b200vis_ctx *ctx, uint32_t n_lights, const uint32_t *light_row, const float *range,
                           const uint64_t *layer_mask /* nullable */);
/* The other objects assign_objects_to_clusters gathers (assign.rs:231-295), in its push order after the point lights: rect
 * lights, then light probes (reflection probes and irradiance volumes interleaved in query order), then clustered decals.
 * Each is clustered with the point-light walk (assign.rs:740-800) on a sphere centred at its GlobalTransform translation;
 * only objects whose ViewVisibility is set this frame take part.  Radius per kind: rect light = range[j] (RectLight::range),
 * probe = GlobalTransform::radius_vec3a(Vec3A::ONE), decal = GlobalTransform::scale().length() -- the last two are
 * computed on the device from this frame's GlobalTransform (global_transform.rs:240-254).  Rect lights carry their own
 * RenderLayers (layer_mask[j], first block; NULL = default layer); probes and decals the default layer.
 *   Object j gets cluster ordinal n_lights + j (n_lights = the current b200vis_set_lights count): that is what
 *   b200vis_download_clusters, b200vis_download_frame, the result sink and the bindings index map see, and b200vis_set_lights
 *   shifts the ordinals of the objects when its count changes.  n_lights + n must be <= max_lights (B200VIS_ERR_CAPACITY).
 *   kind[j] must be grouped in push order: 2 < {3, 4} < 5 (INVALID_ARG otherwise, as for a kind outside 2..5 or a row >=
 *   max_entities); kind 1 (spot light) is B200VIS_ERR_UNSUPPORTED.  n = 0 removes the objects.
 *   Refused: world_size > 1 (UNSUPPORTED: rank-major ordinals would break the grouping by kind), and UNIFORM cluster
 *   bindings (INVALID_ARG, both ways round: the reference clusters none of these kinds without storage buffers).
 * b200vis_set_shadow_lights ordinals still address the point lights only. */
#define B200VIS_CLUSTERABLE_RECT_LIGHT        2u   /* = ClusterableObjectType::ordering().0 (assign.rs:115-131) */
#define B200VIS_CLUSTERABLE_REFLECTION_PROBE  3u
#define B200VIS_CLUSTERABLE_IRRADIANCE_VOLUME 4u
#define B200VIS_CLUSTERABLE_DECAL             5u   /* 1 (spot light) is reserved: B200VIS_ERR_UNSUPPORTED */
B200VIS_API int32_t b200vis_set_clusterable_objects(b200vis_ctx *ctx, uint32_t n, const uint32_t *kind, const uint32_t *row,
                                                    const float *range /* rect lights; ignored otherwise; nullable if none */,
                                                    const uint64_t *layer_mask /* rect lights; nullable => 1 */);
B200VIS_API int32_t b200vis_set_cluster_view(b200vis_ctx *ctx, uint32_t view, const b200vis_cluster_view *params);
/* Cluster grid dimensions of the view as last set (b200vis_set_cluster_view / b200vis_update_camera / b200vis_step);
 * zeros when clustering is off for the view.  The shim sizes Clusters::clusterable_objects from it. */
B200VIS_API int32_t b200vis_cluster_view_dims(const b200vis_ctx *ctx, uint32_t view, uint32_t dims[3]);

/* Frame constants kept in HBM: record_frame_constants snapshots the current views / cluster views (device copy
 * of the packed tables + the host copy the kernel parameters are built from) and returns a slot;
 * use_recorded_frame_constants(slot) makes b200vis_run use that snapshot with no host maths and no upload
 * (-1 returns to the live path).  Lets a recorded frame sequence replay with every input resident. */
B200VIS_API int32_t b200vis_record_frame_constants(b200vis_ctx *ctx, uint32_t *slot);
B200VIS_API int32_t b200vis_use_recorded_frame_constants(b200vis_ctx *ctx, int32_t slot);

/* Optional per-stage device timing: when on, b200vis_run brackets its stages with CUDA events on the
 * context's stream (up to 256 runs are kept).  b200vis_collect_stage_times_ms synchronizes ONCE, returns the
 * summed durations of the tile kernel(s) (propagate+cull), the visible-list expansion and the cluster kernels
 * over the `frames` runs recorded since the last collect, and resets the recorder. */
B200VIS_API int32_t b200vis_set_profiling(b200vis_ctx *ctx, int32_t enabled);
B200VIS_API int32_t b200vis_collect_stage_times_ms(b200vis_ctx *ctx, float *tile_ms, float *expand_ms, float *cluster_ms,
                                                   uint32_t *frames);

/* One call per camera per frame: the host-side work of update_frusta (visibility/mod.rs:627-636) and of the
 * per-view prologue of assign_objects_to_clusters (assign.rs:324-485) for a perspective camera, written
 * straight into the context's frame constants.  cfg == NULL leaves the view without clusters; `out` (nullable)
 * receives the cluster view that was set (its plane pointers are only valid until the next call). */
typedef struct b200vis_camera {
    float    global_transform[12]; /* camera GlobalTransform, layout as in b200vis_upload_global_transforms */
    float    fov_y, aspect, near_z, far_z; /* PerspectiveProjection (projection.rs:419-426) */
    uint64_t layer_mask;
    uint8_t  flags;                /* B200VIS_VIEW_* */
    int8_t   range_view_index;
    uint8_t  pad[6];
} b200vis_camera;
B200VIS_API int32_t b200vis_set_view_count(b200vis_ctx *ctx, uint32_t n_views);
B200VIS_API int32_t b200vis_update_camera(b200vis_ctx *ctx, uint32_t view, const b200vis_camera *camera,
                                          const b200vis_cluster_config *cfg, const b200vis_cluster_feedback *feedback,
                                          b200vis_cluster_view *out);

/* ---- run ----------------------------------------------------------------------- */
B200VIS_API int32_t b200vis_run(b200vis_ctx *ctx, uint32_t stages);

/* One call per frame for a single-GPU host loop: upload the changed Transforms, recompute every camera's frame
 * constants (b200vis_update_camera with the library's own copy of last frame's Clusters feedback), run all stages
 * and -- with B200VIS_STEP_WAIT -- synchronise and refresh that feedback from the frame's statistics.  With a result
 * sink set, the frame's results are in the caller's pinned buffers when the call returns. */
#define B200VIS_STEP_WAIT 0x1u
B200VIS_API int32_t b200vis_step(b200vis_ctx *ctx, uint32_t n_changed, const uint32_t *rows, const float *trs,
                                 uint32_t n_cameras, const b200vis_camera *cameras, const b200vis_cluster_config *cfg,
                                 uint32_t flags);

/* ---- results --------------------------------------------------------------------- */
B200VIS_API int32_t b200vis_download_frame_stats(b200vis_ctx *ctx, b200vis_frame_stats *out);
/* gt[count][stride_floats] (stride 12, or 16 for glam's padded Affine3A layout); changed[count]:
 * 1 where the shim must stamp changed_ticks (set_if_neq semantics, systems.rs:719). Either may be NULL. */
B200VIS_API int32_t b200vis_download_global_transforms(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, float *gt,
                                           uint32_t stride_floats, uint8_t *changed);
B200VIS_API int32_t b200vis_download_view_visibility(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, uint8_t *vv,
                                         uint8_t *changed);
/* VisibleEntities of one view: rows of the visible entities that have a VisibilityClass, ascending by
 * Entity::to_bits() (visibility/mod.rs:861-874).  An inactive view keeps last frame's list (:780-782). */
B200VIS_API int32_t b200vis_download_visible(b200vis_ctx *ctx, uint32_t view, uint32_t *rows, uint32_t capacity,
                                 uint32_t *count);
/* VisibleEntities::entities is one sorted Vec per VisibilityClass, and an entity with k classes is pushed k times
 * (visibility/mod.rs:344-347, 852-857).  classes[i] = the class mask (as uploaded by b200vis_upload_bounds, bit k = class k
 * of the shim's TypeId registry, at most 8) of the i-th row of b200vis_download_visible's list: walking the list once and
 * pushing entity i into every class list whose bit is set yields each class's list already sorted. */
B200VIS_API int32_t b200vis_download_visible_classes(b200vis_ctx *ctx, uint32_t view, uint8_t *classes, uint32_t capacity,
                                                     uint32_t *count);
/* Clusters of one view in CSR form: offsets[n_clusters+1], light ordinals (index into the
 * b200vis_set_lights arrays, then the b200vis_set_clusterable_objects objects; with world_size>1: global ordinal = rank-major) in the reference's
 * push order, cluster index = (y*dims.x + x)*dims.z + z (assign.rs:676-678). */
B200VIS_API int32_t b200vis_download_clusters(b200vis_ctx *ctx, uint32_t view, uint32_t *offsets, uint32_t *indices,
                                  uint32_t indices_capacity, uint32_t *total);

/* Everything the shim writes back after a frame, with two stream synchronisations instead of one per list:
 * the stats block, every view's sorted visible rows (visible_rows[v*visible_capacity ...]) and every view's
 * cluster CSR (cluster_offsets[v*4097 ...], cluster_indices[v*cluster_capacity ...]).  Array pointers may be NULL. */
B200VIS_API int32_t b200vis_download_frame(b200vis_ctx *ctx, b200vis_frame_stats *stats, uint32_t *visible_rows,
                                           uint32_t visible_capacity, uint32_t *cluster_offsets,
                                           uint32_t *cluster_indices, uint32_t cluster_capacity);

/* Result sink: caller-owned PINNED host memory that the frame's results are written into by the GPU itself (small
 * "publish" kernels doing coalesced posted writes over PCIe right after the producing kernels), so that reading a
 * frame back needs ONE stream synchronisation and no size round trip:
 *   stats            the b200vis_frame_stats block
 *   visible_rows     [max_views][visible_capacity]  sorted visible rows per view (count in stats->visible_count)
 *   cluster_offsets  [max_views][4097], cluster_indices [max_views][cluster_capacity]
 * The library registers the ranges with cudaHostRegister if they are not already pinned.  NULL removes the sink. */
typedef struct b200vis_result_sink {
    b200vis_frame_stats *stats;
    uint32_t *visible_rows;   uint32_t visible_capacity;
    uint8_t  *visible_classes; /* nullable: [max_views][visible_capacity] VisibilityClass mask of each listed row */
    uint32_t *cluster_offsets;
    uint32_t *cluster_indices; uint32_t cluster_capacity;
} b200vis_result_sink;
B200VIS_API int32_t b200vis_set_result_sink(b200vis_ctx *ctx, const b200vis_result_sink *sink);

/* ---- write-back of the frame's column results into the caller's ECS columns -------------------------------------------
 * The reference systems leave their results IN the ECS: GlobalTransform (+ Changed<GlobalTransform>) and ViewVisibility
 * (+ Changed<ViewVisibility>) are read downstream (e.g. crates/bevy_pbr/src/render/mesh.rs:1933-1955).  With column sinks
 * registered, b200vis_writeback_columns (or b200vis_step with B200VIS_STEP_WRITEBACK) has the GPU write, over PCIe and
 * straight into host memory -- typically the table column slices `ContiguousMut::bypass_change_detection()` hands out
 * (crates/bevy_ecs/src/change_detection/params.rs:1079-1142):
 *   global_transforms [n][gt_stride_floats]  ONLY the rows whose GlobalTransform changed this frame (set_if_neq semantics:
 *                                            the other rows keep their bytes); stride 16 = glam Affine3A (four 16-byte
 *                                            Vec3A lanes, padding lanes written as 0), stride 12 = packed X,Y,Z,T
 *   gt_changed_bits   [ceil(n/32)]           bit r%32 of word r/32: stamp changed_ticks[r] = this_run
 *   view_visibility   [n]                    the ViewVisibility byte of every row (bit0 current, bit1 previous)
 *   vv_changed_bits   [ceil(n/32)]           Changed<ViewVisibility>
 * Any pointer may be NULL (that column is not delivered).  The memory is registered with cudaHostRegister if it is not
 * pinned already.  Results are complete after b200vis_synchronize (or b200vis_step(.., WAIT)).  NULL removes the sinks. */
typedef struct b200vis_column_sinks {
    float *global_transforms; uint32_t gt_stride_floats;
    uint32_t *gt_changed_bits;
    uint8_t *view_visibility;
    uint32_t *vv_changed_bits;
} b200vis_column_sinks;
B200VIS_API int32_t b200vis_set_column_sinks(b200vis_ctx *ctx, const b200vis_column_sinks *sinks);
B200VIS_API int32_t b200vis_writeback_columns(b200vis_ctx *ctx);
/* The same for a subset of the columns: a shim that runs the stages from separate systems writes the GlobalTransform
 * column back right after PROPAGATE and the ViewVisibility column after CULL (and the light-visibility systems). */
#define B200VIS_WB_GLOBAL_TRANSFORM 0x1u
#define B200VIS_WB_VIEW_VISIBILITY  0x2u
B200VIS_API int32_t b200vis_writeback_columns_ex(b200vis_ctx *ctx, uint32_t which);
#define B200VIS_STEP_WRITEBACK 0x2u  /* b200vis_step: enqueue the column write-back right behind the tile pass */

/* ---- SURVEY.md 8(f) N1: the render world's visible-entity diff ---------------------------------------------
 * RenderVisibleEntitiesClass::update_cpu_culled_entities (crates/bevy_render/src/view/visibility/mod.rs:194-249)
 * marches over last frame's and this frame's sorted list to find the newly added and newly removed entities.  With
 * the diff enabled the CULL stage produces both lists on the device (set algebra on the rank-ordered bit sets, ordered
 * emit), so the shim can feed `added_entities` / `removed_entities` directly and skip the download of the full lists.
 * Rows ascend by Entity::to_bits() like the lists themselves.  "Last frame" = the last frame the view was active; an
 * inactive view reports nothing.  Enabling the diff and b200vis_set_topology (row identities change) reset the old
 * list to empty: the next frame reports every visible row as added, and the shim drops its render-world list. */
B200VIS_API int32_t b200vis_enable_visible_diff(b200vis_ctx *ctx, int32_t enabled);
B200VIS_API int32_t b200vis_download_visible_diff(b200vis_ctx *ctx, uint32_t view, uint32_t *added_rows, uint32_t added_capacity,
                                                  uint32_t *n_added, uint32_t *removed_rows, uint32_t removed_capacity,
                                                  uint32_t *n_removed);
/* Sink form (pinned host memory written by the GPU right after the CULL stage, like b200vis_set_result_sink):
 * rows[2][max_views][capacity] (0 = added, 1 = removed), counts[max_views][2]; a list longer than `capacity` is
 * truncated (the count still says how long it was).  A result sink whose visible_rows is NULL then keeps the full
 * lists on the device.  NULL, 0, NULL removes the sink. */
B200VIS_API int32_t b200vis_set_visible_diff_sink(b200vis_ctx *ctx, uint32_t *rows, uint32_t capacity, uint32_t *counts);

/* ---- SURVEY.md 8(f) N3: shadow-view culling of point lights -------------------------------------------------------
 * check_point_light_mesh_visibility (crates/bevy_light/src/lib.rs:517-668): for every point light that is in some
 * view's VisibleEntities and has shadow maps enabled, every shadow-casting mesh is tested against the light's range
 * sphere (Sphere::intersects_obb, bevy_camera/src/primitives.rs:219-226) and the six CubemapFrusta
 * (Frustum::intersects_obb with near and far planes, :272-294); survivors are set_visible() and land in the light's
 * six sorted CubemapVisibleEntities lists.
 *   caster[count]   1 = the row is in visible_entity_query (Mesh3d, no NotShadowCaster, no DirectionalLight);
 *                   NoCpuCulling, InheritedVisibility, RenderLayers, Aabb, NoFrustumCulling, VisibilityRange come from
 *                   the columns already resident
 *   shadow lights   ordinals into the b200vis_set_lights arrays (the lights with shadow_maps_enabled), their
 *                   CubemapFrusta frusta[n][6 faces][6 half spaces][4] (update_point_light_frusta,
 *                   bevy_light/src/point_light.rs:212-265; b200vis_host_point_light_frusta computes them for hosts
 *                   without glam), RenderLayers (NULL = default), and the bit of get_shadow_lod_origin's view in the
 *                   VisibleEntityRanges masks (-1 = none).  Whether a light is in some view's VisibleEntities is
 *                   decided on the device from the per-view sets of the visible-diff bookkeeping (which
 *                   b200vis_upload_shadow_casters switches on: call it before the frame's CULL stage); the light's
 *                   sphere is its row's GlobalTransform translation and its range.
 *   b200vis_run_shadow_culling  after b200vis_run(.. CULL ..) of the same frame; also folds set_visible() into the
 *                   ViewVisibility column / change flags (download them afterwards).
 *   lists           rows ascending by Entity::to_bits() (sort_unstable, lib.rs:650-661); list_capacity rows per list
 *                   are kept (0 = max_entities). */
B200VIS_API int32_t b200vis_upload_shadow_casters(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const uint8_t *caster);
B200VIS_API int32_t b200vis_set_shadow_lights(b200vis_ctx *ctx, uint32_t n_lights, const uint32_t *light_ordinals, const float *frusta,
                                              const uint64_t *layer_mask, int32_t lod_origin_range_index, uint32_t list_capacity);
/* The general form: point lights, SPOT lights (the second half of check_point_light_mesh_visibility, lib.rs:670-749: one
 * Frustum, near and far planes tested, the same range-sphere pre-test) and DIRECTIONAL-light cascades
 * (check_dir_light_mesh_visibility, lib.rs:342-510: one item per (light, view, cascade) with that cascade's Frustum; the near
 * plane is not tested, :455-458; there is no range sphere; the caller lists only lights with shadow_maps_enabled that are
 * visible, :395-399).  A point / spot item names the light's ROW (spot lights are not clustered, so they have no ordinal);
 * it takes part only while that row is in some view's VisibleEntities.  range_view_index = the bit of the
 * VisibleEntityRanges masks that gates rows with a VisibilityRange: the shadow LOD origin's for point / spot lights, the
 * cascade's own view for directional lights; -1 = that view is not in the map (ranged rows are then skipped).
 * Lists: b200vis_download_shadow_visible(item, face) with face 0 for spot lights and cascades. */
#define B200VIS_SHADOW_POINT 0u
#define B200VIS_SHADOW_SPOT 1u
#define B200VIS_SHADOW_DIRECTIONAL_CASCADE 2u
typedef struct b200vis_shadow_item {
    uint32_t kind;
    uint32_t light_row;          /* point / spot */
    float    range;              /* point / spot: PointLight::range / SpotLight::range */
    int32_t  range_view_index;
    uint64_t layer_mask;         /* the light's RenderLayers (first block; default layer = 1) */
    float    frusta[6][6][4];    /* point: the six CubemapFrusta faces; spot / cascade: frusta[0] */
} b200vis_shadow_item;
B200VIS_API int32_t b200vis_set_shadow_items(b200vis_ctx *ctx, uint32_t n_items, const b200vis_shadow_item *items, uint32_t list_capacity);
B200VIS_API int32_t b200vis_run_shadow_culling(b200vis_ctx *ctx);
B200VIS_API int32_t b200vis_download_shadow_visible(b200vis_ctx *ctx, uint32_t shadow_light, uint32_t face, uint32_t *rows,
                                                    uint32_t capacity, uint32_t *count);
/* update_point_light_frusta for one light (no GPU needed): light_gt12 as in upload_global_transforms */
B200VIS_API void b200vis_host_point_light_frusta(const float *light_gt12, float range, float shadow_map_near_z, float frusta[6][6][4]);

/* ---- SURVEY.md 8(f) N4: the two per-entity passes that feed the cull kernel's flag byte ---------------------------
 * (a) check_visibility_ranges (crates/bevy_camera/src/visibility/range.rs:230-284).  With the VisibilityRange columns
 *     resident -- start_end[count][2] = (start_margin.start, end_margin.end), the two values is_visible_at_all reads
 *     (range.rs:157-159), and use_aabb[count] -- the cull phase evaluates the distance test itself on this frame's
 *     GlobalTransform instead of taking an uploaded range_mask, and keeps the masks for download
 *     (VisibleEntityRanges::entities; 0 = no entry).  Range views: the translations of the views the system indexes, in
 *     its view-query order (only the first 32 count, :247); b200vis_view.range_view_index maps a culled view to its bit. */
B200VIS_API int32_t b200vis_upload_visibility_ranges(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const float *start_end,
                                                     const uint8_t *use_aabb);
B200VIS_API int32_t b200vis_set_visibility_range_views(b200vis_ctx *ctx, uint32_t n_views, const float *positions /* [n][3] */);
B200VIS_API int32_t b200vis_download_visibility_ranges(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, uint32_t *mask);
/* (b) visibility_propagate_system (crates/bevy_camera/src/visibility/mod.rs:638-729).  visibility[count]: 0 Inherited,
 *     1 Hidden, 2 Visible (the enum's order, :83-96), | 4 when the entity lacks Visibility / InheritedVisibility.
 *     b200vis_propagate_visibility walks the same level-ordered tiles as the transform propagation and leaves every
 *     InheritedVisibility (bit 0 of the flags column the cull phase reads) at the value the reference's change-driven
 *     system converges to; a parent that is a root's absence, lacks the components, or is B200VIS_DETACHED counts as
 *     visible (:655-659).  changed[i] = 1 where the value was rewritten (set-if-different, :667), i.e. where the shim
 *     stamps InheritedVisibility's change tick. */
#define B200VIS_VISIBILITY_INHERITED 0u
#define B200VIS_VISIBILITY_HIDDEN 1u
#define B200VIS_VISIBILITY_VISIBLE 2u
#define B200VIS_VISIBILITY_NO_COMPONENTS 4u
B200VIS_API int32_t b200vis_upload_visibility(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, const uint8_t *visibility);
B200VIS_API int32_t b200vis_propagate_visibility(b200vis_ctx *ctx);
B200VIS_API int32_t b200vis_download_inherited_visibility(b200vis_ctx *ctx, uint32_t first_row, uint32_t count, uint8_t *inherited,
                                                          uint8_t *changed);

/* ---- SURVEY.md 8(f) N2: Clusters -> ViewClusterBindings ----------------------------------------------------------
 * extract_clusters_for_cpu_clustering + prepare_clusters_for_cpu_clustering (crates/bevy_pbr/src/cluster/mod.rs:394-582)
 * flatten each view's per-cluster Vec<Entity> into the two GPU buffers of ViewClusterBindings (:584-800).  With a mode
 * set, the CLUSTER_LISTS stage emits that wire format directly from the device CSR:
 *   STORAGE  offsets_and_counts[n_clusters][8] = (offset, point_lights, spot, rect | probes, volumes, decals, 0);
 *            index_lists[n_indices] u32
 *   UNIFORM  offsets_and_counts[4096] = pack_offset_and_counts (:855-859); index_lists[4096] = 16384 8-bit slots,
 *            truncated at ViewClusterBindings::MAX_INDICES exactly like the reference's record loop (:505-514)
 * gpu_index_of_light[n_map] = GlobalClusterableObjectMeta::entity_to_index for each light ordinal (NULL = the ordinal
 * itself); ordinals without an entry get the dummy index !0 (:703-705).
 * With clusterable objects set (STORAGE only), each cluster's counts are split by kind (ObjectsInClusterCpu::add_*,
 * bevy_light/src/cluster/mod.rs:478-512).  Two limits of the bindings, not of Clusters: the index map is one per ordinal and
 * shared by all views (the render world's per-view probe indices are not modelled), and an entity that is both an
 * EnvironmentMapLight probe and an IrradianceVolume is one ordinal here where extract_clusters emits two records
 * (bevy_pbr/src/cluster/mod.rs:454-463). */
#define B200VIS_BINDINGS_OFF 0u
#define B200VIS_BINDINGS_STORAGE 1u
#define B200VIS_BINDINGS_UNIFORM 2u
B200VIS_API int32_t b200vis_set_cluster_bindings(b200vis_ctx *ctx, uint32_t mode, const uint32_t *gpu_index_of_light, uint32_t n_map);
/* capacities in 32-bit words; n_offsets / n_indices = ViewClusterBindings::n_offsets / n_indices */
B200VIS_API int32_t b200vis_download_cluster_bindings(b200vis_ctx *ctx, uint32_t view, uint32_t *offsets_and_counts, uint32_t oc_capacity,
                                                      uint32_t *index_lists, uint32_t il_capacity, uint32_t *n_offsets,
                                                      uint32_t *n_indices);

/* ---- multi-GPU cluster exchange (one all-gather per frame, done by the host's collective) ------- */
/* Each rank fills `slab_bytes` at `send`; after all-gathering the slabs rank-major into `recv`
 * (world_size * slab_bytes) the LISTS stage reads `recv`.  Buffers are caller-allocated device memory
 * (e.g. torch tensors); with world_size <= 1 the library uses its own buffer and no exchange. */
/* Built-in exchange: the library dlopen()s libnccl.so.2 (the copy the host process already loaded, e.g. torch's), rank 0
 * makes a unique id, the host broadcasts those 128 bytes by any means, every rank calls b200vis_comm_init (a collective),
 * and from then on b200vis_run(B200VIS_STAGE_ALL) issues the ncclAllGather of the slabs itself, on the frame's tail
 * stream, between CLUSTER_ASSIGN and CLUSTER_LISTS -- one call per frame, pipelined like the single-GPU path. */
#define B200VIS_COMM_ID_BYTES 128
B200VIS_API int32_t b200vis_comm_unique_id(uint8_t id[B200VIS_COMM_ID_BYTES]);
B200VIS_API int32_t b200vis_comm_init(b200vis_ctx *ctx, const uint8_t id[B200VIS_COMM_ID_BYTES]);
/* Peer-memory exchange (the default in bench.py): no collective call at all.  Every rank exports the CUDA IPC handle of its
 * gathered buffer, the host all-gathers the 64-byte handles (rank-major) by any means, every rank imports them; from then on
 * b200vis_run(B200VIS_STAGE_ALL) has the rank WRITE its slab into every rank's buffer with plain NVLink stores right after
 * CLUSTER_ASSIGN and publish a per-frame stamp (release, system scope); CLUSTER_LISTS spins on all ranks' stamps (acquire)
 * before reading.  world_size 2..8, all ranks on one node with peer access.  A rank that never arrives is reported as
 * cluster_index_overflow[v] == 2 after a few seconds instead of hanging the GPU. */
#define B200VIS_P2P_HANDLE_BYTES 64
B200VIS_API int32_t b200vis_p2p_export(b200vis_ctx *ctx, uint8_t handle[B200VIS_P2P_HANDLE_BYTES]);
B200VIS_API int32_t b200vis_p2p_import(b200vis_ctx *ctx, const uint8_t *handles /* [world_size][64], rank-major */);
/* One process, several GPUs (a Bevy App is one process): link the contexts of the process directly -- plain peer access, no
 * IPC handles, no collective library.  ctxs[r]: created with world_size = n, rank = r, one device each.  Then one host thread
 * calls b200vis_run(ctxs[r], B200VIS_STAGE_ALL) for every r per frame; the slab exchange happens on the devices. */
B200VIS_API int32_t b200vis_p2p_link(b200vis_ctx *const *ctxs, uint32_t n);
B200VIS_API int32_t b200vis_cluster_exchange_bytes(const b200vis_ctx *ctx, size_t *slab_bytes);
B200VIS_API int32_t b200vis_set_cluster_exchange_buffers(b200vis_ctx *ctx, void *send_device, void *recv_device);

/* ---- host-side mirror of the reference's per-view math (no GPU needed) --------------------------- */
/* PerspectiveProjection::get_clip_from_view (crates/bevy_camera/src/projection.rs:339-343) */
B200VIS_API void b200vis_host_perspective(float fov_y, float aspect, float near_z, float *clip_from_view16);
/* CameraProjection::compute_frustum (projection.rs:72-80): camera_gt[12] as in upload_global_transforms */
B200VIS_API void b200vis_host_compute_frustum(const float *clip_from_view16, const float *camera_gt12, float far_z,
                                  float half_spaces[6][4]);


/* The thresholds the device uses in place of view_z_to_z_slice (assign.rs:1046-1062): thresholds[k-1] is the smallest
 * u = -view_z whose slice index (computed with the HOST's libm, exactly the reference's float expression) is >= k;
 * slice(u) = number of thresholds <= u.  z_slices-1 values (NaN where the slice is never reached). */
B200VIS_API void b200vis_host_z_slice_thresholds(const float cluster_factors[2], uint32_t z_slices, uint32_t is_orthographic,
                                                 float *thresholds);
B200VIS_API void b200vis_host_default_cluster_config(b200vis_cluster_config *cfg, uint32_t screen_w, uint32_t screen_h);
/* The per-view prologue of assign_objects_to_clusters (assign.rs:324-485).  planes_scratch must hold
 * 3*4097*4 floats; out->x/y/z_planes point into it. */
B200VIS_API int32_t b200vis_host_cluster_view_setup(const b200vis_cluster_config *cfg, const float *camera_gt12,
                                        const float *clip_from_view16, const float frustum[6][4],
                                        uint64_t layer_mask, const b200vis_cluster_feedback *feedback,
                                        float *planes_scratch, b200vis_cluster_view *out);

#ifdef __cplusplus
}
#endif
#endif /* B200VIS_H */
