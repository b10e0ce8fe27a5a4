//! b200vis_plugin.rs — the Bevy-side shim for libb200vis (SOURCE ONLY: there is no Rust toolchain in the build image;
//! compile it in a crate that depends on bevy 0.20 and links `b200vis`).  `tests/host_shim.c` performs the same sequence
//! through the same C ABI in plain C and is run against the CPU oracle on the GPU box.
//!
//! The plugin removes three reference system sets from `PostUpdate` / `PostStartup` and adds replacements **with the same
//! query signatures, in the same sets**, that call the C ABI of `include/b200vis.h`:
//!   propagate  <- mark_dirty_trees / propagate_parent_transforms / sync_simple_transforms
//!                 (crates/bevy_transform/src/systems.rs:42, 111, 506; registered at plugins.rs:37-47)
//!   cull       <- check_visibility_cpu_culling (crates/bevy_camera/src/visibility/mod.rs:748)
//!   cluster    <- assign_objects_to_clusters   (crates/bevy_light/src/cluster/assign.rs:137; the only member of
//!                 SimulationLightSystems::AssignLightsToClusters, crates/bevy_light/src/lib.rs:187-191)
//! `reset_view_visibility` and `mark_newly_hidden_entities_invisible` are private and share their sets with systems that
//! must stay, so in an UNFORKED Bevy they keep running on the CPU: the cull system below turns the device's "visible in
//! >= 1 view" bit into `set_visible()` calls, which is also what keeps the light-visibility systems (they OR into the same
//! byte) composing correctly (SURVEY.md 8b).  With a three-line patch that makes those two systems removable, the device's
//! ViewVisibility bytes + change bits can be written straight into the column instead (`forked-bevy` feature below).
//!
//! Data flow (INTEGRATION.md section 2): ECS columns -> `upload_*` on change; results -> pinned host buffers the GPU
//! writes itself (`b200vis_set_result_sink`, `b200vis_set_column_sinks`), read after one `b200vis_synchronize` per system.
#![allow(non_camel_case_types, clippy::too_many_arguments, clippy::type_complexity)]
use bevy::camera::primitives::{Aabb, Frustum, Sphere};
use bevy::camera::visibility::*;
use bevy::ecs::entity::EntityHashMap;
use bevy::ecs::schedule::ScheduleCleanupPolicy::RemoveSystemsOnly;
use bevy::light::{cluster::*, EnvironmentMapLight, LightProbe, PointLight, RectLight, SimulationLightSystems};
use bevy::prelude::*;
use bevy::transform::{systems::*, TransformSystems};
use core::any::TypeId;
use core::ffi::c_char;

// ---- FFI (mirrors include/b200vis.h, ABI version 2) -----------------------------------------------------------------------
#[repr(C)] pub struct b200vis_ctx { _p: [u8; 0] }
#[repr(C)] pub struct b200vis_config { device: i32, max_entities: u32, max_lights: u32, max_views: u32, max_cluster_indices: u32,
                                        world_size: u32, rank: u32, reserved: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct b200vis_view { half_spaces: [[f32; 4]; 6], layer_mask: u64, flags: u8, range_view_index: i8, pad: [u8; 6] }
#[repr(C)] #[derive(Default)]
pub struct b200vis_frame_stats { visible_count: [u32; 8], cluster_index_count: [u32; 8], cluster_farthest_z: [f32; 8],
                                 cluster_index_overflow: [u32; 8], gt_changed_count: u32, vv_changed_count: u32, frame: u32, pad: u32 }
#[repr(C)] pub struct b200vis_cluster_view { enabled: u32, dims: [u32; 3], tile_size: [u32; 2], is_orthographic: u32, near_z: f32,
    far_z: f32, cluster_factors: [f32; 2], view_from_world: [f32; 16], clip_from_view: [f32; 16], view_from_world_scale: [f32; 3],
    view_from_world_scale_max: f32, frustum: [[f32; 4]; 6], layer_mask: u64, x_planes: *const f32, y_planes: *const f32,
    z_planes: *const f32 }
#[repr(C)] pub struct b200vis_cluster_config { kind: u32, dims: [u32; 3], total: u32, z_slices: u32, first_slice_depth: f32,
    far_z_mode: u32, far_z_constant: f32, dynamic_resizing: u32, screen_w: u32, screen_h: u32, view_cluster_bindings_max_indices: u32 }
#[repr(C)] #[derive(Default, Clone, Copy)]
pub struct b200vis_cluster_feedback { has_farthest_z: u32, farthest_z: f32, has_index_count: u32, index_count: u32 }
#[repr(C)] pub struct b200vis_result_sink { stats: *mut b200vis_frame_stats, visible_rows: *mut u32, visible_capacity: u32,
    visible_classes: *mut u8, cluster_offsets: *mut u32, cluster_indices: *mut u32, cluster_capacity: u32 }
#[repr(C)] pub struct b200vis_column_sinks { global_transforms: *mut f32, gt_stride_floats: u32, gt_changed_bits: *mut u32,
    view_visibility: *mut u8, vv_changed_bits: *mut u32 }

#[link(name = "b200vis")]
extern "C" {
    fn b200vis_create(cfg: *const b200vis_config, out: *mut *mut b200vis_ctx) -> i32;
    fn b200vis_destroy(ctx: *mut b200vis_ctx);
    fn b200vis_last_error(ctx: *const b200vis_ctx) -> *const c_char;
    fn b200vis_synchronize(ctx: *mut b200vis_ctx) -> i32;
    fn b200vis_set_topology(ctx: *mut b200vis_ctx, n: u32, parent_row: *const u32, entity_bits: *const u64) -> i32;
    fn b200vis_plan_row_order(n: u32, parent_row: *const u32, new_to_old: *mut u32) -> i32;
    fn b200vis_upload_transforms(ctx: *mut b200vis_ctx, first: u32, count: u32, trs: *const f32) -> i32;
    fn b200vis_upload_transforms_scattered(ctx: *mut b200vis_ctx, count: u32, rows: *const u32, trs: *const f32) -> i32;
    fn b200vis_upload_global_transforms(ctx: *mut b200vis_ctx, first: u32, count: u32, gt: *const f32) -> i32;
    fn b200vis_upload_bounds(ctx: *mut b200vis_ctx, first: u32, count: u32, bounds: *const f32, flags: *const u8, class_mask: *const u8,
                             layer_mask: *const u64, range_mask: *const u32) -> i32;
    fn b200vis_upload_view_visibility(ctx: *mut b200vis_ctx, first: u32, count: u32, vv: *const u8) -> i32;
    fn b200vis_set_static_transform_optimizations(ctx: *mut b200vis_ctx, enabled: i32) -> i32;
    fn b200vis_set_views(ctx: *mut b200vis_ctx, n: u32, views: *const b200vis_view) -> i32;
    fn b200vis_set_lights(ctx: *mut b200vis_ctx, n: u32, light_row: *const u32, range: *const f32, layers: *const u64) -> i32;
    fn b200vis_set_cluster_view(ctx: *mut b200vis_ctx, view: u32, p: *const b200vis_cluster_view) -> i32;
    fn b200vis_set_clusterable_objects(ctx: *mut b200vis_ctx, n: u32, kind: *const u32, row: *const u32, range: *const f32,
                                       layers: *const u64) -> i32;
    fn b200vis_host_cluster_view_setup(cfg: *const b200vis_cluster_config, camera_gt12: *const f32, clip_from_view16: *const f32,
                                       frustum: *const [f32; 4], layer_mask: u64, feedback: *const b200vis_cluster_feedback,
                                       planes_scratch: *mut f32, out: *mut b200vis_cluster_view) -> i32;
    fn b200vis_run(ctx: *mut b200vis_ctx, stages: u32) -> i32;
    fn b200vis_set_result_sink(ctx: *mut b200vis_ctx, sink: *const b200vis_result_sink) -> i32;
    fn b200vis_set_column_sinks(ctx: *mut b200vis_ctx, sinks: *const b200vis_column_sinks) -> i32;
    fn b200vis_writeback_columns_ex(ctx: *mut b200vis_ctx, which: u32) -> i32;
}
const NO_PARENT: u32 = 0xFFFF_FFFF; const DETACHED: u32 = 0xFFFF_FFFE;
const STAGE_PROPAGATE: u32 = 1; const STAGE_CULL: u32 = 2; const STAGE_CLUSTER: u32 = 12;
const WB_GLOBAL_TRANSFORM: u32 = 1; const WB_VIEW_VISIBILITY: u32 = 2;
const F_INHERITED: u8 = 0x01; const F_AABB: u8 = 0x02; const F_SPHERE: u8 = 0x04; const F_NO_FRUSTUM: u8 = 0x08;
const F_RANGE: u8 = 0x10; const F_SPHERE_FROM_GT: u8 = 0x40;
const VIEW_ACTIVE: u8 = 1; const VIEW_NO_CPU_CULLING: u8 = 2;
const ERR_HIERARCHY_CYCLE: i32 = 4;
// ClusterableObjectType::ordering().0 (assign.rs:115-131) = B200VIS_CLUSTERABLE_*
const KIND_RECT_LIGHT: u32 = 2; const KIND_REFLECTION_PROBE: u32 = 3; const KIND_IRRADIANCE_VOLUME: u32 = 4; const KIND_DECAL: u32 = 5;
const MAX_VIEWS: usize = 8; const MAX_CLUSTERS: usize = 4096;

/// Device context, the entity <-> row map, and the pinned host buffers the GPU writes into.  `Send + Sync`: exactly one
/// system touches it at a time (`ResMut`).  The result buffers are allocated once at full capacity and never reallocated:
/// the library registers them with cudaHostRegister and the GPU keeps their addresses.
#[derive(Resource)]
pub struct B200Vis {
    ctx: *mut b200vis_ctx,
    max_entities: usize,
    n: usize,
    row_of: EntityHashMap<u32>,
    entity_of: Vec<Entity>,
    columns_epoch: u64,           // bumped when rows are renumbered: every mirrored column must be uploaded again
    bounds_epoch: u64,
    lights_epoch: u64,
    classes: Vec<TypeId>,         // VisibilityClass registry: bit k of the class mask = classes[k] (at most 8)
    view_entities: Vec<Entity>,   // view v of the device = this camera entity (query order of the cull system)
    light_entities: Vec<Entity>,  // cluster ordinal -> entity: the point lights in query order, then the clusterable objects
    object_kinds: Vec<u32>,       // kind of ordinal light_entities.len() - object_kinds.len() + j
    // sinks
    stats: Box<b200vis_frame_stats>,
    gt_col: Vec<[f32; 16]>, gt_bits: Vec<u32>, vv_col: Vec<u8>, vv_bits: Vec<u32>,
    visible_rows: Vec<u32>, visible_classes: Vec<u8>, cluster_offsets: Vec<u32>, cluster_indices: Vec<u32>, cluster_cap: usize,
    planes_scratch: Vec<f32>,
}
unsafe impl Send for B200Vis {}
unsafe impl Sync for B200Vis {}
impl Drop for B200Vis { fn drop(&mut self) { unsafe { b200vis_destroy(self.ctx) } } }

impl B200Vis {
    fn check(&self, rc: i32) -> Result<(), BevyError> {
        if rc == 0 { return Ok(()); }
        let msg = unsafe { std::ffi::CStr::from_ptr(b200vis_last_error(self.ctx)) }.to_string_lossy().into_owned();
        // crates/bevy_transform/src/systems.rs:715 panics on a malformed hierarchy; keep that behaviour
        if rc == ERR_HIERARCHY_CYCLE { panic!("Malformed hierarchy: {msg}"); }
        Err(format!("b200vis error {rc}: {msg}").into())
    }
    fn class_bit(&mut self, id: TypeId) -> u8 {
        if let Some(k) = self.classes.iter().position(|c| *c == id) { return 1 << k; }
        assert!(self.classes.len() < 8, "libb200vis carries at most 8 VisibilityClass ids");
        self.classes.push(id);
        1 << (self.classes.len() - 1)
    }
}

pub struct B200VisibilityPlugin { pub max_entities: u32, pub max_lights: u32 }

impl Plugin for B200VisibilityPlugin {
    fn build(&self, app: &mut App) {
        let cfg = b200vis_config { device: 0, max_entities: self.max_entities, max_lights: self.max_lights, max_views: MAX_VIEWS as u32,
                                   max_cluster_indices: 0, world_size: 1, rank: 0, reserved: 0 };
        let mut ctx = core::ptr::null_mut();
        let rc = unsafe { b200vis_create(&cfg, &mut ctx) };
        assert_eq!(rc, 0, "b200vis_create failed: there is no CPU fallback");
        let n = self.max_entities as usize;
        let cluster_cap = 1usize << 18;
        let mut vis = B200Vis {
            ctx, max_entities: n, n: 0, row_of: Default::default(), entity_of: Vec::new(), columns_epoch: 0, bounds_epoch: u64::MAX,
            lights_epoch: u64::MAX, classes: Vec::new(), view_entities: Vec::new(), light_entities: Vec::new(), object_kinds: Vec::new(),
            stats: Box::default(), gt_col: vec![[0.0; 16]; n], gt_bits: vec![0; n.div_ceil(32)], vv_col: vec![0; n],
            vv_bits: vec![0; n.div_ceil(32)], visible_rows: vec![0; MAX_VIEWS * n], visible_classes: vec![0; MAX_VIEWS * n],
            cluster_offsets: vec![0; MAX_VIEWS * (MAX_CLUSTERS + 1)], cluster_indices: vec![0; MAX_VIEWS * cluster_cap], cluster_cap,
            planes_scratch: vec![0.0; 3 * 4097 * 4],
        };
        let rs = b200vis_result_sink { stats: &mut *vis.stats, visible_rows: vis.visible_rows.as_mut_ptr(), visible_capacity: n as u32,
            visible_classes: vis.visible_classes.as_mut_ptr(), cluster_offsets: vis.cluster_offsets.as_mut_ptr(),
            cluster_indices: vis.cluster_indices.as_mut_ptr(), cluster_capacity: cluster_cap as u32 };
        let cs = b200vis_column_sinks { global_transforms: vis.gt_col.as_mut_ptr().cast(), gt_stride_floats: 16,
            gt_changed_bits: vis.gt_bits.as_mut_ptr(), view_visibility: vis.vv_col.as_mut_ptr(), vv_changed_bits: vis.vv_bits.as_mut_ptr() };
        unsafe { assert_eq!(b200vis_set_result_sink(ctx, &rs), 0); assert_eq!(b200vis_set_column_sinks(ctx, &cs), 0); }
        app.insert_resource(vis);
        // CPU clustering mode, so that `Clusters` holds `ClusterableObjects::Cpu`, which the cluster system fills (SURVEY.md 0)
        app.insert_resource(GlobalClusterSettings { gpu_clustering: None, supports_storage_buffers: true,
            clustered_decals_are_usable: false, max_uniform_buffer_clusterable_objects: 204, view_cluster_bindings_max_indices: 16384 });
    }
    fn finish(&self, app: &mut App) {
        for schedule in [PostStartup.intern(), PostUpdate.intern()] {
            app.remove_systems_in_set(schedule, mark_dirty_trees, RemoveSystemsOnly);
            app.remove_systems_in_set(schedule, propagate_parent_transforms, RemoveSystemsOnly);
            app.remove_systems_in_set(schedule, sync_simple_transforms, RemoveSystemsOnly);
            app.add_systems(schedule, b200_propagate.in_set(TransformSystems::Propagate));
        }
        app.remove_systems_in_set(PostUpdate, check_visibility_cpu_culling, RemoveSystemsOnly);
        app.remove_systems_in_set(PostUpdate, SimulationLightSystems::AssignLightsToClusters, RemoveSystemsOnly);
        app.add_systems(PostUpdate, (
            b200_check_visibility.in_set(VisibilitySystems::CheckVisibility),
            b200_assign_lights_to_clusters.in_set(SimulationLightSystems::AssignLightsToClusters)
                .after(TransformSystems::Propagate).after(VisibilitySystems::CheckVisibility),
        ));
    }
}

fn pack_trs(t: &Transform, out: &mut Vec<f32>) {
    out.extend_from_slice(&[t.translation.x, t.translation.y, t.translation.z, t.rotation.x, t.rotation.y, t.rotation.z, t.rotation.w,
                            t.scale.x, t.scale.y, t.scale.z]);
}
fn pack_gt12(g: &GlobalTransform, out: &mut Vec<f32>) {
    let a = g.affine();
    out.extend_from_slice(&[a.matrix3.x_axis.x, a.matrix3.x_axis.y, a.matrix3.x_axis.z, a.matrix3.y_axis.x, a.matrix3.y_axis.y,
                            a.matrix3.y_axis.z, a.matrix3.z_axis.x, a.matrix3.z_axis.y, a.matrix3.z_axis.z, a.translation.x,
                            a.translation.y, a.translation.z]);
}
fn affine_from_col(m: &[f32; 16]) -> GlobalTransform {
    // the sink's layout IS glam's Affine3A: x_axis, y_axis, z_axis, translation as four 16-byte Vec3A lanes
    GlobalTransform::from(bevy::math::Affine3A::from_cols(
        bevy::math::Vec3A::new(m[0], m[1], m[2]), bevy::math::Vec3A::new(m[4], m[5], m[6]),
        bevy::math::Vec3A::new(m[8], m[9], m[10]), bevy::math::Vec3A::new(m[12], m[13], m[14])))
}
fn set_bits(words: &[u32], n: usize) -> impl Iterator<Item = usize> + '_ {
    words.iter().enumerate().flat_map(move |(w, &bits)| {
        let mut b = bits;
        core::iter::from_fn(move || { if b == 0 { None } else { let k = b.trailing_zeros() as usize; b &= b - 1; Some(w * 32 + k) } })
    }).filter(move |r| *r < n)
}

/// propagate: the data propagate_parent_transforms' queries (systems.rs:506-520) and sync_simple_transforms'
/// (systems.rs:42-55) read and write, as one query.
fn b200_propagate(
    mut vis: ResMut<B200Vis>,
    mut q: Query<(Entity, Ref<Transform>, &mut GlobalTransform, Option<&Children>, Option<&ChildOf>)>,
    structure_changed: Query<(), Or<(Added<GlobalTransform>, Changed<ChildOf>)>>,
    mut orphaned: RemovedComponents<ChildOf>,
    mut despawned: RemovedComponents<GlobalTransform>,
    opts: Res<StaticTransformOptimizations>,
) -> Result<(), BevyError> {
    let vis = &mut *vis;
    let rebuild = vis.n != q.iter().len() || !structure_changed.is_empty() || orphaned.read().next().is_some()
        || despawned.read().next().is_some();
    if rebuild {
        // ---- rows are renumbered: tree-contiguous BFS order (the layout the tile kernel likes), then every column again ----
        let old: Vec<(Entity, Option<Entity>)> = q.iter().map(|(e, _, _, _, p)| (e, p.map(|p| p.parent()))).collect();
        let n = old.len();
        assert!(n <= vis.max_entities, "B200VisibilityPlugin::max_entities is too small");
        let old_row: EntityHashMap<u32> = old.iter().enumerate().map(|(i, (e, _))| (*e, i as u32)).collect();
        // ChildOf whose parent lacks Transform/GlobalTransform is outside NodeQuery (systems.rs:752-764): DETACHED
        let parent_old: Vec<u32> = old.iter().map(|(_, p)| match p { None => NO_PARENT, Some(p) => *old_row.get(p).unwrap_or(&DETACHED) }).collect();
        let mut new_to_old = vec![0u32; n];
        vis.check(unsafe { b200vis_plan_row_order(n as u32, parent_old.as_ptr(), new_to_old.as_mut_ptr()) })?;
        let mut new_of_old = vec![0u32; n];
        for (new, &o) in new_to_old.iter().enumerate() { new_of_old[o as usize] = new as u32; }
        vis.entity_of = new_to_old.iter().map(|&o| old[o as usize].0).collect();
        vis.row_of = vis.entity_of.iter().enumerate().map(|(r, e)| (*e, r as u32)).collect();
        let parent_new: Vec<u32> = new_to_old.iter().map(|&o| { let p = parent_old[o as usize]; if p < n as u32 { new_of_old[p as usize] } else { p } }).collect();
        let bits: Vec<u64> = vis.entity_of.iter().map(|e| e.to_bits()).collect();
        vis.check(unsafe { b200vis_set_topology(vis.ctx, n as u32, parent_new.as_ptr(), bits.as_ptr()) })?;
        let (mut trs, mut gt) = (Vec::with_capacity(n * 10), Vec::with_capacity(n * 12));
        for e in &vis.entity_of {
            let (_, t, g, _, _) = q.get(*e).unwrap();
            pack_trs(&t, &mut trs); pack_gt12(&g, &mut gt);
            vis.gt_col[vis.row_of[e] as usize] = { let mut m = [0.0; 16]; let a = g.affine().to_cols_array(); // 12 floats, column major
                m[0..3].copy_from_slice(&a[0..3]); m[4..7].copy_from_slice(&a[3..6]); m[8..11].copy_from_slice(&a[6..9]); m[12..15].copy_from_slice(&a[9..12]); m };
        }
        // upload_transforms marks every row Changed<Transform>: the first propagate visits everything, like Added<GlobalTransform>
        vis.check(unsafe { b200vis_upload_transforms(vis.ctx, 0, n as u32, trs.as_ptr()) })?;
        vis.check(unsafe { b200vis_upload_global_transforms(vis.ctx, 0, n as u32, gt.as_ptr()) })?;
        vis.n = n;
        vis.columns_epoch += 1;
    } else {
        // ---- steady state: only rows matching Changed<Transform> cross PCIe ----
        let (mut rows, mut trs) = (Vec::new(), Vec::new());
        for (e, t, _, _, _) in q.iter() {
            if t.is_changed() { rows.push(vis.row_of[&e]); pack_trs(&t, &mut trs); }
        }
        if !rows.is_empty() {
            vis.check(unsafe { b200vis_upload_transforms_scattered(vis.ctx, rows.len() as u32, rows.as_ptr(), trs.as_ptr()) })?;
        }
    }
    unsafe {
        vis.check(b200vis_set_static_transform_optimizations(vis.ctx, opts.is_enabled() as i32))?;
        vis.check(b200vis_run(vis.ctx, STAGE_PROPAGATE))?;
        vis.check(b200vis_writeback_columns_ex(vis.ctx, WB_GLOBAL_TRANSFORM))?;      // changed rows only, straight into gt_col
        vis.check(b200vis_synchronize(vis.ctx))?;
    }
    // set_if_neq semantics (systems.rs:719): only the rows whose bits changed are written, and exactly those get their
    // change tick stamped (assigning through `Mut` does both).  When the table rows happen to be in device-row order the
    // same can be done in bulk: `q.contiguous_iter_mut()` -> `ContiguousMut::bypass_change_detection()` as the column sink
    // itself and `changed_ticks_slice_mut()[r] = this_run_tick()` per set bit (change_detection/params.rs:1079-1142).
    for r in set_bits(&vis.gt_bits, vis.n) {
        if let Ok((_, _, mut g, _, _)) = q.get_mut(vis.entity_of[r]) { *g = affine_from_col(&vis.gt_col[r]); }
    }
    Ok(())
}

/// cull: the parameter list of check_visibility_cpu_culling (visibility/mod.rs:748-774); `Ref` instead of `&` where the shim
/// needs change detection for its column mirror.
fn b200_check_visibility(
    mut vis: ResMut<B200Vis>,
    mut view_query: Query<(Entity, &mut VisibleEntities, &Frustum, Option<&RenderLayers>, &Camera, Has<NoCpuCulling>)>,
    mut visible_aabb_query: Query<(Entity, Ref<InheritedVisibility>, &mut ViewVisibility, Option<Ref<VisibilityClass>>, Option<Ref<RenderLayers>>,
                                   Option<Ref<Aabb>>, Option<Ref<Sphere>>, &GlobalTransform, Has<NoFrustumCulling>, Has<VisibilityRange>,
                                   Has<PointLight>), Without<NoCpuCulling>>,
    visible_entity_ranges: Option<Res<VisibleEntityRanges>>,
) -> Result<(), BevyError> {
    let vis = &mut *vis;
    // ---- views: half spaces copied verbatim from `Frustum` (bit-identical by construction) ----
    let mut views = Vec::new();
    vis.view_entities.clear();
    for (entity, _, frustum, layers, camera, no_cpu_culling) in view_query.iter() {
        let mut v = b200vis_view { half_spaces: [[0.0; 4]; 6], layer_mask: layers.map_or(1, |l| l.bits()[0]),
                                   flags: (camera.is_active as u8 * VIEW_ACTIVE) | (no_cpu_culling as u8 * VIEW_NO_CPU_CULLING),
                                   range_view_index: -1, pad: [0; 6] };
        for (k, hs) in frustum.half_spaces.iter().enumerate() { v.half_spaces[k] = hs.normal_d().to_array(); }
        // VisibleEntityRanges keeps its view -> bit table private; the shim builds its own masks below with bit v = device view v
        if visible_entity_ranges.is_some() { v.range_view_index = views.len() as i8; }
        views.push(v); vis.view_entities.push(entity);
        if views.len() == MAX_VIEWS { break; }
    }
    vis.check(unsafe { b200vis_set_views(vis.ctx, views.len() as u32, views.as_ptr()) })?;
    // ---- row columns: everything after a renumbering, otherwise the rows whose components changed, as contiguous ranges ----
    let all = vis.bounds_epoch != vis.columns_epoch;
    let mut dirty: Vec<u32> = Vec::new();
    let n = vis.n;
    let (mut bounds, mut flags, mut class, mut layer, mut range) = (vec![0f32; n * 6], vec![0u8; n], vec![0u8; n], vec![1u64; n], vec![0u32; n]);
    for (e, inherited, _, vclass, layers, aabb, sphere, _, no_frustum, has_range, is_light) in visible_aabb_query.iter() {
        let Some(&r) = vis.row_of.get(&e) else { continue };
        // (VisibleEntityRanges is rebuilt by check_visibility_ranges every frame: rows with a VisibilityRange are always refreshed)
        let changed = all || has_range || inherited.is_changed() || vclass.as_ref().is_some_and(|c| c.is_changed()) || layers.as_ref().is_some_and(|c| c.is_changed())
            || aabb.as_ref().is_some_and(|c| c.is_changed()) || sphere.as_ref().is_some_and(|c| c.is_changed());
        if !changed { continue; }
        let r = r as usize;
        let mut f = if inherited.get() { F_INHERITED } else { 0 } | if no_frustum { F_NO_FRUSTUM } else { 0 } | if has_range { F_RANGE } else { 0 };
        if let Some(a) = &aabb { f |= F_AABB; bounds[r * 6..r * 6 + 6].copy_from_slice(&[a.center.x, a.center.y, a.center.z, a.half_extents.x, a.half_extents.y, a.half_extents.z]); }
        else if let Some(s) = &sphere {
            // a point light's Sphere is rebuilt from its GlobalTransform every frame (point_light.rs:195-209): the device does the
            // same from the row's own translation (F_SPHERE_FROM_GT) and only needs the radius
            f |= F_SPHERE | if is_light { F_SPHERE_FROM_GT } else { 0 };
            bounds[r * 6..r * 6 + 4].copy_from_slice(&[s.center.x, s.center.y, s.center.z, s.radius]);
        }
        flags[r] = f;
        class[r] = vclass.as_ref().map_or(0, |c| c.iter().fold(0u8, |m, id| m | vis.class_bit(*id)));
        layer[r] = layers.as_ref().map_or(1, |l| l.bits()[0]);
        range[r] = match (&visible_entity_ranges, has_range) {       // entity_is_in_range_of_view (visibility/range.rs:214-222)
            (Some(vr), true) => vis.view_entities.iter().enumerate().fold(0u32, |m, (v, view)| m | ((vr.entity_is_in_range_of_view(e, *view) as u32) << v)),
            _ => 0,
        };
        dirty.push(r as u32);
    }
    dirty.sort_unstable();
    let mut i = 0;
    while i < dirty.len() {                                     // coalesce into [first, first + count) ranges
        let first = dirty[i] as usize;
        let mut j = i + 1;
        while j < dirty.len() && dirty[j] == dirty[j - 1] + 1 { j += 1; }
        let c = j - i;
        vis.check(unsafe { b200vis_upload_bounds(vis.ctx, first as u32, c as u32, bounds[first * 6..].as_ptr(), flags[first..].as_ptr(),
            class[first..].as_ptr(), layer[first..].as_ptr(), if visible_entity_ranges.is_some() { range[first..].as_ptr() } else { core::ptr::null() }) })?;
        i = j;
    }
    if all {
        #[cfg(feature = "forked-bevy")]
        { let vv: Vec<u8> = vis.entity_of.iter().map(|e| visible_aabb_query.get(*e).map_or(0, |q| q.2.bits())).collect();
          vis.check(unsafe { b200vis_upload_view_visibility(vis.ctx, 0, n as u32, vv.as_ptr()) })?; }
        vis.bounds_epoch = vis.columns_epoch;
    }
    unsafe {
        vis.check(b200vis_run(vis.ctx, STAGE_CULL))?;
        vis.check(b200vis_writeback_columns_ex(vis.ctx, WB_VIEW_VISIBILITY))?;
        vis.check(b200vis_synchronize(vis.ctx))?;       // stats, sorted lists + class masks, ViewVisibility bytes are in host memory now
    }
    // ---- VisibleEntities: one sorted Vec per class; an entity is pushed once per class it carries (mod.rs:846-857).  The device
    // list is already in Entity::to_bits() order, so every class list comes out sorted and the reference's sort_unstable
    // (mod.rs:870-874) has nothing left to do ----
    for (v, view_entity) in vis.view_entities.iter().enumerate() {
        let Ok((_, mut visible_entities, _, _, camera, _)) = view_query.get_mut(*view_entity) else { continue };
        if !camera.is_active { continue; }                       // an inactive view keeps its lists (mod.rs:780-782)
        for list in visible_entities.entities.values_mut() { list.clear(); }
        let count = vis.stats.visible_count[v] as usize;
        let (rows, masks) = (&vis.visible_rows[v * vis.max_entities..][..count], &vis.visible_classes[v * vis.max_entities..][..count]);
        for (row, mask) in rows.iter().zip(masks) {
            let entity = vis.entity_of[*row as usize];
            let mut m = *mask;
            while m != 0 { let k = m.trailing_zeros() as usize; m &= m - 1; visible_entities.get_mut(vis.classes[k]).push(entity); }
        }
    }
    // ---- ViewVisibility ----
    #[cfg(not(feature = "forked-bevy"))]
    for (r, byte) in vis.vv_col[..n].iter().enumerate() {        // the CPU bracket systems own the 2-bit state machine and the ticks
        if byte & 1 != 0 { if let Ok(mut q) = visible_aabb_query.get_mut(vis.entity_of[r]) { q.2.set_visible(); } }
    }
    #[cfg(feature = "forked-bevy")]
    for r in 0..n {                                              // the device owns it: bytes via bypass, ticks where the bit is set
        if let Ok(mut q) = visible_aabb_query.get_mut(vis.entity_of[r]) {
            *q.2.bypass_change_detection() = ViewVisibility::from_bits(vis.vv_col[r]);
            if vis.vv_bits[r / 32] >> (r % 32) & 1 != 0 { q.2.set_changed(); }
        }
    }
    Ok(())
}

/// cluster: the queries of assign_objects_to_clusters (assign.rs:137-178) except spot lights -- an app with spot lights keeps
/// the reference system (INTEGRATION.md).
fn b200_assign_lights_to_clusters(
    mut vis: ResMut<B200Vis>,
    mut views: Query<(Entity, &GlobalTransform, &Camera, &Frustum, Option<&ClusterConfig>, &mut Clusters, Option<&RenderLayers>)>,
    point_lights_query: Query<(Entity, &GlobalTransform, &ViewVisibility, Ref<PointLight>, Option<Ref<RenderLayers>>)>,
    rect_lights_query: Query<(Entity, &GlobalTransform, &ViewVisibility, Ref<RectLight>, Option<Ref<RenderLayers>>)>,
    light_probes_query: Query<(Entity, &GlobalTransform, &ViewVisibility, Has<EnvironmentMapLight>), With<LightProbe>>,
    decals_query: Query<(Entity, &GlobalTransform, &ViewVisibility), With<ClusteredDecal>>,
    mut removed_lights: RemovedComponents<PointLight>,
    mut removed_rect_lights: RemovedComponents<RectLight>,
    mut removed_probes: RemovedComponents<LightProbe>,
    mut removed_decals: RemovedComponents<ClusteredDecal>,
    added_objects: Query<(), Or<(Added<LightProbe>, Added<ClusteredDecal>, Changed<EnvironmentMapLight>)>>,
    settings: Res<GlobalClusterSettings>,
) -> Result<(), BevyError> {
    let vis = &mut *vis;
    // ---- lights: ordinal = query order; positions and ViewVisibility are read on the device from the lights' own rows ----
    let mut removed = removed_lights.read().count() + removed_rect_lights.read().count();
    removed += removed_probes.read().count() + removed_decals.read().count();
    let lights_changed = vis.lights_epoch != vis.columns_epoch || removed > 0 || !added_objects.is_empty()
        || point_lights_query.iter().any(|(_, _, _, l, r)| l.is_changed() || r.is_some_and(|r| r.is_changed()))
        || rect_lights_query.iter().any(|(_, _, _, l, r)| l.is_changed() || r.is_some_and(|r| r.is_changed()));
    if lights_changed {
        vis.light_entities.clear();
        let (mut rows, mut ranges, mut layers) = (Vec::new(), Vec::new(), Vec::new());
        for (e, _, _, light, layer) in point_lights_query.iter() {
            let Some(&r) = vis.row_of.get(&e) else { continue };
            vis.light_entities.push(e); rows.push(r); ranges.push(light.range); layers.push(layer.map_or(1, |l| l.bits()[0]));
        }
        vis.check(unsafe { b200vis_set_lights(vis.ctx, rows.len() as u32, rows.as_ptr(), ranges.as_ptr(), layers.as_ptr()) })?;
        // the other kinds, in the reference's push order and under its settings gates (assign.rs:231-295); their radius and
        // ViewVisibility are taken on the device from this frame's rows, only a rect light's range and layers are uploaded
        let (mut kinds, mut orows, mut oranges, mut olayers) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
        let mut push = |vis: &mut B200Vis, e: Entity, kind: u32, range: f32, layer: u64| {
            let Some(&r) = vis.row_of.get(&e) else { return };
            vis.light_entities.push(e); kinds.push(kind); orows.push(r); oranges.push(range); olayers.push(layer);
        };
        if settings.supports_storage_buffers {
            for (e, _, _, light, layer) in rect_lights_query.iter() { push(vis, e, KIND_RECT_LIGHT, light.range, layer.map_or(1, |l| l.bits()[0])); }
            for (e, _, _, is_reflection_probe) in light_probes_query.iter() {
                push(vis, e, if is_reflection_probe { KIND_REFLECTION_PROBE } else { KIND_IRRADIANCE_VOLUME }, 0.0, 1);
            }
        }
        if settings.clustered_decals_are_usable {
            for (e, _, _) in decals_query.iter() { push(vis, e, KIND_DECAL, 0.0, 1); }
        }
        vis.check(unsafe { b200vis_set_clusterable_objects(vis.ctx, kinds.len() as u32, kinds.as_ptr(), orows.as_ptr(), oranges.as_ptr(),
                                                           olayers.as_ptr()) })?;
        vis.object_kinds = kinds;
        vis.lights_epoch = vis.columns_epoch;
    }
    // ---- per view: the prologue of assign_objects_to_clusters (assign.rs:324-485) through the library's host helper, which
    // restates it op for op (dims via ClusterConfig::dimensions_for_screen_size, Clusters::update, far_z / cluster_factors
    // from last frame's feedback, the x / y / z HalfSpace tables) ----
    let mut order = Vec::new();
    for (entity, camera_transform, camera, frustum, config, clusters, layers) in views.iter() {
        let Some(v) = vis.view_entities.iter().position(|e| *e == entity) else { continue };
        let size = camera.physical_viewport_size().unwrap_or(UVec2::ZERO);
        let config = config.copied().unwrap_or_default();
        let (kind, dims, total, z_slices, z_cfg, dyn_resize) = match config {        // cluster/mod.rs:107-139
            ClusterConfig::None => (0, [0; 3], 0, 0, ClusterZConfig::default(), false),
            ClusterConfig::Single => (1, [1; 3], 0, 0, ClusterZConfig::default(), false),
            ClusterConfig::XYZ { dimensions, z_config, dynamic_resizing } => (2, dimensions.to_array(), 0, 0, z_config, dynamic_resizing),
            ClusterConfig::FixedZ { total, z_slices, z_config, dynamic_resizing } => (3, [0; 3], total, z_slices, z_config, dynamic_resizing),
        };
        let (far_z_mode, far_z_constant) = match z_cfg.far_z_mode {
            ClusterFarZMode::MaxClusterableObjectRange => (0, 0.0), ClusterFarZMode::Constant(z) => (1, z) };
        let cfg = b200vis_cluster_config { kind, dims, total, z_slices, first_slice_depth: z_cfg.first_slice_depth, far_z_mode,
            far_z_constant, dynamic_resizing: dyn_resize as u32, screen_w: size.x, screen_h: size.y,
            view_cluster_bindings_max_indices: settings.view_cluster_bindings_max_indices as u32 };
        let fb = b200vis_cluster_feedback { has_farthest_z: clusters.last_frame_farthest_z.is_some() as u32,
            farthest_z: clusters.last_frame_farthest_z.unwrap_or(0.0),
            has_index_count: clusters.last_frame_total_cluster_index_count.is_some() as u32,
            index_count: clusters.last_frame_total_cluster_index_count.unwrap_or(0) as u32 };
        let mut gt12 = Vec::with_capacity(12); pack_gt12(camera_transform, &mut gt12);
        let cfv = camera.clip_from_view().to_cols_array();
        let hs: Vec<[f32; 4]> = frustum.half_spaces.iter().map(|h| h.normal_d().to_array()).collect();
        let mut cv = core::mem::MaybeUninit::<b200vis_cluster_view>::zeroed();
        unsafe {
            vis.check(b200vis_host_cluster_view_setup(&cfg, gt12.as_ptr(), cfv.as_ptr(), hs.as_ptr(), layers.map_or(1, |l| l.bits()[0]), &fb,
                                                      vis.planes_scratch.as_mut_ptr(), cv.as_mut_ptr()))?;
            vis.check(b200vis_set_cluster_view(vis.ctx, v as u32, cv.as_ptr()))?;
            order.push((entity, v, cv.assume_init()));
        }
    }
    unsafe { vis.check(b200vis_run(vis.ctx, STAGE_CLUSTER))?; vis.check(b200vis_synchronize(vis.ctx))?; }
    // ---- results: Clusters::update / reset_for_new_frame restated (cluster/mod.rs:398-468), then one add_point_light per index ----
    for (entity, v, cv) in order {
        let Ok((_, _, _, _, _, mut clusters, _)) = views.get_mut(entity) else { continue };
        if cv.enabled == 0 {                                     // clusters.clear(): ClusterConfig::None or an empty viewport (assign.rs:334-340)
            clusters.tile_size = UVec2::ONE; clusters.dimensions = UVec3::ZERO; clusters.near = 0.0; clusters.far = 0.0;
            if let ClusterableObjects::Cpu(list) = &mut clusters.clusterable_objects { list.clear(); }
            continue;
        }
        clusters.tile_size = UVec2::new(cv.tile_size[0], cv.tile_size[1]);
        clusters.dimensions = UVec3::new(cv.dims[0], cv.dims[1], cv.dims[2]);
        clusters.near = cv.near_z; clusters.far = cv.far_z;
        let nc = (cv.dims[0] * cv.dims[1] * cv.dims[2]) as usize;
        let mut cells = vec![ObjectsInClusterCpu::default(); nc];
        let off = &vis.cluster_offsets[v * (MAX_CLUSTERS + 1)..][..nc + 1];
        let idx = &vis.cluster_indices[v * vis.cluster_cap..];
        let first_object = vis.light_entities.len() - vis.object_kinds.len();
        for (c, cell) in cells.iter_mut().enumerate() {
            for i in off[c]..off[c + 1] {                        // ascending ordinal = push order (assign.rs:487, 740-800)
                let o = idx[i as usize] as usize;
                let e = vis.light_entities[o];
                if o < first_object { cell.add_point_light(e); continue; }
                match vis.object_kinds[o - first_object] {
                    KIND_RECT_LIGHT => cell.add_rect_light(e),
                    KIND_REFLECTION_PROBE => cell.add_reflection_probe(e),
                    KIND_IRRADIANCE_VOLUME => cell.add_irradiance_volume(e),
                    _ => cell.add_decal(e),
                }
            }
        }
        clusters.clusterable_objects = ClusterableObjects::Cpu(cells);
        clusters.last_frame_total_cluster_index_count = Some(vis.stats.cluster_index_count[v] as usize);
        clusters.last_frame_farthest_z = Some(vis.stats.cluster_farthest_z[v]);     // assign.rs:810-811
    }
    Ok(())
}
